// dfb_params.h -- host-side validation of the C-ABI structs (include/dfb.h) and construction of the
// kernel parameter blocks (dfb_voxel.h).  Plain C++ (no CUDA runtime calls) so that the CPU logic tests
// (tests/hostshim/) build the exact same parameter blocks as the library.
#pragma once
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include "dfb_require.h"
#include "dfb_voxel.h"

namespace dfb {

inline void mat34_mul(const double* A, const double* B, double* C) {  // C = A * B as 4x4 affine maps
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) {
            double s = 0;
            for (int j = 0; j < 3; ++j) s += A[4 * r + j] * B[4 * j + c];
            if (c == 3) s += A[4 * r + 3];
            C[4 * r + c] = s;
        }
}

inline void k_mul34(const double* K, const double* A, double* C) {  // C(3x4) = K(3x3) * A(3x4)
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) {
            double s = 0;
            for (int j = 0; j < 3; ++j) s += K[3 * r + j] * A[4 * j + c];
            C[4 * r + c] = s;
        }
}

// largest magnitude of any term / result when A is applied to the corners of the box [0,ex]x[0,ey]x[0,ez]
inline double affine_corner_mag(const double* A, double ex, double ey, double ez) {
    double mag = 0;
    for (int c = 0; c < 8; ++c) {
        const double p[3] = {(c & 1) * ex, ((c >> 1) & 1) * ey, ((c >> 2) & 1) * ez};
        for (int r = 0; r < 3; ++r) {
            const double v = A[4 * r] * p[0] + A[4 * r + 1] * p[1] + A[4 * r + 2] * p[2] + A[4 * r + 3];
            mag = fmax(mag, fabs(v));
            for (int j = 0; j < 3; ++j) mag = fmax(mag, fabs(A[4 * r + j] * p[j]));
            mag = fmax(mag, fabs(A[4 * r + 3]));
        }
    }
    return mag;
}

inline int validate_volume(const dfb_volume* vol) {
    DFB_REQUIRE(vol && vol->tsdf && vol->weight, "volume pointers are null");
    DFB_REQUIRE(vol->rx > 0 && vol->ry > 0 && vol->rz > 0, "bad volume resolution");
    DFB_REQUIRE(vol->x0 >= 0 && vol->x1 > vol->x0 && vol->x1 <= vol->rx, "bad slab [%d,%d) of %d", vol->x0, vol->x1, vol->rx);
    DFB_REQUIRE(vol->ry <= 65535 && (vol->x1 - vol->x0) <= 65535, "ry and slab thickness must be <= 65535");
    DFB_REQUIRE((size_t)(vol->x1 - vol->x0) * vol->ry * vol->rz < ((size_t)1 << 32), "slab has >= 2^32 voxels");
    return DFB_OK;
}

inline int validate_warpfield(const dfb_warpfield* wf, bool need_knn) {
    DFB_REQUIRE(wf, "warpfield is null");
    DFB_REQUIRE(wf->k >= 0 && wf->k <= DFB_MAX_K, "k=%d out of range [0,%d]", wf->k, DFB_MAX_K);
    if (wf->k > 0) {
        DFB_REQUIRE(wf->node_rec && wf->node_pos && wf->node_dq && wf->node_w, "node arrays are null");
        DFB_REQUIRE(wf->n_nodes >= wf->k && wf->n_nodes <= 65535, "n_nodes=%d must be in [k,65535]", wf->n_nodes);
        if (need_knn) DFB_REQUIRE(wf->knn, "knn table is null");
    }
    return DFB_OK;
}

inline int validate_ws(const dfb_workspace* ws) {
    DFB_REQUIRE(ws && ws->counters, "workspace/counters are null");
    DFB_REQUIRE(ws->capacity == 0 || ws->list, "workspace list is null");
    return DFB_OK;
}

inline void fill_common(ProjParams& P, const dfb_volume* vol, const dfb_workspace* ws, double tdist, double wmax,
                        uint8_t* mask_out, uint8_t* frustum_out) {
    P.tsdf = vol->tsdf; P.weight = vol->weight;
    P.rx = vol->rx; P.ry = vol->ry; P.rz = vol->rz; P.x0 = vol->x0; P.x1 = vol->x1;
    P.tdist = fabs(tdist); P.wmax = wmax;
    P.tdist_f = (float)fabs(tdist); P.wmax_f = (float)wmax;
    P.list = ws->list; P.capacity = ws->capacity; P.counters = ws->counters; P.overflow_bits = ws->overflow_bits;
    P.mask_out = mask_out; P.frustum_out = frustum_out;
}

inline void fill_intrinsics(ProjParams& P, const double* K, const double* Kinv) {
    for (int i = 0; i < 9; ++i) { P.K[i] = K[i]; P.Kinv[i] = Kinv[i]; }
    for (int i = 0; i < 3; ++i) P.kin[i] = (float)Kinv[6 + i];
    for (int i = 0; i < 6; ++i) P.kf[i] = (float)K[i];
    P.k_pinhole = (K[6] == 0.0 && K[7] == 0.0 && K[8] == 1.0) ? 1 : 0;
    P.knorm = (float)fmax(fabs(K[0]) + fabs(K[1]) + fabs(K[2]), fabs(K[3]) + fabs(K[4]) + fabs(K[5]));
    P.kin_uv = (float)(fabs(Kinv[6]) + fabs(Kinv[7]));
    P.ezf = (float)(fmax(1.0, fabs(K[6]) + fabs(K[7]) + fabs(K[8])) * 1.000001);
}

static const double kIdent34[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};

inline int build_projective(ProjParams& P, const dfb_volume* vol, const dfb_warpfield* wf, const dfb_views* views,
                            double tdist, double wmax, int mode, const dfb_workspace* ws, uint8_t* mask_out,
                            uint8_t* frustum_out) {
    if (int r = validate_volume(vol)) return r;
    if (int r = validate_warpfield(wf, true)) return r;
    if (int r = validate_ws(ws)) return r;
    DFB_REQUIRE(views && views->n_views >= 1 && views->n_views <= DFB_MAX_VIEWS, "n_views out of range");
    DFB_REQUIRE(views->rows >= 2 && views->cols >= 2, "depth map too small");
    DFB_REQUIRE(mode >= DFB_MODE_HYBRID && mode <= DFB_MODE_BRICK_UPDATE, "bad mode");
    DFB_REQUIRE(wf->k > 0, "projective update needs k >= 1 (use dfb_fuse_depth_rigid for the rigid path)");
    DFB_REQUIRE(tdist != 0, "truncation distance must be non-zero");
    memset(&P, 0, sizeof(P));
    fill_common(P, vol, ws, tdist, wmax, mask_out, frustum_out);
    P.scale = 1.0;
    P.node_rec = reinterpret_cast<const float4*>(wf->node_rec);
    P.node_pos = wf->node_pos; P.node_dq = wf->node_dq; P.node_w = wf->node_w; P.knn = wf->knn; P.k = wf->k;
    P.has_lw = wf->has_lw; P.lw_is_f32 = wf->lw_is_f32;
    for (int i = 0; i < 8; ++i) P.lw[i] = wf->lw[i];
    P.n_views = views->n_views; P.rows = views->rows; P.cols = views->cols; P.has_E = views->has_extrinsics;
    fill_intrinsics(P, views->K, views->Kinv);
    double A[12];
    if (wf->has_lw) dq_to_affine(wf->lw, A);
    else memcpy(A, kIdent34, sizeof(A));
    double mag = fmax(fmax(vol->rx, vol->ry), vol->rz);
    mag = fmax(mag, affine_corner_mag(A, vol->rx, vol->ry, vol->rz));
    double tnorm = 0.0;
    for (int v = 0; v < views->n_views; ++v) {
        DFB_REQUIRE(views->depth[v], "depth[%d] is null", v);
        P.depth[v] = views->depth[v];
        double T[12], PK[12];
        if (views->has_extrinsics) {
            for (int i = 0; i < 12; ++i) P.E[v][i] = views->E[v][i];
            mat34_mul(views->E[v], A, T);
        } else {
            memcpy(T, A, sizeof(T));
        }
        mag = fmax(mag, affine_corner_mag(T, vol->rx, vol->ry, vol->rz));
        k_mul34(views->K, T, PK);
        for (int i = 0; i < 12; ++i) P.vf[v].P[i] = (float)PK[i];
        for (int i = 0; i < 4; ++i) P.vf[v].L[i] = (float)T[8 + i];
        for (int i = 0; i < 12; ++i) P.vf[v].T[i] = (float)T[i];
        for (int r = 0; r < 3; ++r) tnorm = fmax(tnorm, fabs(T[4 * r]) + fabs(T[4 * r + 1]) + fabs(T[4 * r + 2]));
    }
    P.tnorm = (float)(tnorm * 1.000001);
    P.coord_mag = (float)(2.0 * mag + 8.0);
    return DFB_OK;
}

inline int build_rigid(ProjParams& P, const dfb_volume* vol, int tsdf_res, const float* depth, int rows, int cols,
                       const double* lw34, const double* K, const double* Kinv, double scale, const double* center,
                       double tdist, double wmax, int mode, const dfb_workspace* ws, uint8_t* mask_out,
                       uint8_t* frustum_out) {
    if (int r = validate_volume(vol)) return r;
    if (int r = validate_ws(ws)) return r;
    DFB_REQUIRE(depth && lw34 && K && Kinv && center, "null pointer");
    DFB_REQUIRE(rows >= 2 && cols >= 2, "depth map too small");
    DFB_REQUIRE(mode >= DFB_MODE_HYBRID && mode <= DFB_MODE_BRICK_UPDATE, "bad mode");
    DFB_REQUIRE(scale > 0, "scale must be positive");
    DFB_REQUIRE(tdist != 0, "truncation distance must be non-zero");
    memset(&P, 0, sizeof(P));
    fill_common(P, vol, ws, tdist, wmax, mask_out, frustum_out);
    P.scale = scale;
    P.rigid = 1;
    P.k = 0;
    P.g_scale = scale; P.g_half = tsdf_res / 2.0;
    for (int i = 0; i < 3; ++i) P.g_center[i] = center[i];
    for (int i = 0; i < 12; ++i) P.lw34[i] = lw34[i];
    P.n_views = 1; P.rows = rows; P.cols = cols; P.has_E = 0;
    P.depth[0] = depth;
    fill_intrinsics(P, K, Kinv);
    const double G[12] = {scale, 0, 0, center[0] - scale * P.g_half, 0, scale, 0, center[1] - scale * P.g_half,
                          0, 0, scale, center[2] - scale * P.g_half};
    double T[12], PK[12];
    mat34_mul(lw34, G, T);
    k_mul34(K, T, PK);
    for (int i = 0; i < 12; ++i) P.vf[0].P[i] = (float)PK[i];
    for (int i = 0; i < 4; ++i) P.vf[0].L[i] = (float)T[8 + i];
    for (int i = 0; i < 12; ++i) P.vf[0].T[i] = (float)T[i];
    const double mag = fmax(affine_corner_mag(G, vol->rx, vol->ry, vol->rz), affine_corner_mag(T, vol->rx, vol->ry, vol->rz));
    P.coord_mag = (float)(2.0 * mag + 8.0 * scale);
    return DFB_OK;
}

inline int build_volume(VolParams& P, const dfb_volume* vol, const dfb_warpfield* wf, const float* curr, int cx, int cy,
                        int cz, double tdist, double wmax, int mode, const dfb_workspace* ws, uint8_t* mask_out) {
    if (int r = validate_volume(vol)) return r;
    if (int r = validate_warpfield(wf, true)) return r;
    if (int r = validate_ws(ws)) return r;
    DFB_REQUIRE(curr && cx > 0 && cy > 0 && cz > 0, "tsdf of live frame has not been loaded");
    DFB_REQUIRE(mode >= DFB_MODE_HYBRID && mode <= DFB_MODE_BRICK_UPDATE, "bad mode");
    DFB_REQUIRE(tdist != 0, "truncation distance must be non-zero");
    memset(&P, 0, sizeof(P));
    P.tsdf = vol->tsdf; P.weight = vol->weight;
    P.rx = vol->rx; P.ry = vol->ry; P.rz = vol->rz; P.x0 = vol->x0; P.x1 = vol->x1;
    P.node_rec = reinterpret_cast<const float4*>(wf->node_rec);
    P.node_pos = wf->node_pos; P.node_dq = wf->node_dq; P.node_w = wf->node_w; P.knn = wf->knn; P.k = wf->k;
    P.has_lw = wf->has_lw; P.lw_is_f32 = wf->lw_is_f32;
    for (int i = 0; i < 8; ++i) P.lw[i] = wf->lw[i];
    double A[12];
    if (wf->has_lw) dq_to_affine(wf->lw, A);
    else memcpy(A, kIdent34, sizeof(A));
    for (int i = 0; i < 12; ++i) P.A[i] = (float)A[i];
    P.curr = curr; P.cx = cx; P.cy = cy; P.cz = cz;
    P.tdist = fabs(tdist); P.wmax = wmax; P.tdist_f = (float)fabs(tdist); P.wmax_f = (float)wmax;
    double mag = fmax(fmax(vol->rx, vol->ry), vol->rz);
    mag = fmax(mag, affine_corner_mag(A, vol->rx, vol->ry, vol->rz));
    P.coord_mag = (float)(2.0 * mag + 8.0);
    P.list = ws->list; P.capacity = ws->capacity; P.counters = ws->counters; P.overflow_bits = ws->overflow_bits;
    P.mask_out = mask_out;
    return DFB_OK;
}

}  // namespace dfb
