// dfb_raycast.h -- per-ray arithmetic of raycasting the fused volume (csrc/raycast.cu, include/dfb.h dfb_raycast).
//
// The definition is oracle/raycast.py.  Every sample goes through the tracker's own functions (dfb_track.h: track_point_cell,
// track_cell_value), so the raycast surface is the one dfb_track_normal_eq aligns frames to, and every float64 operation of the
// march, the refinement and the box clip is written in the oracle's order with the explicit-rounding helpers of dfb_math.h:
// the device kernel and the test suite's host build both reproduce every ray bit for bit.
#pragma once
#include "dfb_require.h"
#include "dfb_track.h"

namespace dfb {

// One whole volume (rx, ry, rz) on the grid g = (p - center) / scale + half, the gate tdist, and the samples
// z_k = z_near + k step, z_k <= z_far.
struct RaycastParams {
    double center[3];
    double scale, half, tdist, step, z_near, z_far;
    int rows, cols, rx, ry, rz;
};

// The cameras: the inverse intrinsics and one world -> camera pose per view (the identity without extrinsics).
struct RaycastCams {
    double Kinv[9];
    double E[DFB_MAX_VIEWS * 12];
};

// The checks of dfb_raycast, and the blocks of the call.
inline int build_raycast(RaycastParams& P, RaycastCams& cams, const dfb_volume* vol, int tsdf_res, double scale, const double* center,
                         const dfb_views* views, double tdist, double step, double z_near, double z_far, const float* depth,
                         const float* normal) {
    DFB_REQUIRE(vol && center && views && depth && normal, "null pointer");
    DFB_REQUIRE(vol->tsdf && vol->weight, "null pointer (volume)");
    DFB_REQUIRE(vol->rx >= 2 && vol->ry >= 2 && vol->rz >= 2, "volume %dx%dx%d is smaller than one cell", vol->rx, vol->ry, vol->rz);
    DFB_REQUIRE(vol->x0 == 0 && vol->x1 == vol->rx, "slab [%d,%d) of %d planes: raycasting needs the whole volume (trilinear cells "
                "span neighbouring planes)", vol->x0, vol->x1, vol->rx);
    DFB_REQUIRE(tsdf_res >= 1, "tsdf_res=%d must be positive", tsdf_res);
    DFB_REQUIRE(views->n_views >= 1 && views->n_views <= DFB_MAX_VIEWS, "n_views=%d out of range [1,%d]", views->n_views, DFB_MAX_VIEWS);
    DFB_REQUIRE(views->rows >= 1 && views->cols >= 1, "image %dx%d is empty", views->rows, views->cols);
    DFB_REQUIRE(scale > 0, "scale must be positive");
    DFB_REQUIRE(tdist > 0, "truncation distance must be positive");
    DFB_REQUIRE(step > 0, "ray step must be positive");
    DFB_REQUIRE(isfinite(z_near) && isfinite(z_far) && z_near >= 0 && z_near < z_far, "ray range z_near=%g, z_far=%g: need "
                "0 <= z_near < z_far, both finite", z_near, z_far);
    DFB_REQUIRE((z_far - z_near) / step < 1073741824.0, "ray range of (z_far - z_near) / step = %g samples exceeds 2^30",
                (z_far - z_near) / step);
    for (int i = 0; i < 3; ++i) P.center[i] = center[i];
    P.scale = scale; P.half = tsdf_res / 2.0; P.tdist = tdist; P.step = step; P.z_near = z_near; P.z_far = z_far;
    P.rows = views->rows; P.cols = views->cols; P.rx = vol->rx; P.ry = vol->ry; P.rz = vol->rz;
    for (int i = 0; i < 9; ++i) cams.Kinv[i] = views->Kinv[i];
    for (int v = 0; v < views->n_views; ++v)
        for (int i = 0; i < 12; ++i) cams.E[12 * v + i] = views->has_extrinsics ? views->E[v][i] : (i % 5 == 0 ? 1.0 : 0.0);
    return DFB_OK;
}

// Step 5 of oracle/raycast.py: the range [*k0, *k1] of samples the ray of pixel (r, c) can take (*k0 > *k1: none).  The ray's
// grid coordinate og + z dg is clipped to the box [-1/2, r_a - 1/2] (half a cell wider than the cell range) and the range is
// widened by one sample on each side; every sample outside it fails the cell-range test.
DFB_HDN void raycast_clip(const RaycastParams& P, const double* Kinv, const double* lw, int r, int c, int64_t* k0, int64_t* k1) {
    double d[3], e[3];
    for (int k = 0; k < 3; ++k) d[k] = dot3_ref(Kinv + 3 * k, (double)c, (double)r, 1.0);
    for (int k = 0; k < 3; ++k) e[k] = dsub(0.0, lw[4 * k + 3]);
    const int R[3] = {P.rx, P.ry, P.rz};
    double z_in = -INFINITY, z_out = INFINITY;
    for (int a = 0; a < 3; ++a) {
        const double o = dadd(dadd(dmul(lw[a], e[0]), dmul(lw[4 + a], e[1])), dmul(lw[8 + a], e[2]));
        const double og = dadd(ddiv(dsub(o, P.center[a]), P.scale), P.half);
        const double dg = ddiv(dadd(dadd(dmul(lw[a], d[0]), dmul(lw[4 + a], d[1])), dmul(lw[8 + a], d[2])), P.scale);
        const double lo = -0.5, hi = dsub((double)R[a], 0.5);
        double zl, zh;
        if (dg != 0.0) {
            const double z0 = ddiv(dsub(lo, og), dg), z1 = ddiv(dsub(hi, og), dg);
            zl = z0 < z1 ? z0 : z1;
            zh = z0 < z1 ? z1 : z0;
        } else {
            const bool inside = og >= lo && og <= hi;
            zl = inside ? -INFINITY : INFINITY;
            zh = inside ? INFINITY : -INFINITY;
        }
        z_in = zl > z_in ? zl : z_in;
        z_out = zh < z_out ? zh : z_out;
    }
    double kf = dsub(ceil(ddiv(dsub(z_in, P.z_near), P.step)), 1.0);
    kf = kf > 0.0 ? kf : 0.0;
    const double kcap = dadd(floor(ddiv(dsub(P.z_far, P.z_near), P.step)), 1.0);
    double kl = dadd(floor(ddiv(dsub(z_out, P.z_near), P.step)), 1.0);
    kl = kl < kcap ? kl : kcap;
    if (!(z_in <= z_out) || kl < kf) {
        *k0 = 1; *k1 = 0;
        return;
    }
    *k0 = (int64_t)kf; *k1 = (int64_t)kl;
}

// Steps 1-2: whether the sample of pixel (r, c) at camera depth z is valid, its value D and, when `n` is not null, its
// gradient (per grid unit).
DFB_HDN bool raycast_sample(const RaycastParams& P, const double* Kinv, const double* lw, const float* tsdf, const float* weight,
                            int r, int c, double z, double* D, double* n) {
    double p[3], f[3], gn[3];
    int i[3];
    if (!track_point_cell(Kinv, lw, P.center, P.scale, P.half, P.rx, P.ry, P.rz, r, c, z, p, i, f)) return false;
    return track_cell_value(tsdf, weight, P.ry, P.rz, P.scale, P.tdist, i, f, D, n ? n : gn);
}

// Steps 1-5 for the ray of pixel (r, c) of the view with inverse intrinsics Kinv and pose lw (world -> camera): writes the
// pixel's depth (-float32(z*), 0 = no hit) and normal (world frame, 0 = no hit or zero gradient).
DFB_HDN void raycast_ray(const RaycastParams& P, const double* Kinv, const double* lw, const float* tsdf, const float* weight,
                         int r, int c, float* depth, float* normal) {
    *depth = 0.0f;
    normal[0] = normal[1] = normal[2] = 0.0f;
    int64_t k0, k1;
    raycast_clip(P, Kinv, lw, r, c, &k0, &k1);
    bool prev_ok = false, hit = false;
    double prev_d = 0.0, prev_z = 0.0, d_hi = 0.0;
    for (int64_t k = k0; k <= k1; ++k) {
        const double z = dadd(P.z_near, dmul((double)k, P.step));
        if (!(z <= P.z_far)) break;
        double D = 0.0;
        const bool ok = raycast_sample(P, Kinv, lw, tsdf, weight, r, c, z, &D, nullptr);
        if (ok && prev_ok) {
            if (prev_d > 0.0 && D <= 0.0) { hit = true; d_hi = D; break; }
            if (prev_d < 0.0 && D >= 0.0) break;                  // back face: the ray ends with no hit
        }
        prev_ok = ok; prev_d = D; prev_z = z;
    }
    if (!hit) return;
    const double zs = dadd(prev_z, dmul(P.step, ddiv(prev_d, dsub(prev_d, d_hi))));
    double D, n[3];
    if (!raycast_sample(P, Kinv, lw, tsdf, weight, r, c, zs, &D, n)) return;
    *depth = -(float)zs;
    const double nn = dadd(dadd(dmul(n[0], n[0]), dmul(n[1], n[1])), dmul(n[2], n[2]));
    if (nn == 0.0) return;
    const double len = dsqrt(nn);
    for (int k = 0; k < 3; ++k) normal[k] = (float)ddiv(n[k], len);
}

}  // namespace dfb
