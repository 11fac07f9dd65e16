// dfb_render.h -- per-face and per-pixel arithmetic of the z-buffer rasteriser (csrc/render.cu, include/dfb.h dfb_render).
//
// The definition is oracle/render.py; every float64 operation below is written in its order with the explicit-rounding
// helpers of dfb_math.h, so the device kernels and the test suite's host build both reproduce it bit for bit.
// The winner of a pixel is the smallest 64-bit key (float32 depth bits << 32 | face id): an atomicMin on the device, a plain
// min on the host, and the result does not depend on the order in which faces arrive.
#pragma once
#include <string.h>

#include "dfb_math.h"
#include "dfb_require.h"

namespace dfb {

// z-buffer value of a pixel no face covers
#define DFB_RENDER_EMPTY 0xFFFFFFFFFFFFFFFFull

// A face projected into one view: pixel coordinates and inverse camera depths of its vertices, its signed doubled area and
// its inclusive pixel box (non-empty when render_face_setup returns true).
struct RenderFace {
    double x[3], y[3], w[3];
    double A;
    int c0, c1, r0, r1;
};

// The cameras of one call: intrinsics, one world -> camera extrinsic per view when has_e, and the image size.
struct RenderCams {
    double K[9];
    double E[DFB_MAX_VIEWS * 12];
    int n_views, rows, cols, has_e;
};

// The checks of dfb_render other than its workspace's, and the camera block of the call.
inline int build_render(RenderCams& cams, const double* pts, int64_t n_pts, const int32_t* faces, int64_t n_faces, const dfb_views* views,
                        const float* depth, const int32_t* face, const float* normal) {
    DFB_REQUIRE(views && depth && face && normal && (pts || n_pts == 0) && (faces || n_faces == 0), "null pointer");
    DFB_REQUIRE(n_pts >= 0 && n_faces >= 0, "negative count");
    DFB_REQUIRE(n_faces <= INT32_MAX, "n_faces=%lld exceeds the int32 face ids", (long long)n_faces);
    DFB_REQUIRE(views->n_views >= 1 && views->n_views <= DFB_MAX_VIEWS, "n_views=%d out of range [1,%d]", views->n_views, DFB_MAX_VIEWS);
    DFB_REQUIRE(views->rows >= 1 && views->cols >= 1, "image %dx%d is empty", views->rows, views->cols);
    for (int i = 0; i < 9; ++i) cams.K[i] = views->K[i];
    for (int v = 0; v < views->n_views; ++v)
        for (int i = 0; i < 12; ++i) cams.E[12 * v + i] = views->E[v][i];
    cams.n_views = views->n_views; cams.rows = views->rows; cams.cols = views->cols; cams.has_e = views->has_extrinsics ? 1 : 0;
    return DFB_OK;
}

// E(a, b, p) = (xb - xa)(py - ya) - (yb - ya)(px - xa), each product rounded
DFB_HD double render_edge(double xa, double ya, double xb, double yb, double px, double py) {
    return dsub(dmul(dsub(xb, xa), dsub(py, ya)), dmul(dsub(yb, ya), dsub(px, xa)));
}

// Steps 1-5 of oracle/render.py for face `t` in the view with intrinsics K (row-major 3x3) and extrinsic Ev (row-major 3x4,
// nullptr = none).  Returns false when the face is culled or its box holds no pixel of the rows x cols image.
DFB_HDN bool render_face_setup(const double* pts, int64_t n_pts, const int32_t* faces, int64_t t, const double* K, const double* Ev,
                               int rows, int cols, RenderFace* f) {
    int32_t id[3];
    for (int i = 0; i < 3; ++i) {
        id[i] = faces[3 * t + i];
        if (id[i] < 0 || (int64_t)id[i] >= n_pts) return false;
    }
    for (int i = 0; i < 3; ++i) {
        const double* P = pts + 3 * (int64_t)id[i];
        double l[3];
        for (int r = 0; r < 3; ++r) l[r] = Ev ? dot4_ref(Ev + 4 * r, P[0], P[1], P[2], 1.0) : P[r];
        if (!(l[2] > 0.0)) return false;
        const double q0 = dot3_ref(K, l[0], l[1], l[2]);
        const double q1 = dot3_ref(K + 3, l[0], l[1], l[2]);
        const double q2 = dot3_ref(K + 6, l[0], l[1], l[2]);
        f->x[i] = ddiv(q0, q2);
        f->y[i] = ddiv(q1, q2);
        f->w[i] = ddiv(1.0, l[2]);
    }
    f->A = render_edge(f->x[0], f->y[0], f->x[1], f->y[1], f->x[2], f->y[2]);
    if (f->A == 0.0 || !isfinite(f->A)) return false;
    const double cl = fmax(ceil(fmin(fmin(f->x[0], f->x[1]), f->x[2])), 0.0);
    const double ch = fmin(floor(fmax(fmax(f->x[0], f->x[1]), f->x[2])), (double)(cols - 1));
    const double rl = fmax(ceil(fmin(fmin(f->y[0], f->y[1]), f->y[2])), 0.0);
    const double rh = fmin(floor(fmax(fmax(f->y[0], f->y[1]), f->y[2])), (double)(rows - 1));
    if (!(cl <= ch && rl <= rh)) return false;
    f->c0 = (int)cl; f->c1 = (int)ch; f->r0 = (int)rl; f->r1 = (int)rh;
    return true;
}

// Steps 6-8 at the centre of pixel (r, c): returns false when the face does not cover it, else its key.
DFB_HDN bool render_pixel_key(const RenderFace& f, int r, int c, uint32_t t, uint64_t* key) {
    const double px = (double)c, py = (double)r;
    const double e0 = render_edge(f.x[1], f.y[1], f.x[2], f.y[2], px, py);
    const double e1 = render_edge(f.x[2], f.y[2], f.x[0], f.y[0], px, py);
    const double e2 = render_edge(f.x[0], f.y[0], f.x[1], f.y[1], px, py);
    const bool in = f.A > 0.0 ? (e0 >= 0.0 && e1 >= 0.0 && e2 >= 0.0) : (e0 <= 0.0 && e1 <= 0.0 && e2 <= 0.0);
    if (!in) return false;
    const double inv = ddiv(dadd(dadd(dmul(e0, f.w[0]), dmul(e1, f.w[1])), dmul(e2, f.w[2])), f.A);
    if (!(inv > 0.0)) return false;
#if defined(__CUDA_ARCH__)
    const float zf = __double2float_rn(ddiv(1.0, inv));
    const uint32_t bits = __float_as_uint(zf);
#else
    const float zf = (float)ddiv(1.0, inv);
    uint32_t bits;
    memcpy(&bits, &zf, 4);
#endif
    *key = ((uint64_t)bits << 32) | (uint64_t)t;
    return true;
}

// Unit normal of face (a, b, c) in the frame of pts: n = (Pb - Pa) x (Pc - Pa) / sqrt(n.n), rounded to float32; 0 when n.n == 0.
DFB_HDN void render_face_normal(const double* pts, const int32_t* tri, float* out) {
    const double* Pa = pts + 3 * (int64_t)tri[0];
    const double* Pb = pts + 3 * (int64_t)tri[1];
    const double* Pc = pts + 3 * (int64_t)tri[2];
    const double u[3] = {dsub(Pb[0], Pa[0]), dsub(Pb[1], Pa[1]), dsub(Pb[2], Pa[2])};
    const double v[3] = {dsub(Pc[0], Pa[0]), dsub(Pc[1], Pa[1]), dsub(Pc[2], Pa[2])};
    const double n[3] = {dsub(dmul(u[1], v[2]), dmul(u[2], v[1])), dsub(dmul(u[2], v[0]), dmul(u[0], v[2])),
                         dsub(dmul(u[0], v[1]), dmul(u[1], v[0]))};
    const double nn = dot3_ref(n, n[0], n[1], n[2]);
    if (nn == 0.0) { out[0] = out[1] = out[2] = 0.0f; return; }
    const double s = dsqrt(nn);
    for (int i = 0; i < 3; ++i) out[i] = (float)ddiv(n[i], s);
}

// Decodes one z-buffer word into the outputs of its pixel (depth = -zf, face id, face normal; 0 / -1 / 0 when empty).
DFB_HDN void render_resolve(uint64_t key, const double* pts, const int32_t* faces, float* depth, int32_t* face, float* normal) {
    if (key == DFB_RENDER_EMPTY) {
        *depth = 0.0f; *face = -1;
        normal[0] = normal[1] = normal[2] = 0.0f;
        return;
    }
    const uint32_t bits = (uint32_t)(key >> 32);
    const int32_t t = (int32_t)(uint32_t)key;
#if defined(__CUDA_ARCH__)
    const float zf = __uint_as_float(bits);
#else
    float zf;
    memcpy(&zf, &bits, 4);
#endif
    *depth = -zf;
    *face = t;
    render_face_normal(pts, faces + 3 * (int64_t)t, normal);
}

}  // namespace dfb
