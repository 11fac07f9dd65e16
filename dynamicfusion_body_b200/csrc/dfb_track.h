// dfb_track.h -- per-pixel arithmetic of rigid point-to-TSDF tracking (csrc/track.cu, include/dfb.h dfb_track_normal_eq).
//
// The definition is oracle/track.py; every float64 operation below is written in its order with the explicit-rounding helpers
// of dfb_math.h, so the device kernel and the test suite's host build both reproduce the gate, the residual and the Jacobian
// of every pixel bit for bit.  Only the sums over pixels differ in their order of addition.
#pragma once
#include "dfb_math.h"
#include "dfb_require.h"

namespace dfb {

// H upper triangle (21), g (6), robust cost, pixel count
#define DFB_TRACK_SUMS 29

// One frame against one whole volume: the camera (Kinv, lw = [R|t] world -> camera), the grid (world point p lies at grid
// coordinate (p - center) / scale + half, half = tsdf_res / 2), the gate (tdist) and the Huber threshold (delta).
struct TrackParams {
    double Kinv[9], lw[12], center[3];
    double scale, half, tdist, delta;
    int rows, cols, stride, rows_s, cols_s;   // rows_s x cols_s sampled pixels (r, c) = (stride * i, stride * j)
    int rx, ry, rz;
};

// The checks of dfb_track_normal_eq other than its workspace's, and the block of the call.
inline int build_track(TrackParams& P, const dfb_volume* vol, int tsdf_res, double scale, const double* center, const float* depth,
                       int rows, int cols, const double* K, const double* Kinv, const double* lw34, int stride, double tdist,
                       double delta, const double* out29) {
    DFB_REQUIRE(vol && center && depth && K && Kinv && lw34 && out29, "null pointer");
    DFB_REQUIRE(vol->tsdf && vol->weight, "null pointer (volume)");
    DFB_REQUIRE(vol->rx >= 2 && vol->ry >= 2 && vol->rz >= 2, "volume %dx%dx%d is smaller than one cell", vol->rx, vol->ry, vol->rz);
    DFB_REQUIRE(vol->x0 == 0 && vol->x1 == vol->rx, "slab [%d,%d) of %d planes: tracking needs the whole volume (trilinear cells "
                "span neighbouring planes)", vol->x0, vol->x1, vol->rx);
    DFB_REQUIRE(tsdf_res >= 1, "tsdf_res=%d must be positive", tsdf_res);
    DFB_REQUIRE(rows >= 1 && cols >= 1, "depth map %dx%d is empty", rows, cols);
    DFB_REQUIRE(stride >= 1, "stride=%d must be >= 1", stride);
    DFB_REQUIRE(scale > 0, "scale must be positive");
    DFB_REQUIRE(tdist > 0, "truncation distance must be positive");
    DFB_REQUIRE(delta > 0, "Huber threshold must be positive");
    for (int i = 0; i < 9; ++i) P.Kinv[i] = Kinv[i];
    for (int i = 0; i < 12; ++i) P.lw[i] = lw34[i];
    for (int i = 0; i < 3; ++i) P.center[i] = center[i];
    P.scale = scale; P.half = tsdf_res / 2.0; P.tdist = tdist; P.delta = delta;
    P.rows = rows; P.cols = cols; P.stride = stride;
    P.rows_s = (rows + stride - 1) / stride; P.cols_s = (cols + stride - 1) / stride;
    P.rx = vol->rx; P.ry = vol->ry; P.rz = vol->rz;
    return DFB_OK;
}

// Steps 2-4 of oracle/track.py for pixel (r, c) at camera depth z: camera point x = Kinv [c z, r z, z], world point
// p = R^T (x - t) for lw = [R|t], grid coordinate g = (p - center) / scale + half, cell i = floor(g) and fraction f = g - i.
// Returns false when the cell lies outside 0 <= i <= r - 2 on some axis.  Shared with the raycaster (dfb_raycast.h), so a
// raycast depth back-projects exactly as the tracker back-projects it.
DFB_HDN bool track_point_cell(const double* Kinv, const double* lw, const double* center, double scale, double half, int rx, int ry,
                              int rz, int r, int c, double z, double* p, int* i, double* f) {
    const double a = dmul((double)c, z), b = dmul((double)r, z);
    double x[3], e[3];
    for (int k = 0; k < 3; ++k) x[k] = dot3_ref(Kinv + 3 * k, a, b, z);
    for (int k = 0; k < 3; ++k) e[k] = dsub(x[k], lw[4 * k + 3]);
    for (int k = 0; k < 3; ++k) p[k] = dadd(dadd(dmul(lw[k], e[0]), dmul(lw[4 + k], e[1])), dmul(lw[8 + k], e[2]));
    const int R[3] = {rx, ry, rz};
    for (int k = 0; k < 3; ++k) {
        const double g = dadd(ddiv(dsub(p[k], center[k]), scale), half);
        const double fl = floor(g);
        if (!(fl >= 0.0 && fl <= (double)(R[k] - 2))) return false;
        i[k] = (int)fl;
        f[k] = dsub(g, fl);
    }
    return true;
}

// Steps 5-6 for cell i at fraction f of a (rx, ry, rz) volume: false unless every one of the 8 corners has weight > 0 and
// |tsdf| * scale < tdist (the first failing corner decides), else D, the standard trilinear interpolant (along z, then y,
// then x), and n = grad D per grid unit.
DFB_HDN bool track_cell_value(const float* tsdf, const float* weight, int ry, int rz, double scale, double tdist, const int* i,
                              const double* f, double* D, double* n) {
    // corners v[dx][dy][dz]; every one observed and inside the truncation band
    double v[2][2][2];
    for (int dx = 0; dx < 2; ++dx)
        for (int dy = 0; dy < 2; ++dy)
            for (int dz = 0; dz < 2; ++dz) {
                const int64_t o = ((int64_t)(i[0] + dx) * ry + (i[1] + dy)) * rz + (i[2] + dz);
                const double t = (double)tsdf[o];
                if (!((double)weight[o] > 0.0) || !(dmul(fabs(t), scale) < tdist)) return false;
                v[dx][dy][dz] = t;
            }
    const double ix = dsub(1.0, f[0]), iy = dsub(1.0, f[1]), iz = dsub(1.0, f[2]);
    // along z, then y, then x; the gradient of the same interpolant alongside
    double ez[2][2], gz[2][2], ey[2], gy[2], gzy[2];
    for (int dx = 0; dx < 2; ++dx)
        for (int dy = 0; dy < 2; ++dy) {
            ez[dx][dy] = dadd(dmul(v[dx][dy][0], iz), dmul(v[dx][dy][1], f[2]));
            gz[dx][dy] = dsub(v[dx][dy][1], v[dx][dy][0]);
        }
    for (int dx = 0; dx < 2; ++dx) {
        ey[dx] = dadd(dmul(ez[dx][0], iy), dmul(ez[dx][1], f[1]));
        gy[dx] = dsub(ez[dx][1], ez[dx][0]);
        gzy[dx] = dadd(dmul(gz[dx][0], iy), dmul(gz[dx][1], f[1]));
    }
    *D = dadd(dmul(ey[0], ix), dmul(ey[1], f[0]));
    n[0] = dsub(ey[1], ey[0]);
    n[1] = dadd(dmul(gy[0], ix), dmul(gy[1], f[0]));
    n[2] = dadd(dmul(gzy[0], ix), dmul(gzy[1], f[0]));
    return true;
}

// Steps 1-7 of oracle/track.py for pixel (r, c): returns false when the pixel does not contribute, else its residual
// rho = scale * D (world units) and J = [grad D, p x grad D], the derivative of rho under p -> p + tau + omega x p.
DFB_HDN bool track_pixel(const TrackParams& P, const float* tsdf, const float* weight, const float* depth, int r, int c,
                         double* rho, double* J) {
    const double z = -1.0 * (double)depth[(int64_t)r * P.cols + c];
    if (!(z > 0.0)) return false;
    double p[3], f[3], n[3], D;
    int i[3];
    if (!track_point_cell(P.Kinv, P.lw, P.center, P.scale, P.half, P.rx, P.ry, P.rz, r, c, z, p, i, f)) return false;
    if (!track_cell_value(tsdf, weight, P.ry, P.rz, P.scale, P.tdist, i, f, &D, n)) return false;
    *rho = dmul(P.scale, D);
    J[0] = n[0]; J[1] = n[1]; J[2] = n[2];
    J[3] = dsub(dmul(p[1], n[2]), dmul(p[2], n[1]));
    J[4] = dsub(dmul(p[2], n[0]), dmul(p[0], n[2]));
    J[5] = dsub(dmul(p[0], n[1]), dmul(p[1], n[0]));
    return true;
}

// The 29 terms of one contributing pixel: Huber weight w = min(1, delta / |rho|), H_ij = (w J_i) J_j for i <= j (row-major upper
// triangle), g_i = (w J_i) rho, cost 0.5 rho^2 (|rho| <= delta) or delta (|rho| - 0.5 delta), count 1.
DFB_HDN void track_terms(double rho, const double* J, double delta, double* out) {
    const double ar = fabs(rho);
    const bool in = ar <= delta;
    const double w = in ? 1.0 : ddiv(delta, ar);
    double wJ[6];
    for (int k = 0; k < 6; ++k) wJ[k] = dmul(w, J[k]);
    int o = 0;
    for (int a = 0; a < 6; ++a)
        for (int b = a; b < 6; ++b) out[o++] = dmul(wJ[a], J[b]);
    for (int a = 0; a < 6; ++a) out[21 + a] = dmul(wJ[a], rho);
    out[27] = in ? dmul(0.5, dmul(rho, rho)) : dmul(delta, dsub(ar, dmul(0.5, delta)));
    out[28] = 1.0;
}

}  // namespace dfb
