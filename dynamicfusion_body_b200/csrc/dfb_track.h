// dfb_track.h -- per-pixel arithmetic of rigid point-to-TSDF tracking (csrc/track.cu, include/dfb.h dfb_track_normal_eq).
//
// The definition is oracle/track.py; every float64 operation below is written in its order with the explicit-rounding helpers
// of dfb_math.h, so the device kernel and the test suite's host build (tests/track_shim.py) both reproduce the gate, the
// residual and the Jacobian of every pixel bit for bit.  Only the sums over pixels differ in their order of addition.
#pragma once
#include "dfb_math.h"

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

// Steps 1-7 of oracle/track.py for pixel (r, c): returns false when the pixel does not contribute, else its residual
// rho = scale * D (world units) and J = [grad D, p x grad D], the derivative of rho under p -> p + tau + omega x p.
DFB_HDN bool track_pixel(const TrackParams& P, const float* tsdf, const float* weight, const float* depth, int r, int c,
                         double* rho, double* J) {
    const double z = -1.0 * (double)depth[(int64_t)r * P.cols + c];
    if (!(z > 0.0)) return false;
    const double a = dmul((double)c, z), b = dmul((double)r, z);
    double x[3], e[3], p[3], g[3], f[3];
    int i[3];
    for (int k = 0; k < 3; ++k) x[k] = dot3_ref(P.Kinv + 3 * k, a, b, z);
    for (int k = 0; k < 3; ++k) e[k] = dsub(x[k], P.lw[4 * k + 3]);
    for (int k = 0; k < 3; ++k) p[k] = dadd(dadd(dmul(P.lw[k], e[0]), dmul(P.lw[4 + k], e[1])), dmul(P.lw[8 + k], e[2]));
    const int R[3] = {P.rx, P.ry, P.rz};
    for (int k = 0; k < 3; ++k) {
        g[k] = dadd(ddiv(dsub(p[k], P.center[k]), P.scale), P.half);
        const double fl = floor(g[k]);
        if (!(fl >= 0.0 && fl <= (double)(R[k] - 2))) return false;
        i[k] = (int)fl;
        f[k] = dsub(g[k], fl);
    }
    // corners v[dx][dy][dz]; every one observed and inside the truncation band
    double v[2][2][2];
    for (int dx = 0; dx < 2; ++dx)
        for (int dy = 0; dy < 2; ++dy)
            for (int dz = 0; dz < 2; ++dz) {
                const int64_t o = ((int64_t)(i[0] + dx) * P.ry + (i[1] + dy)) * P.rz + (i[2] + dz);
                const double t = (double)tsdf[o];
                if (!((double)weight[o] > 0.0) || !(dmul(fabs(t), P.scale) < P.tdist)) return false;
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
    const double D = dadd(dmul(ey[0], ix), dmul(ey[1], f[0]));
    const double n[3] = {dsub(ey[1], ey[0]), dadd(dmul(gy[0], ix), dmul(gy[1], f[0])), dadd(dmul(gzy[0], ix), dmul(gzy[1], f[0]))};
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
