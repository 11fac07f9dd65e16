// track_shim.cpp -- TEST INFRASTRUCTURE ONLY.  dfb_track_normal_eq (dynamicfusion_body_b200/csrc/track.cu) as a serial loop over
// HOST pointers, around the very same set-up and per-pixel functions (csrc/dfb_track.h), so that the CPU test-suite can check the
// tracker's arithmetic against the oracle (oracle/track.py) on a box that has no GPU.  The sums are added in pixel order here, in
// a tree on the device: they agree to rounding, the per-pixel values bit for bit.  Build with -ffp-contract=off.  The product
// never loads this library.
#include "../../include/dfb.h"
#include "../../dynamicfusion_body_b200/csrc/dfb_track.h"

using namespace dfb;

// dfb_track_normal_eq without its device workspace; residual [rows_s][cols_s] (NaN = no contribution) and jac [rows_s][cols_s][6]
// (0 = no contribution) of every sampled pixel.
extern "C" int hs_track_normal_eq(const dfb_volume* vol, int tsdf_res, double scale, const double* center, const float* depth, int rows,
                                  int cols, const double* K, const double* Kinv, const double* lw34, int stride, double tdist, double delta,
                                  double* out29, double* residual, double* jac) {
    TrackParams P;
    if (int r = build_track(P, vol, tsdf_res, scale, center, depth, rows, cols, K, Kinv, lw34, stride, tdist, delta, out29)) return r;
    for (int k = 0; k < DFB_TRACK_SUMS; ++k) out29[k] = 0.0;
    for (int i = 0; i < P.rows_s; ++i)
        for (int j = 0; j < P.cols_s; ++j) {
            const int64_t s = (int64_t)i * P.cols_s + j;
            double rho, J[6], t[DFB_TRACK_SUMS];
            const bool ok = track_pixel(P, vol->tsdf, vol->weight, depth, i * P.stride, j * P.stride, &rho, J);
            residual[s] = ok ? rho : NAN;
            for (int k = 0; k < 6; ++k) jac[6 * s + k] = ok ? J[k] : 0.0;
            if (!ok) continue;
            track_terms(rho, J, P.delta, t);
            for (int k = 0; k < DFB_TRACK_SUMS; ++k) out29[k] = dadd(out29[k], t[k]);
        }
    return DFB_OK;
}
