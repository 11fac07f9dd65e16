// raycast_shim.cpp -- TEST INFRASTRUCTURE ONLY.  dfb_raycast (dynamicfusion_body_b200/csrc/raycast.cu) as a serial loop over
// HOST pointers, around the very same per-ray function (csrc/dfb_raycast.h), so that the CPU test-suite can check the
// raycaster's arithmetic against the oracle (oracle/raycast.py) on a box that has no GPU.  Every pixel is independent, so the
// maps agree bit for bit.  Build with -ffp-contract=off.  The product never loads this library.
#include "../../include/dfb.h"
#include "../../dynamicfusion_body_b200/csrc/dfb_raycast.h"

using namespace dfb;

// depth [V][rows][cols], normal [V][rows][cols][3]; the arguments are assumed valid (dfb_raycast checks them).
extern "C" int rc_raycast(const float* tsdf, const float* weight, int rx, int ry, int rz, int tsdf_res, double scale,
                          const double* center, const dfb_views* views, double tdist, double step, double z_near, double z_far,
                          float* depth, float* normal) {
    RaycastParams P;
    for (int i = 0; i < 3; ++i) P.center[i] = center[i];
    P.scale = scale; P.half = tsdf_res / 2.0; P.tdist = tdist; P.step = step; P.z_near = z_near; P.z_far = z_far;
    P.rows = views->rows; P.cols = views->cols; P.rx = rx; P.ry = ry; P.rz = rz;
    for (int v = 0; v < views->n_views; ++v) {
        double lw[12];
        for (int i = 0; i < 12; ++i) lw[i] = views->has_extrinsics ? views->E[v][i] : (i % 5 == 0 ? 1.0 : 0.0);
        for (int r = 0; r < P.rows; ++r)
            for (int c = 0; c < P.cols; ++c) {
                const int64_t o = ((int64_t)v * P.rows + r) * P.cols + c;
                raycast_ray(P, views->Kinv, lw, tsdf, weight, r, c, depth + o, normal + 3 * o);
            }
    }
    return DFB_OK;
}
