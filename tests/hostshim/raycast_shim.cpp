// raycast_shim.cpp -- TEST INFRASTRUCTURE ONLY.  dfb_raycast (dynamicfusion_body_b200/csrc/raycast.cu) as a serial loop over
// HOST pointers, around the very same set-up and per-ray functions (csrc/dfb_raycast.h), so that the CPU test-suite can check the
// raycaster's arithmetic against the oracle (oracle/raycast.py) on a box that has no GPU.  Every pixel is independent, so the
// maps agree bit for bit.  Build with -ffp-contract=off.  The product never loads this library.
#include "../../include/dfb.h"
#include "../../dynamicfusion_body_b200/csrc/dfb_raycast.h"

using namespace dfb;

// depth [V][rows][cols], normal [V][rows][cols][3]
extern "C" int hs_raycast(const dfb_volume* vol, int tsdf_res, double scale, const double* center, const dfb_views* views, double tdist,
                          double step, double z_near, double z_far, float* depth, float* normal) {
    RaycastParams P;
    RaycastCams cams;
    if (int r = build_raycast(P, cams, vol, tsdf_res, scale, center, views, tdist, step, z_near, z_far, depth, normal)) return r;
    for (int v = 0; v < views->n_views; ++v)
        for (int r = 0; r < P.rows; ++r)
            for (int c = 0; c < P.cols; ++c) {
                const int64_t o = ((int64_t)v * P.rows + r) * P.cols + c;
                raycast_ray(P, cams.Kinv, cams.E + 12 * v, vol->tsdf, vol->weight, r, c, depth + o, normal + 3 * o);
            }
    return DFB_OK;
}
