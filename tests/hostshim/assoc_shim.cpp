// assoc_shim.cpp -- TEST INFRASTRUCTURE ONLY.  The loop of corr_projective_kernel (dynamicfusion_body_b200/csrc/graph.cu) with
// HOST pointers, around the very same per-vertex function (csrc/dfb_math.h assoc_projective_ref), so that the CPU test-suite
// can check projective data association against the oracle (oracle/assoc.py) on a box that has no GPU.  Build with
// -ffp-contract=off.  The product never loads this library.
#include "../../include/dfb.h"
#include "../../dynamicfusion_body_b200/csrc/dfb_math.h"

using namespace dfb;

extern "C" int as_corr_projective(const double* warped_pts, const double* warped_normals, int64_t m, const dfb_views* views,
                                  double max_distance, double min_normal_dot, int32_t* view, double* cost, double* corr) {
    const float* depth[DFB_MAX_VIEWS];
    for (int v = 0; v < views->n_views; ++v) depth[v] = views->depth[v];
    for (int64_t t = 0; t < m; ++t)
        view[t] = assoc_projective_ref(warped_pts + 3 * t, warped_normals + 3 * t, depth, views->n_views, views->rows, views->cols, views->K,
                                       views->Kinv, views->has_extrinsics ? &views->E[0][0] : nullptr, max_distance, min_normal_dot,
                                       cost + t, corr + 3 * t);
    return DFB_OK;
}
