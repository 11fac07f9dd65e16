// raycast.cu -- depth and normal maps of the whole fused volume seen from up to DFB_MAX_VIEWS cameras, by marching every pixel's
// ray through the signed-distance field to its first zero crossing: the model's view from any pose with no surface extraction.
// Per-ray arithmetic in dfb_raycast.h (each sample through the tracker's functions of dfb_track.h), the definition
// oracle/raycast.py.
//
// raycast_kernel: one thread per ray, 16x8 pixel tiles per block so that neighbouring rays read neighbouring voxels, one grid
// plane per view.  No reduction, no atomics, no workspace: each thread writes its own pixel, so the maps are identical run to
// run and equal to the oracle's bit for bit.
#include "common.h"
#include "dfb_raycast.h"

namespace dfb {
namespace {

constexpr int RAY_TX = 16, RAY_TY = 8;

__global__ void __launch_bounds__(RAY_TX * RAY_TY) raycast_kernel(const RaycastParams P, const RaycastCams cams,
                                                                  const float* __restrict__ tsdf, const float* __restrict__ weight,
                                                                  float* __restrict__ depth, float* __restrict__ normal) {
    // the view's Kinv and pose staged in shared memory: the per-ray function reads them through pointers
    __shared__ double sKinv[9], sE[12];
    const int v = blockIdx.z, t = threadIdx.y * RAY_TX + threadIdx.x;
    if (t < 9) sKinv[t] = cams.Kinv[t];
    else if (t < 21) sE[t - 9] = cams.E[12 * v + (t - 9)];
    __syncthreads();
    const int c = blockIdx.x * RAY_TX + threadIdx.x, r = blockIdx.y * RAY_TY + threadIdx.y;
    if (r >= P.rows || c >= P.cols) return;
    const int64_t o = ((int64_t)v * P.rows + r) * P.cols + c;
    raycast_ray(P, sKinv, sE, tsdf, weight, r, c, depth + o, normal + 3 * o);
}

}  // namespace
}  // namespace dfb

using namespace dfb;

extern "C" int dfb_raycast(const dfb_volume* vol, int tsdf_res, double scale, const double center[3], const dfb_views* views,
                           double tdist, double step, double z_near, double z_far, float* depth, float* normal, dfb_stream_t stream) {
    RaycastParams P;
    RaycastCams cams;
    if (int r = build_raycast(P, cams, vol, tsdf_res, scale, center, views, tdist, step, z_near, z_far, depth, normal)) return r;
    const dim3 block(RAY_TX, RAY_TY), grid((views->cols + RAY_TX - 1) / RAY_TX, (views->rows + RAY_TY - 1) / RAY_TY, views->n_views);
    raycast_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(P, cams, vol->tsdf, vol->weight, depth, normal);
    DFB_LAUNCH_CHECK("raycast_kernel");
    return DFB_OK;
}
