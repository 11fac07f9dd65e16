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

struct RaycastCams {
    double Kinv[9];
    double E[DFB_MAX_VIEWS * 12];
};

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
    RaycastParams P;
    for (int i = 0; i < 3; ++i) P.center[i] = center[i];
    P.scale = scale; P.half = tsdf_res / 2.0; P.tdist = tdist; P.step = step; P.z_near = z_near; P.z_far = z_far;
    P.rows = views->rows; P.cols = views->cols; P.rx = vol->rx; P.ry = vol->ry; P.rz = vol->rz;
    RaycastCams cams;
    for (int i = 0; i < 9; ++i) cams.Kinv[i] = views->Kinv[i];
    for (int v = 0; v < views->n_views; ++v)
        for (int i = 0; i < 12; ++i) cams.E[12 * v + i] = views->has_extrinsics ? views->E[v][i] : (i % 5 == 0 ? 1.0 : 0.0);
    const dim3 block(RAY_TX, RAY_TY), grid((views->cols + RAY_TX - 1) / RAY_TX, (views->rows + RAY_TY - 1) / RAY_TY, views->n_views);
    raycast_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(P, cams, vol->tsdf, vol->weight, depth, normal);
    DFB_LAUNCH_CHECK("raycast_kernel");
    return DFB_OK;
}
