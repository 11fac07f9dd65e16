// track.cu -- normal equations of rigid point-to-TSDF tracking: every sampled pixel of a depth frame, back-projected and moved
// to the world by the current pose, is compared with the fused signed-distance field it should lie on (the residual is the
// interpolated distance itself), so a camera pose follows from a depth frame and the volume with no surface extraction and no
// correspondence search.  Per-pixel arithmetic in dfb_track.h, the definition oracle/track.py.
//
//   1. track_pixel_kernel, one thread per sampled pixel: gate, residual, Jacobian and the pixel's 29 terms; the block adds them
//      with warp shuffles and a fixed pass over its warps into one partial row of the caller's workspace (and writes the
//      residual map when asked);
//   2. track_sum_kernel, one block: adds the partial rows column by column in a fixed order.
// No atomics: the sums of a call are identical run to run, so the host's Levenberg-Marquardt trajectory is deterministic.
#include "common.h"
#include "dfb_track.h"

namespace dfb {
namespace {

constexpr int TRACK_THREADS = 256;
constexpr int TRACK_WARPS = TRACK_THREADS / 32;

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) x = dadd(x, __shfl_down_sync(0xffffffffu, x, off));
    return x;
}

__global__ void __launch_bounds__(TRACK_THREADS) track_pixel_kernel(const TrackParams P, const float* __restrict__ tsdf,
                                                                    const float* __restrict__ weight, const float* __restrict__ depth,
                                                                    double* __restrict__ partial, double* __restrict__ residual) {
    __shared__ double sh[TRACK_WARPS][DFB_TRACK_SUMS];
    const int64_t s = (int64_t)blockIdx.x * TRACK_THREADS + threadIdx.x;
    double t[DFB_TRACK_SUMS];
#pragma unroll
    for (int k = 0; k < DFB_TRACK_SUMS; ++k) t[k] = 0.0;
    if (s < (int64_t)P.rows_s * P.cols_s) {
        const int i = (int)(s / P.cols_s), j = (int)(s - (int64_t)i * P.cols_s);
        double rho, J[6];
        const bool ok = track_pixel(P, tsdf, weight, depth, i * P.stride, j * P.stride, &rho, J);
        if (ok) track_terms(rho, J, P.delta, t);
        if (residual) residual[s] = ok ? rho : __longlong_as_double(0x7ff8000000000000ll);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < DFB_TRACK_SUMS; ++k) {
        const double x = warp_sum(t[k]);
        if (lane == 0) sh[warp][k] = x;
    }
    __syncthreads();
    if (threadIdx.x < DFB_TRACK_SUMS) {
        double acc = sh[0][threadIdx.x];
        for (int w = 1; w < TRACK_WARPS; ++w) acc = dadd(acc, sh[w][threadIdx.x]);
        partial[(int64_t)blockIdx.x * DFB_TRACK_SUMS + threadIdx.x] = acc;
    }
}

__global__ void __launch_bounds__(TRACK_THREADS) track_sum_kernel(const double* __restrict__ partial, int n_blocks,
                                                                  double* __restrict__ out) {
    __shared__ double sh[TRACK_WARPS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = 0; k < DFB_TRACK_SUMS; ++k) {
        double acc = 0.0;
        for (int b = threadIdx.x; b < n_blocks; b += TRACK_THREADS) acc = dadd(acc, partial[(int64_t)b * DFB_TRACK_SUMS + k]);
        acc = warp_sum(acc);
        if (lane == 0) sh[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double x = sh[0];
            for (int w = 1; w < TRACK_WARPS; ++w) x = dadd(x, sh[w]);
            out[k] = x;
        }
        __syncthreads();
    }
}

int64_t track_blocks(int rows, int cols, int stride) {
    const int64_t n = (int64_t)((rows + stride - 1) / stride) * ((cols + stride - 1) / stride);
    return (n + TRACK_THREADS - 1) / TRACK_THREADS;
}

}  // namespace
}  // namespace dfb

using namespace dfb;

extern "C" int64_t dfb_track_workspace_doubles(int rows, int cols, int stride) {
    if (rows < 1 || cols < 1 || stride < 1) return -1;
    return track_blocks(rows, cols, stride) * DFB_TRACK_SUMS;
}

extern "C" int dfb_track_normal_eq(const dfb_volume* vol, int tsdf_res, double scale, const double center[3], const float* depth,
                                   int rows, int cols, const double K[9], const double Kinv[9], const double lw34[12], int stride,
                                   double tdist, double delta, double* workspace, int64_t workspace_doubles, double* out29,
                                   double* residual, dfb_stream_t stream) {
    DFB_REQUIRE(workspace, "null pointer");
    TrackParams P;
    if (int r = build_track(P, vol, tsdf_res, scale, center, depth, rows, cols, K, Kinv, lw34, stride, tdist, delta, out29)) return r;
    const int64_t need = dfb_track_workspace_doubles(rows, cols, stride);
    DFB_REQUIRE(workspace_doubles >= need, "workspace of %lld doubles is smaller than the %lld dfb_track_workspace_doubles asks for",
                (long long)workspace_doubles, (long long)need);
    const cudaStream_t s = (cudaStream_t)stream;
    const int64_t blocks = track_blocks(rows, cols, stride);
    track_pixel_kernel<<<(unsigned)blocks, TRACK_THREADS, 0, s>>>(P, vol->tsdf, vol->weight, depth, workspace, residual);
    DFB_LAUNCH_CHECK("track_pixel_kernel");
    track_sum_kernel<<<1, TRACK_THREADS, 0, s>>>(workspace, (int)blocks, out29);
    DFB_LAUNCH_CHECK("track_sum_kernel");
    return DFB_OK;
}
