// render.cu -- z-buffer rasteriser of a triangle mesh into the depth views: depth, face-id and face-normal maps of the live
// model as the live cameras see it, with no GL context (the reference's only renderer is its GL/GLUT off-screen vertex-id and
// depth renderer, core/gl/glrender.py).  Per-face and per-pixel arithmetic in dfb_render.h, the definition oracle/render.py.
//
//   1. the caller's z-buffer is filled with all ones (no face);
//   2. raster_small_kernel, one thread per (face, view): faces whose pixel box holds at most RENDER_SMALL_PIXELS pixels are
//      rasterised by that thread, each covered pixel an atomicMin of its 64-bit key (float32 depth bits << 32 | face id);
//      larger faces are appended to a list with one warp-aggregated atomic per warp;
//   3. raster_large_kernel, one warp per listed face, lanes striding its box: any face size, up to one covering the image;
//   4. resolve_kernel, one thread per pixel: decodes the key into depth, face id and the face's normal.
// The min over keys does not depend on the order in which faces arrive, so the maps are identical run to run and equal to
// the oracle's bit for bit.  A 640x480 view's z-buffer is 2.4 MB and stays in L2.
#include "common.h"
#include "dfb_render.h"

namespace dfb {
namespace {

constexpr int RENDER_SMALL_PIXELS = 16;
constexpr int RENDER_THREADS = 256;
constexpr int RENDER_MAX_BLOCKS = 148 * 8;   // 8 blocks per SM, grid-stride beyond

// the camera block is read through pointers by the per-face function: staged in shared memory (indexing the kernel
// parameter through a pointer would make every thread copy the whole struct to its local stack)
__device__ __forceinline__ void stage_cams(const RenderCams& c, double* sK, double* sE) {
    for (int i = threadIdx.x; i < 9; i += blockDim.x) sK[i] = c.K[i];
    for (int i = threadIdx.x; i < 12 * c.n_views; i += blockDim.x) sE[i] = c.E[i];
    __syncthreads();
}

__global__ void __launch_bounds__(RENDER_THREADS) raster_small_kernel(const double* __restrict__ pts, int64_t n_pts,
                                                                      const int32_t* __restrict__ faces, int64_t n_faces, const RenderCams cams,
                                                                      unsigned long long* __restrict__ zbuf, unsigned long long* __restrict__ n_large,
                                                                      unsigned long long* __restrict__ large) {
    __shared__ double sK[9], sE[DFB_MAX_VIEWS * 12];
    stage_cams(cams, sK, sE);
    const int V = cams.n_views, lane = threadIdx.x & 31;
    const int64_t total = n_faces * V, npix = (int64_t)cams.rows * cams.cols;
    // every lane of a block runs the same number of rounds, so the ballot below always sees the full warp
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x; i0 < total; i0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = i0 + threadIdx.x;
        bool big = false;
        if (i < total) {
            const int64_t t = i / V;
            const int v = (int)(i - t * V);
            RenderFace f;
            if (render_face_setup(pts, n_pts, faces, t, sK, cams.has_e ? sE + 12 * v : nullptr, cams.rows, cams.cols, &f)) {
                const int w = f.c1 - f.c0 + 1, h = f.r1 - f.r0 + 1;
                if ((int64_t)w * h > RENDER_SMALL_PIXELS) {
                    big = true;
                } else {
                    unsigned long long* zv = zbuf + v * npix;
                    for (int r = f.r0; r <= f.r1; ++r)
                        for (int c = f.c0; c <= f.c1; ++c) {
                            uint64_t key;
                            if (render_pixel_key(f, r, c, (uint32_t)t, &key)) atomicMin(zv + (int64_t)r * cams.cols + c, (unsigned long long)key);
                        }
                }
            }
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, big);
        if (ballot) {
            const int leader = __ffs(ballot) - 1;
            unsigned long long base = 0;
            if (lane == leader) base = atomicAdd(n_large, (unsigned long long)__popc(ballot));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (big) large[base + __popc(ballot & ((1u << lane) - 1u))] = (unsigned long long)i;
        }
    }
}

__global__ void __launch_bounds__(RENDER_THREADS) raster_large_kernel(const double* __restrict__ pts, int64_t n_pts,
                                                                      const int32_t* __restrict__ faces, const RenderCams cams,
                                                                      unsigned long long* __restrict__ zbuf, const unsigned long long* __restrict__ n_large,
                                                                      const unsigned long long* __restrict__ large) {
    __shared__ double sK[9], sE[DFB_MAX_VIEWS * 12];
    stage_cams(cams, sK, sE);
    const int V = cams.n_views, lane = threadIdx.x & 31;
    const int64_t npix = (int64_t)cams.rows * cams.cols, count = (int64_t)*n_large;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t j = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < count; j += warps) {
        const int64_t i = (int64_t)large[j], t = i / V;
        const int v = (int)(i - t * V);
        RenderFace f;
        // every lane repeats the face's set-up (a handful of divisions) rather than waiting on a broadcast
        if (!render_face_setup(pts, n_pts, faces, t, sK, cams.has_e ? sE + 12 * v : nullptr, cams.rows, cams.cols, &f)) continue;
        const int64_t w = f.c1 - f.c0 + 1, area = w * (f.r1 - f.r0 + 1);
        unsigned long long* zv = zbuf + v * npix;
        for (int64_t p = lane; p < area; p += 32) {
            const int r = f.r0 + (int)(p / w), c = f.c0 + (int)(p % w);
            uint64_t key;
            if (render_pixel_key(f, r, c, (uint32_t)t, &key)) atomicMin(zv + (int64_t)r * cams.cols + c, (unsigned long long)key);
        }
    }
}

__global__ void __launch_bounds__(RENDER_THREADS) resolve_kernel(const double* __restrict__ pts, const int32_t* __restrict__ faces,
                                                                 const unsigned long long* __restrict__ zbuf, int64_t n, float* __restrict__ depth,
                                                                 int32_t* __restrict__ face, float* __restrict__ normal) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        float nrm[3];
        render_resolve((uint64_t)zbuf[p], pts, faces, depth + p, face + p, nrm);
        normal[3 * p] = nrm[0]; normal[3 * p + 1] = nrm[1]; normal[3 * p + 2] = nrm[2];
    }
}

unsigned grid_for(int64_t items) {
    const int64_t need = (items + RENDER_THREADS - 1) / RENDER_THREADS;
    return (unsigned)(need < 1 ? 1 : (need < RENDER_MAX_BLOCKS ? need : RENDER_MAX_BLOCKS));
}

}  // namespace
}  // namespace dfb

using namespace dfb;

extern "C" int64_t dfb_render_workspace_words(int64_t n_faces, int n_views, int rows, int cols) {
    if (n_faces < 0 || n_views < 1 || rows < 1 || cols < 1) return -1;
    return 1 + (int64_t)n_views * rows * cols + n_faces * n_views;
}

extern "C" int dfb_render(const double* pts, int64_t n_pts, const int32_t* faces, int64_t n_faces, const dfb_views* views,
                          uint64_t* workspace, int64_t workspace_words, float* depth, int32_t* face, float* normal,
                          dfb_stream_t stream) {
    DFB_REQUIRE(workspace, "null pointer");
    RenderCams cams;
    if (int r = build_render(cams, pts, n_pts, faces, n_faces, views, depth, face, normal)) return r;
    const int64_t need = dfb_render_workspace_words(n_faces, views->n_views, views->rows, views->cols);
    DFB_REQUIRE(workspace_words >= need, "workspace of %lld words is smaller than the %lld dfb_render_workspace_words asks for",
                (long long)workspace_words, (long long)need);
    const cudaStream_t s = (cudaStream_t)stream;
    const int64_t npix = (int64_t)views->n_views * views->rows * views->cols;
    unsigned long long* n_large = (unsigned long long*)workspace;
    unsigned long long* zbuf = n_large + 1;
    unsigned long long* large = zbuf + npix;
    DFB_CUDA(cudaMemsetAsync(n_large, 0, sizeof(unsigned long long), s));
    DFB_CUDA(cudaMemsetAsync(zbuf, 0xFF, (size_t)npix * sizeof(unsigned long long), s));
    if (n_faces > 0) {
        raster_small_kernel<<<grid_for(n_faces * views->n_views), RENDER_THREADS, 0, s>>>(pts, n_pts, faces, n_faces, cams, zbuf, n_large, large);
        DFB_LAUNCH_CHECK("raster_small_kernel");
        raster_large_kernel<<<RENDER_MAX_BLOCKS, RENDER_THREADS, 0, s>>>(pts, n_pts, faces, cams, zbuf, n_large, large);
        DFB_LAUNCH_CHECK("raster_large_kernel");
    }
    resolve_kernel<<<grid_for(npix), RENDER_THREADS, 0, s>>>(pts, faces, zbuf, npix, depth, face, normal);
    DFB_LAUNCH_CHECK("resolve_kernel");
    return DFB_OK;
}
