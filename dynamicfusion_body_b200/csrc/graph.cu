// graph.cu -- SURVEY 8f ranks 1 and 2: the callers either side of the two hot paths.
//   * point-set search grid: exact k nearest points of a float32 point set for float64 queries, replacing the
//     scipy KDTree the reference builds over live / canonical surface vertices (core/fusion.py:255,264,308,
//     204; core/fusion_dm.py:226,232);
//   * closest-point correspondences with the best-of-k point-to-plane cost (core/fusion.py:258-276,
//     core/fusion_dm.py:229-244);
//   * deformation-graph maintenance: unsupported surface points (core/fusion.py:211-215) and the greedy
//     radius sampling `uniform_sample` (core/util.py:27-47) as a parallel lexicographic maximal independent set.
#include <float.h>

#include "common.h"
#include "dfb_math.h"

namespace dfb {
namespace {

struct Grid {
    const float* pts;
    int64_t n;
    double ox, oy, oz, h;
    int dx, dy, dz;
    const int32_t* cell_start;
    const int32_t* order;
};

__host__ __device__ inline Grid to_grid(const dfb_point_grid& g) {
    Grid r;
    r.pts = g.pts; r.n = g.n;
    r.ox = g.origin[0]; r.oy = g.origin[1]; r.oz = g.origin[2]; r.h = g.cell;
    r.dx = g.dims[0]; r.dy = g.dims[1]; r.dz = g.dims[2];
    r.cell_start = g.cell_start; r.order = g.order;
    return r;
}

__device__ __forceinline__ int cell_coord(double p, double o, double h, int d) {
    const int c = (int)floor((p - o) / h);
    return c < 0 ? 0 : (c >= d ? d - 1 : c);
}

__device__ __forceinline__ int cell_of(const Grid& g, double x, double y, double z) {
    return (cell_coord(z, g.oz, g.h, g.dz) * g.dy + cell_coord(y, g.oy, g.h, g.dy)) * g.dx + cell_coord(x, g.ox, g.h, g.dx);
}

// ---- build: count -> three-launch scan -> fill -> per-cell sort by id ------------------------------------------------
__global__ void grid_count_kernel(Grid g, int32_t* count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n) return;
    atomicAdd(&count[cell_of(g, g.pts[3 * i], g.pts[3 * i + 1], g.pts[3 * i + 2])], 1);
}

// Exclusive scan of count[0..cells) into start[0..cells] in three launches: every CTA scans its own 4096-cell chunk and
// reports the chunk total; one CTA scans the (<= 16385) chunk totals; the chunk offsets are added back.
constexpr int SCAN_CHUNK = 4096;   // 1024 threads x 4 consecutive cells

// block-wide exclusive scan of one chunk; returns this thread's exclusive prefix of its four cells, `total` = chunk sum
__device__ __forceinline__ int32_t chunk_scan(const int32_t c[4], int32_t* warp_sum, int32_t& total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int32_t mine = c[0] + c[1] + c[2] + c[3];
    int32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sum[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int32_t s = warp_sum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        warp_sum[lane] = s;
    }
    __syncthreads();
    total = warp_sum[31];
    return (wid ? warp_sum[wid - 1] : 0) + incl - mine;
}

__global__ void __launch_bounds__(1024) scan_chunks_kernel(const int32_t* count, int64_t n, int32_t* start, int32_t* chunk_total) {
    __shared__ int32_t warp_sum[32];
    const int64_t i0 = (int64_t)blockIdx.x * SCAN_CHUNK + 4 * (int64_t)threadIdx.x;
    int32_t c[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) c[j] = (i0 + j < n) ? count[i0 + j] : 0;
    int32_t total;
    int32_t run = chunk_scan(c, warp_sum, total);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (i0 + j < n) start[i0 + j] = run;
        run += c[j];
    }
    if (threadIdx.x == 0) chunk_total[blockIdx.x] = total;
}

// one CTA: in-place exclusive scan of v[0..n), grand total to *total_out
__global__ void __launch_bounds__(1024) scan_totals_kernel(int32_t* v, int n, int32_t* total_out) {
    __shared__ int32_t warp_sum[32];
    int32_t carry = 0;
    for (int base = 0; base < n; base += SCAN_CHUNK) {
        const int i0 = base + 4 * (int)threadIdx.x;
        int32_t c[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) c[j] = (i0 + j < n) ? v[i0 + j] : 0;
        int32_t total;
        int32_t run = carry + chunk_scan(c, warp_sum, total);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (i0 + j < n) v[i0 + j] = run;
            run += c[j];
        }
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(1024) scan_add_kernel(int32_t* start, int64_t n, const int32_t* chunk_offset) {
    const int64_t i0 = (int64_t)blockIdx.x * SCAN_CHUNK + 4 * (int64_t)threadIdx.x;
    const int32_t off = chunk_offset[blockIdx.x];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (i0 + j < n) start[i0 + j] += off;
}

__global__ void grid_fill_kernel(Grid g, int32_t* cursor, int32_t* order) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n) return;
    const int c = cell_of(g, g.pts[3 * i], g.pts[3 * i + 1], g.pts[3 * i + 2]);
    order[g.cell_start[c] + atomicAdd(&cursor[c], 1)] = (int32_t)i;
}

// the atomics leave a cell's members in arrival order; ascending ids make every later scan deterministic
__global__ void grid_sort_kernel(const int32_t* start, int64_t cells, int32_t* order) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    const int a = start[c], b = start[c + 1];
    for (int i = a + 1; i < b; ++i) {
        const int32_t v = order[i];
        int j = i - 1;
        while (j >= a && order[j] > v) { order[j + 1] = order[j]; --j; }
        order[j + 1] = v;
    }
}

// ---- exact kNN ------------------------------------------------------------------------------------------
// Squared distance the way scipy's KDTree accumulates it: float64, x then y then z, no contraction.
__device__ __forceinline__ double dist2_ref(double qx, double qy, double qz, const float* p) {
    const double ax = dsub(qx, (double)p[0]), ay = dsub(qy, (double)p[1]), az = dsub(qz, (double)p[2]);
    return dadd(dadd(dmul(ax, ax), dmul(ay, ay)), dmul(az, az));
}

template <int KMAX>
struct TopK {
    double d[KMAX];
    int32_t id[KMAX];
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int j = 0; j < KMAX; ++j) { d[j] = DBL_MAX; id[j] = 0x7fffffff; }
    }
    // ascending (distance, id): equal distances keep the lower id first, like a stable argsort of brute-force distances
    __device__ __forceinline__ void push(double dd, int32_t ii, int k) {
        if (!(dd < d[k - 1] || (dd == d[k - 1] && ii < id[k - 1]))) return;
        // compare-and-swap chain: the new element sinks to its place, the displaced ones move up, the last falls out
#pragma unroll
        for (int j = 0; j < KMAX; ++j) {
            if (j < k && (dd < d[j] || (dd == d[j] && ii < id[j]))) {
                const double td = d[j]; d[j] = dd; dd = td;
                const int32_t ti = id[j]; id[j] = ii; ii = ti;
            }
        }
    }
};

template <int KMAX>
__device__ __forceinline__ void scan_cells(const Grid& g, int c0, int c1, double qx, double qy, double qz, int k, TopK<KMAX>& top) {
    const int a = g.cell_start[c0], b = g.cell_start[c1 + 1];
    for (int t = a; t < b; ++t) {
        const int32_t i = g.order[t];
        top.push(dist2_ref(qx, qy, qz, g.pts + 3 * (size_t)i), i, k);
    }
}

// One query per thread; rings of cells of growing Chebyshev radius around the query's (clamped) cell.  Before ring r is
// scanned every unvisited point is at least (r-1)*h - off away (off = distance of the query from the grid box), so the
// search stops as soon as the k-th distance is strictly below that (strictly: equal-distance points with a lower id may
// still be unvisited).
template <int KMAX>
__global__ void __launch_bounds__(128) grid_knn_kernel(Grid g, const double* q, int64_t m, int k, int32_t* idx, double* d2out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const double qx = q[3 * t], qy = q[3 * t + 1], qz = q[3 * t + 2];
    const int cx = cell_coord(qx, g.ox, g.h, g.dx), cy = cell_coord(qy, g.oy, g.h, g.dy), cz = cell_coord(qz, g.oz, g.h, g.dz);
    const double hx = g.ox + g.h * g.dx, hy = g.oy + g.h * g.dy, hz = g.oz + g.h * g.dz;
    const double ex = qx < g.ox ? g.ox - qx : (qx > hx ? qx - hx : 0.0);
    const double ey = qy < g.oy ? g.oy - qy : (qy > hy ? qy - hy : 0.0);
    const double ez = qz < g.oz ? g.oz - qz : (qz > hz ? qz - hz : 0.0);
    const double off = sqrt(ex * ex + ey * ey + ez * ez);
    TopK<KMAX> top;
    top.init();
    int rmax = max(max(cx, g.dx - 1 - cx), max(max(cy, g.dy - 1 - cy), max(cz, g.dz - 1 - cz)));
    for (int r = 0; r <= rmax; ++r) {
        if (r >= 2 && top.id[k - 1] != 0x7fffffff) {
            const double reach = (r - 1) * g.h * (1.0 - 1e-6) - off - 1e-9 * g.h;
            if (reach > 0.0 && top.d[k - 1] < reach * reach) break;
        }
        const int z0 = max(cz - r, 0), z1 = min(cz + r, g.dz - 1);
        const int y0 = max(cy - r, 0), y1 = min(cy + r, g.dy - 1);
        const int x0 = max(cx - r, 0), x1 = min(cx + r, g.dx - 1);
        for (int z = z0; z <= z1; ++z) {
            const bool zface = (z == cz - r) || (z == cz + r);
            for (int y = y0; y <= y1; ++y) {
                const int row = (z * g.dy + y) * g.dx;
                if (zface || y == cy - r || y == cy + r) {
                    scan_cells<KMAX>(g, row + x0, row + x1, qx, qy, qz, k, top);   // a whole x-run of the shell
                } else {
                    if (cx - r >= 0) scan_cells<KMAX>(g, row + cx - r, row + cx - r, qx, qy, qz, k, top);
                    if (r > 0 && cx + r < g.dx) scan_cells<KMAX>(g, row + cx + r, row + cx + r, qx, qy, qz, k, top);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
        if (j < k) {
            idx[t * k + j] = top.id[j] == 0x7fffffff ? -1 : top.id[j];
            if (d2out) d2out[t * k + j] = top.d[j];
        }
    }
}

// ---- correspondences ------------------------------------------------------------------------------------
// core/fusion.py:266-274 / core/fusion_dm.py:233-241: best_pt = first neighbour, best_cost = 1; a neighbour replaces it
// when cost = |n . (v - p)| < best_cost.  np.dot of two float64 3-vectors: products summed left to right.
__global__ void corr_select_kernel(const double* wv, const double* wn, int64_t m, const float* lverts, const int32_t* nn, int k,
                                   int32_t* best, double* best_cost) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const double vx = wv[3 * t], vy = wv[3 * t + 1], vz = wv[3 * t + 2];
    const double nx = wn[3 * t], ny = wn[3 * t + 1], nz = wn[3 * t + 2];
    int32_t b = nn[t * k];
    double bc = 1.0;
    for (int j = 0; j < k; ++j) {
        const int32_t i = nn[t * k + j];
        if (i < 0) continue;
        const float* p = lverts + 3 * (size_t)i;
        const double c = fabs(dadd(dadd(dmul(nx, dsub(vx, (double)p[0])), dmul(ny, dsub(vy, (double)p[1]))), dmul(nz, dsub(vz, (double)p[2]))));
        if (c < bc) { bc = c; b = i; }
    }
    best[t] = b;
    best_cost[t] = bc;
}

// Projective data association (dfb_math.h assoc_projective_ref): one thread per warped canonical point, grid-stride.
__global__ void __launch_bounds__(128) corr_projective_kernel(const double* wv, const double* wn, int64_t m, const dfb_views views,
                                                              double max_distance, double min_normal_dot, int32_t* view, double* cost,
                                                              double* corr) {
    // the camera block is read through pointers by the per-point function: staged in shared memory (indexing the kernel
    // parameter through a pointer would make every thread copy the whole struct to its local stack)
    __shared__ double sK[9], sKinv[9], sE[DFB_MAX_VIEWS * 12];
    __shared__ const float* sD[DFB_MAX_VIEWS];
    for (int i = threadIdx.x; i < 9; i += blockDim.x) { sK[i] = views.K[i]; sKinv[i] = views.Kinv[i]; }
    for (int i = threadIdx.x; i < 12 * views.n_views; i += blockDim.x) sE[i] = views.E[i / 12][i % 12];
    for (int i = threadIdx.x; i < views.n_views; i += blockDim.x) sD[i] = views.depth[i];
    __syncthreads();
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m; t += (int64_t)gridDim.x * blockDim.x) {
        const double w[3] = {wv[3 * t], wv[3 * t + 1], wv[3 * t + 2]};
        const double n[3] = {wn[3 * t], wn[3 * t + 1], wn[3 * t + 2]};
        double c, p[3];
        view[t] = assoc_projective_ref(w, n, sD, views.n_views, views.rows, views.cols, sK, sKinv, views.has_extrinsics ? sE : nullptr,
                                       max_distance, min_normal_dot, &c, p);
        cost[t] = c;
        corr[3 * t] = p[0]; corr[3 * t + 1] = p[1]; corr[3 * t + 2] = p[2];
    }
}

// ---- graph maintenance ----------------------------------------------------------------------------------
// core/fusion.py:212-215: a surface point is unsupported when min_i |node_i - vert| / dg_w_i >= 1 over its k nearest nodes
// (float32 difference and norm, then the quotient in float64).
__global__ void graph_unsupported_kernel(const float* verts, int64_t m, const int32_t* vknn, int k, const float* node_pos,
                                         const float* node_w, uint8_t* out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const float x = verts[3 * t], y = verts[3 * t + 1], z = verts[3 * t + 2];
    double mn = DBL_MAX;
    for (int j = 0; j < k; ++j) {
        const int32_t i = vknn[t * k + j];
        const float nr = norm3_f32_ref(node_pos[3 * i], node_pos[3 * i + 1], node_pos[3 * i + 2], x, y, z);
        mn = fmin(mn, ddiv((double)nr, (double)node_w[i]));
    }
    out[t] = mn >= 1.0 ? 1 : 0;
}

// core/util.py:27-47 keeps candidate i iff no KEPT candidate j < i lies within `radius` (the loop removes everything within
// the radius of the sample it just took, the sample itself included).  That is the lexicographically first maximal
// independent set of the "closer than radius" graph; it is computed by rounds: an undecided candidate is dropped as soon
// as one earlier neighbour is kept, and kept once all its earlier neighbours are dropped.  state: 0 undecided, 1 kept,
// 2 dropped.  Reads of a state another thread is changing in the same round are harmless (states only ever leave 0).
// distance: np.column_stack promotes the candidates to float64; norm = sqrt(dot(d, d)).
__global__ void __launch_bounds__(128) sample_round_kernel(Grid g, double radius, uint8_t* state, int32_t* undecided) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n || state[i] != 0) return;
    const double qx = g.pts[3 * i], qy = g.pts[3 * i + 1], qz = g.pts[3 * i + 2];
    const int rc = (int)ceil(radius / g.h * (1.0 + 1e-6));
    const int cx = cell_coord(qx, g.ox, g.h, g.dx), cy = cell_coord(qy, g.oy, g.h, g.dy), cz = cell_coord(qz, g.oz, g.h, g.dz);
    bool open = false;
    for (int z = max(cz - rc, 0); z <= min(cz + rc, g.dz - 1); ++z)
        for (int y = max(cy - rc, 0); y <= min(cy + rc, g.dy - 1); ++y) {
            const int row = (z * g.dy + y) * g.dx;
            const int a = g.cell_start[row + max(cx - rc, 0)], b = g.cell_start[row + min(cx + rc, g.dx - 1) + 1];
            for (int t = a; t < b; ++t) {
                const int32_t j = g.order[t];
                if (j >= i) continue;
                const uint8_t s = ((volatile uint8_t*)state)[j];
                if (s == 2) continue;
                if (!(dsqrt(dist2_ref(qx, qy, qz, g.pts + 3 * (size_t)j)) < radius)) continue;
                if (s == 1) { state[i] = 2; return; }
                open = true;
            }
        }
    if (open) atomicAdd(undecided, 1);
    else state[i] = 1;
}

int check_grid(const dfb_point_grid* g) {
    DFB_REQUIRE(g && g->pts && g->cell_start && g->order, "null pointer in point grid");
    DFB_REQUIRE(g->n >= 0 && g->n < ((int64_t)1 << 31), "point count out of range");
    DFB_REQUIRE(g->cell > 0 && g->dims[0] > 0 && g->dims[1] > 0 && g->dims[2] > 0, "bad grid geometry");
    DFB_REQUIRE((int64_t)g->dims[0] * g->dims[1] * g->dims[2] <= ((int64_t)1 << 26), "more than 2^26 grid cells");
    return DFB_OK;
}
}  // namespace
}  // namespace dfb
using namespace dfb;

extern "C" int64_t dfb_point_grid_scratch_ints(int64_t cells) { return cells + (cells + SCAN_CHUNK - 1) / SCAN_CHUNK + 1; }

extern "C" int dfb_point_grid_build(const dfb_point_grid* g, int32_t* cell_start, int32_t* order, int32_t* scratch, dfb_stream_t stream) {
    DFB_REQUIRE(g && g->pts && cell_start && order && scratch, "null pointer");
    dfb_point_grid gg = *g;
    gg.cell_start = cell_start;
    gg.order = order;
    int rc = check_grid(&gg);
    if (rc != DFB_OK) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t cells = (int64_t)g->dims[0] * g->dims[1] * g->dims[2];
    Grid G = to_grid(gg);
    DFB_CUDA(cudaMemsetAsync(scratch, 0, sizeof(int32_t) * cells, s));
    const unsigned pb = (unsigned)((g->n + 255) / 256), cb = (unsigned)((cells + 255) / 256);
    if (g->n) grid_count_kernel<<<pb, 256, 0, s>>>(G, scratch);
    const int chunks = (int)((cells + SCAN_CHUNK - 1) / SCAN_CHUNK);
    int32_t* chunk_total = scratch + cells;
    scan_chunks_kernel<<<chunks, 1024, 0, s>>>(scratch, cells, cell_start, chunk_total);
    scan_totals_kernel<<<1, 1024, 0, s>>>(chunk_total, chunks, cell_start + cells);
    scan_add_kernel<<<chunks, 1024, 0, s>>>(cell_start, cells, chunk_total);
    DFB_CUDA(cudaMemsetAsync(scratch, 0, sizeof(int32_t) * cells, s));
    if (g->n) {
        grid_fill_kernel<<<pb, 256, 0, s>>>(G, scratch, order);
        grid_sort_kernel<<<cb, 256, 0, s>>>(cell_start, cells, order);
    }
    DFB_LAUNCH_CHECK("point grid build");
    return DFB_OK;
}

extern "C" int dfb_point_grid_knn(const dfb_point_grid* g, const double* queries, int64_t m, int k, int32_t* idx, double* dist2,
                                  dfb_stream_t stream) {
    int rc = check_grid(g);
    if (rc != DFB_OK) return rc;
    DFB_REQUIRE(queries && idx && m >= 0, "null pointer / negative count");
    DFB_REQUIRE(k >= 1 && k <= DFB_MAX_K, "k=%d out of range [1,%d]", k, DFB_MAX_K);
    if (m == 0) return DFB_OK;
    const unsigned blocks = (unsigned)((m + 127) / 128);
    Grid G = to_grid(*g);
    if (k <= 4) grid_knn_kernel<4><<<blocks, 128, 0, (cudaStream_t)stream>>>(G, queries, m, k, idx, dist2);
    else grid_knn_kernel<8><<<blocks, 128, 0, (cudaStream_t)stream>>>(G, queries, m, k, idx, dist2);
    DFB_LAUNCH_CHECK("grid_knn_kernel");
    return DFB_OK;
}

extern "C" int dfb_corr_select(const double* warped_pts, const double* warped_normals, int64_t m, const float* live_verts,
                               const int32_t* nn, int k, int32_t* best, double* best_cost, dfb_stream_t stream) {
    DFB_REQUIRE(warped_pts && warped_normals && live_verts && nn && best && best_cost && m >= 0, "null pointer / negative count");
    DFB_REQUIRE(k >= 1 && k <= DFB_MAX_K, "k=%d out of range [1,%d]", k, DFB_MAX_K);
    if (m == 0) return DFB_OK;
    corr_select_kernel<<<(unsigned)((m + 127) / 128), 128, 0, (cudaStream_t)stream>>>(warped_pts, warped_normals, m, live_verts, nn, k,
                                                                                      best, best_cost);
    DFB_LAUNCH_CHECK("corr_select_kernel");
    return DFB_OK;
}

extern "C" int dfb_corr_projective(const double* warped_pts, const double* warped_normals, int64_t m, const dfb_views* views,
                                   double max_distance, double min_normal_dot, int32_t* view, double* cost, double* corr,
                                   dfb_stream_t stream) {
    DFB_REQUIRE(warped_pts && warped_normals && views && view && cost && corr && m >= 0, "null pointer / negative count");
    DFB_REQUIRE(views->n_views >= 1 && views->n_views <= DFB_MAX_VIEWS, "n_views=%d out of range [1,%d]", views->n_views, DFB_MAX_VIEWS);
    DFB_REQUIRE(views->rows >= 3 && views->cols >= 3, "depth map %dx%d smaller than 3x3", views->rows, views->cols);
    for (int v = 0; v < views->n_views; ++v) DFB_REQUIRE(views->depth[v], "depth[%d] is null", v);
    DFB_REQUIRE(max_distance > 0, "max_distance must be positive");
    DFB_REQUIRE(min_normal_dot >= -1.0 && min_normal_dot <= 1.0, "min_normal_dot must be in [-1,1]");
    if (m == 0) return DFB_OK;
    const int64_t need = (m + 127) / 128;
    const unsigned blocks = (unsigned)(need < 148 * 16 ? need : 148 * 16);   // 16 blocks per SM, grid-stride beyond
    corr_projective_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(warped_pts, warped_normals, m, *views, max_distance, min_normal_dot,
                                                                       view, cost, corr);
    DFB_LAUNCH_CHECK("corr_projective_kernel");
    return DFB_OK;
}

extern "C" int dfb_graph_unsupported(const float* verts, int64_t m, const int32_t* vert_knn, int k, const float* node_pos,
                                     const float* node_w, uint8_t* unsupported, dfb_stream_t stream) {
    DFB_REQUIRE(verts && vert_knn && node_pos && node_w && unsupported && m >= 0, "null pointer / negative count");
    DFB_REQUIRE(k >= 1 && k <= DFB_MAX_K, "k=%d out of range [1,%d]", k, DFB_MAX_K);
    if (m == 0) return DFB_OK;
    graph_unsupported_kernel<<<(unsigned)((m + 127) / 128), 128, 0, (cudaStream_t)stream>>>(verts, m, vert_knn, k, node_pos, node_w,
                                                                                            unsupported);
    DFB_LAUNCH_CHECK("graph_unsupported_kernel");
    return DFB_OK;
}

extern "C" int dfb_graph_sample_rounds(const dfb_point_grid* g, double radius, int rounds, uint8_t* state, int32_t* undecided,
                                       dfb_stream_t stream) {
    int rc = check_grid(g);
    if (rc != DFB_OK) return rc;
    DFB_REQUIRE(state && undecided && radius > 0 && rounds >= 1, "bad arguments");
    if (g->n == 0) return DFB_OK;
    cudaStream_t s = (cudaStream_t)stream;
    Grid G = to_grid(*g);
    for (int r = 0; r < rounds; ++r) {
        DFB_CUDA(cudaMemsetAsync(undecided, 0, sizeof(int32_t), s));
        sample_round_kernel<<<(unsigned)((g->n + 127) / 128), 128, 0, s>>>(G, radius, state, undecided);
    }
    DFB_LAUNCH_CHECK("sample_round_kernel");
    return DFB_OK;
}
