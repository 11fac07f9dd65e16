/*
 * dfb.h -- C ABI of libdfb_b200.so: B200 (sm_100a) kernels for the two hot paths of
 * nintendops/DynamicFusion_Body, called from the Python classes that mirror the reference's
 * Fusion / FusionDM method surface (dynamicfusion_body_b200/fusion.py).
 *
 * The reference has no FFI: its replacement mechanism is "subclass and override the hot method"
 * (FusionDM_GPU overrides FusionDM.fuseDepths, core/fusion_dm.py:563-600,737).  Each entry point
 * below names the reference method body it replaces.
 *
 * Conventions
 *   - every bulk pointer is a DEVICE pointer owned by the caller; small matrices inside the
 *     parameter structs are HOST values copied into kernel arguments;
 *   - every call is asynchronous on `stream` (a cudaStream_t) and makes no hidden allocation;
 *   - return 0 on success, <0 on error (dfb_last_error() gives the text);  there is no CPU path;
 *   - volumes are C-ordered [x][y][z] float32 (np.nditer order, core/fusion.py:171), optionally a
 *     slab x in [x0,x1) of the full grid whose pointer addresses voxel (x0,0,0).
 */
#ifndef DFB_H_
#define DFB_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFB_MAX_K 8
#define DFB_MAX_VIEWS 8
#define DFB_NODE_REC_FLOATS 12 /* pos xyz, exp2 coefficient, dq[8] */

#define DFB_OK 0
#define DFB_ERR_INVALID (-1)
#define DFB_ERR_CUDA (-2)

#define DFB_MODE_HYBRID 0 /* fp32 classify + clamped update, reference-exact fp64 pass for the rest */
#define DFB_MODE_EXACT 1  /* every voxel through the reference-exact pass (validation / debugging) */
#define DFB_MODE_FAST_ONLY 2 /* profiling: pass 1 only (deferred voxels are left untouched, list is filled) */
#define DFB_MODE_LIST_ONLY 3 /* profiling: pass 2 only, over the list a DFB_MODE_FAST_ONLY call left behind */
#define DFB_MODE_BRICK_CLASSIFY 4 /* profiling: brick classification only (fills the brick lists) */
#define DFB_MODE_BRICK_STREAM 5   /* profiling: streaming pass over the CLAMP bricks of the last classification */
#define DFB_MODE_BRICK_MIXED 6    /* profiling: per-voxel pass over the MIXED bricks of the last classification */
#define DFB_MODE_BRICK_UPDATE 7   /* profiling: the production fused CLAMP+MIXED pass after a DFB_MODE_BRICK_CLASSIFY call */

typedef void* dfb_stream_t; /* cudaStream_t */

typedef struct dfb_volume {
    float* tsdf;   /* Fusion._tsdf   (core/fusion.py:76),  slab-local */
    float* weight; /* Fusion._tsdfw  (core/fusion.py:74),  slab-local */
    int rx, ry, rz; /* full grid resolution */
    int x0, x1;     /* this slab: x in [x0,x1) */
} dfb_volume;

typedef struct dfb_warpfield {
    const float* node_rec; /* [n_nodes][12] from dfb_nodes_pack */
    const float* node_pos; /* [n_nodes][3]  float32 node positions dg_v  (core/fusion.py:114) */
    const float* node_dq;  /* [n_nodes][8]  float32 dual quaternions dg_se3 (core/fusion.py:115) */
    const float* node_w;   /* [n_nodes]     dg_w = 2*radius (core/fusion.py:116) */
    int n_nodes;
    int k;               /* neighbours per voxel (Fusion._knn); 0 = rigid (FusionDM.updateTSDF) */
    const uint16_t* knn; /* [(x1-x0)*ry*rz][k] from dfb_knn_build_volume, ascending distance */
    int has_lw;          /* apply the global rigid dq `lw` (Fusion._lw, m_lw of Fusion.warp) */
    int lw_is_f32;       /* lw is a float32 array in the reference (its initial state): the first
                            dual-quaternion product of dqb_warp then runs in float32 (core/util.py:69-70) */
    double lw[8];
    /* optional (NULL = no brick culling): per-brick union of the voxels' kNN sets, from dfb_brick_nodes_build */
    const uint16_t* brick_nodes; /* [n_bricks][24] */
    const uint8_t* brick_count;  /* [n_bricks], 255 = more than 24 */
    const uint32_t* brick_pairs; /* [n_bricks][10]: bit i*(i+1)/2+j set when candidates i>=j share a voxel's kNN set (NULL = all pairs) */
    /* optional (NULL = per-brick pairwise hull + per-voxel DQB tier): 16x16x32-voxel regions from dfb_region_build */
    const uint16_t* region_nodes; /* [n_regions][64] */
    const uint8_t* region_count;  /* [n_regions], 255 = more than 64 distinct nodes */
    const uint32_t* region_pairs; /* [n_regions][65] pair bit masks */
    float* region_rec;            /* [n_regions][32] scratch: reference map + deviation bound + view 0's composed map, rewritten by every update call */
} dfb_warpfield;

typedef struct dfb_views {
    int n_views;                        /* applied sequentially in index order (core/fusion_dm.py:166-170) */
    const float* depth[DFB_MAX_VIEWS];  /* [rows][cols] float32, depth stored NEGATIVE, 0 = no data */
    int rows, cols;                     /* (dmx, dmy) = dm.shape (core/fusion_dm.py:181) */
    double K[9];                        /* FusionDM._K    row-major 3x3 */
    double Kinv[9];                     /* FusionDM._Kinv row-major 3x3 */
    int has_extrinsics;                 /* lpos = E_v @ [p',1] */
    double E[DFB_MAX_VIEWS][12];        /* row-major 3x4 */
} dfb_views;

typedef struct dfb_workspace {
    uint32_t* list;     /* device [capacity]: voxels deferred to the exact pass */
    uint32_t capacity;
    uint32_t* counters; /* device [8]; counters[0] = voxels deferred to the exact pass by the last call,
                           counters[1] = voxels the exact pass processed, counters[2] = bricks streamed (CLAMP),
                           counters[3] = bricks evaluated per voxel (MIXED), counters[4] = voxels of MIXED bricks the quad
                           pre-test left to the pointwise DQB tier */
    /* optional (NULL = no brick culling), n_bricks = dfb_brick_count(x1-x0, ry, rz): */
    uint8_t* brick_cls;    /* device [4*n_bricks]: class (0xFF = MIXED), frustum bits, open views, settled CLAMP bits */
    uint32_t* brick_lists; /* device [2*n_bricks] */
    /* optional, device [ceil(slab voxels / 32)], zeroed once by the caller: voxels deferred after `list` has filled up are
     * marked here instead and the exact pass consumes (and clears) the marks -- a call that overflows the list is then
     * still exact.  NULL: an overflowing call re-scans the volume with the per-voxel classifier, which is only equivalent
     * when no brick workspace is given (brick-level decisions are not replayed by the re-scan). */
    uint32_t* overflow_bits;
} dfb_workspace;

int dfb_version(void);
const char* dfb_last_error(void);

/* node table: (pos, dq, w) -> 48-byte records used by the update kernels. */
int dfb_nodes_pack(const float* node_pos, const float* node_dq, const float* node_w, int n_nodes,
                   float* node_rec, dfb_stream_t stream);

/* scipy KDTree.query(pos, k+1)[:-1] for every voxel centre of a slab (core/fusion.py:175-176):
 * k nearest node ids in ascending float64 distance (lower id first on exact ties). */
int dfb_knn_build_volume(const float* node_pos, int n_nodes, int k, int rx, int ry, int rz, int x0, int x1,
                         uint16_t* knn, dfb_stream_t stream);
/* Graph revisions (core/fusion.py:216-229: update_graph only ever APPENDS nodes).  The build works on 8x8x8-voxel bricks;
 * dfb_knn_build_volume_radii also stores the search radius of every brick (float [dfb_knn_brick_count]), with which
 * dfb_knn_update_volume brings the table up to date after nodes [n_old, n_nodes) were appended: only bricks a new node can reach are
 * rebuilt (the others leave at once), dirty [dfb_knn_brick_count] = 1 for those.  The table equals a full rebuild bit for bit. */
int64_t dfb_knn_brick_count(int slab_x, int ry, int rz);
int dfb_knn_build_volume_radii(const float* node_pos, int n_nodes, int k, int rx, int ry, int rz, int x0, int x1, uint16_t* knn,
                               float* brick_radius, dfb_stream_t stream);
int dfb_knn_update_volume(const float* node_pos, int n_old, int n_nodes, int k, int rx, int ry, int rz, int x0, int x1, uint16_t* knn,
                          float* brick_radius, uint8_t* dirty, dfb_stream_t stream);
/* Brick culling support (4x4x32-voxel bricks): number of bricks of a slab, and the per-brick candidate node sets
 * derived from the kNN table (once per graph revision). */
int64_t dfb_brick_count(int slab_x, int ry, int rz);
int dfb_brick_nodes_build(const uint16_t* knn, int k, int rx, int ry, int rz, int x0, int x1, uint16_t* brick_nodes,
                          uint8_t* brick_count, uint32_t* brick_pairs, dfb_stream_t stream);
/* Regions (16x16x32 voxels): distinct nodes and co-occurring node pairs of each region (once per graph revision). */
int64_t dfb_region_count(int slab_x, int ry, int rz);
int dfb_region_build(const uint16_t* knn, int k, int rx, int ry, int rz, int x0, int x1, uint16_t* region_nodes,
                     uint8_t* region_count, uint32_t* region_pairs, dfb_stream_t stream);
/* the same two, restricted to the bricks / regions that overlap an 8^3 brick flagged by dfb_knn_update_volume (dirty8 NULL = all) */
int dfb_brick_nodes_update(const uint16_t* knn, int k, int rx, int ry, int rz, int x0, int x1, const uint8_t* dirty8, uint16_t* brick_nodes,
                           uint8_t* brick_count, uint32_t* brick_pairs, dfb_stream_t stream);
int dfb_region_update(const uint16_t* knn, int k, int rx, int ry, int rz, int x0, int x1, const uint8_t* dirty8, uint16_t* region_nodes,
                      uint8_t* region_count, uint32_t* region_pairs, dfb_stream_t stream);
/* KDTree.query(vert, k) for arbitrary float32 points (core/fusion.py:122,232). */
int dfb_knn_points(const float* pts, int64_t m, const float* node_pos, int n_nodes, int k, int32_t* idx,
                   dfb_stream_t stream);

/* a3: Fusion.warp (core/fusion.py:502-520) + per-voxel body of FusionDM.fuseDepths
 * (core/fusion_dm.py:193-210) with scale=1, center=0, all views fused in one pass.
 * mask_out / frustum_out (optional, [slab voxels] uint8): bit v = view v updated the voxel /
 * voxel projected inside view v's image (core/fusion_dm.py:195). */
int dfb_tsdf_update_projective(const dfb_volume* vol, const dfb_warpfield* wf, const dfb_views* views,
                               double tdist, double wmax, int mode, const dfb_workspace* ws,
                               uint8_t* mask_out, uint8_t* frustum_out, dfb_stream_t stream);

/* a1: Fusion.updateTSDF (core/fusion.py:171-190); with wf->k == 0: FusionDM.updateTSDF
 * (core/fusion_dm.py:300-316).  curr = live TSDF volume [cx][cy][cz] float32. */
int dfb_tsdf_update_volume(const dfb_volume* vol, const dfb_warpfield* wf, const float* curr, int cx, int cy,
                           int cz, double tdist, double wmax, int mode, const dfb_workspace* ws,
                           uint8_t* mask_out, dfb_stream_t stream);

/* a2: FusionDM.fuseDepths (core/fusion_dm.py:180-217): rigid 3x4 `lw`, grid->world
 * pos = scale*(idx - tsdf_res/2) + center. */
int dfb_fuse_depth_rigid(const dfb_volume* vol, int tsdf_res, const float* depth, int rows, int cols,
                         const double lw34[12], const double K[9], const double Kinv[9], double scale,
                         const double center[3], double tdist, double wmax, int mode, const dfb_workspace* ws,
                         uint8_t* mask_out, uint8_t* frustum_out, dfb_stream_t stream);

/* a4: Fusion.warp for arbitrary float32 points (+ optional normals) with explicit neighbours
 * idx [m][k]; outputs float64 [m][3], computed with the reference's arithmetic. */
int dfb_warp_points(const float* pts, const float* normals, int64_t m, const int32_t* idx, const dfb_warpfield* wf,
                    double* out_pts, double* out_normals, dfb_stream_t stream);

/* a5: Fusion.dq_blend (core/fusion.py:527-551) for float32 points: blended, 8-norm-normalised dq [m][8] float64. */
int dfb_dq_blend_points(const float* pts, int64_t m, const int32_t* idx, const dfb_warpfield* wf, double* out_dq,
                        dfb_stream_t stream);

/* ---- warp-field least squares (Fusion.solve, core/fusion.py:327-491) ------------------------------------ */
typedef struct dfb_gn_problem {
    int64_t n_vert;
    const float* vertices;    /* [V][3]  Fusion._vertices */
    const float* normals;     /* [V][3]  Fusion._normals */
    const double* corr;       /* [V][3]  Fusion._correspondences */
    const int32_t* vert_knn;  /* [V][k]  Fusion._neighbor_look_up */
    int n_nodes, k;
    const float* node_pos;    /* [N][3] */
    const float* node_w;      /* [N] */
    const int32_t* node_nbr;  /* [N][k]  _neighbor_look_up[_nodes[i][0]] (core/fusion.py:477) */
    double lw[8];             /* Fusion._lw */
    int lw_is_f32;
    double rw;                /* regularization_weight */
    int huber;                /* 1: IRLS weights min(1, f_scale/|f|) (scipy loss='huber' counterpart) */
    double f_scale;
    const int32_t* order;     /* optional [V]: a permutation of the data residuals, sorted by (ascending) node tuple.  dfb_gn_normal_eq
                                 walks the residuals in this order and accumulates a run of equal tuples in registers before it
                                 touches H (NULL = natural order: correct, but one atomic burst per residual and block) */
} dfb_gn_problem;

/* a9: Fusion.computef (core/fusion.py:459-491): f [V + 3*k*N], reference arithmetic.  x = node dual quaternions
 * [N][8] as float64 values; x_is_f32: they are float32 in the reference (its first call, core/fusion.py:373-375). */
int dfb_gn_residuals(const dfb_gn_problem* prob, const double* x, int x_is_f32, double* f_out, dfb_stream_t stream);
/* a11: Fusion.computef_lw (core/fusion.py:444-456): f [V] as a function of the global rigid dq `lw` (host, 8). */
int dfb_gn_residuals_lw(const dfb_gn_problem* prob, const double* node_dq, int dq_is_f32, const double* lw, int lw_is_f32,
                        double* f_out, dfb_stream_t stream);
/* Block pattern of J^T J over node pairs (the CORRECT pattern; core/fusion.py:416-442 is not reproduced, SURVEY Q7).
 * rows: marks bitmap [N][ceil(N/32)], writes row_ptr [N+1] (row_ptr[N] = number of 8x8 blocks);
 * cols: writes col_idx [row_ptr[N]] ascending per row. */
int dfb_gn_pattern_rows(const dfb_gn_problem* prob, uint32_t* bitmap, int32_t* row_ptr, dfb_stream_t stream);
int dfb_gn_pattern_cols(int n_nodes, const uint32_t* bitmap, const int32_t* row_ptr, int32_t* col_idx, dfb_stream_t stream);
/* Analytic Jacobian -> BSR normal equations H = J^T W J [nnzb][8][8], g = J^T W f [N][8], cost[0] = robust cost,
 * cost[1] = 0.5 |f|^2 (all zeroed first).  Replaces scipy's finite-difference Jacobian (core/fusion.py:382-392).
 * BSR contract (here and in dfb_gn_solve): the columns of every row ascend, every diagonal block (i, i) is present, and the
 * pattern is symmetric and holds every node pair of the problem -- dfb_gn_pattern_* produce exactly that.  Blocks are looked up
 * by binary search; a missing block is NOT detected: its contribution lands in a wrong slot. */
int dfb_gn_normal_eq(const dfb_gn_problem* prob, const double* x, const int32_t* row_ptr, const int32_t* col_idx, int64_t nnzb,
                     double* H, double* g, double* cost, dfb_stream_t stream);
/* 8x8 normal equations of the rigid fit (core/fusion.py:356-360): H8 [64], g8 [8], cost [2] on the device. */
int dfb_gn_lw_normal_eq(const dfb_gn_problem* prob, const double* node_dq, const double* lw, double* H8, double* g8, double* cost,
                        dfb_stream_t stream);
/* Damped node-space solve (H + lambda*mean(diag H)*I) delta = -g by block-Jacobi PCG, then x_new = x + delta.
 * H: BSR as for dfb_gn_normal_eq, and symmetric (CG).  The solve stops once (r,z) <= tol^2 (r0,z0) or after max_iter updates.
 * workspace: dfb_gn_solve_workspace_doubles(N) doubles; workspace[0..7] = {mu, final (r,z), -, -, initial (r,z), -, iterations, trace},
 * where iterations = the number of updates of delta applied (every kernel variant counts the same way). */
int64_t dfb_gn_solve_workspace_doubles(int n_nodes);
int dfb_gn_solve(int n_nodes, const int32_t* row_ptr, const int32_t* col_idx, const double* H, const double* g, double lambda,
                 int max_iter, double tol, const double* x, double* x_new, double* delta, double* workspace, dfb_stream_t stream);

/* ---- SURVEY 8f ranks 1-2: correspondences and deformation-graph maintenance --------------------------------- */
/* Uniform search grid over a float32 point set: the replacement of the scipy KDTree the reference builds over live /
 * canonical surface vertices (core/fusion.py:204,255,308; core/fusion_dm.py:226).  Cell (cx,cy,cz) has index
 * (cz*dims[1] + cy)*dims[0] + cx; its members are order[cell_start[c] .. cell_start[c+1]) in ascending id. */
typedef struct dfb_point_grid {
    const float* pts; /* [n][3] */
    int64_t n;
    double origin[3]; /* lower corner of cell (0,0,0) */
    double cell;      /* edge length */
    int dims[3];
    const int32_t* cell_start; /* [cells + 1] */
    const int32_t* order;      /* [n] */
} dfb_point_grid;

/* Fills cell_start / order for the geometry in *g (its own cell_start / order members are ignored);
 * scratch: dfb_point_grid_scratch_ints(cells) int32. */
int64_t dfb_point_grid_scratch_ints(int64_t cells);
int dfb_point_grid_build(const dfb_point_grid* g, int32_t* cell_start, int32_t* order, int32_t* scratch, dfb_stream_t stream);
/* KDTree.query(q, k) for float64 queries [m][3]: idx [m][k] ascending (float64 squared distance, id); -1 pads when the
 * set has fewer than k points; dist2 [m][k] optional. */
int dfb_point_grid_knn(const dfb_point_grid* g, const double* queries, int64_t m, int k, int32_t* idx, double* dist2,
                       dfb_stream_t stream);
/* Best-of-k point-to-plane candidate (core/fusion.py:264-274, core/fusion_dm.py:232-241): best [m] = index into
 * live_verts, best_cost [m] = min(1, min_j |n . (v - p_j)|) with the reference's first-neighbour default. */
int dfb_corr_select(const double* warped_pts, const double* warped_normals, int64_t m, const float* live_verts,
                    const int32_t* nn, int k, int32_t* best, double* best_cost, dfb_stream_t stream);
/* Projective data association (SURVEY 8f rank 1, DynamicFusion's correspondence step) of warped canonical points /
 * normals [m][3] (from dfb_warp_points) against the depth views: view [m] (-1 = none), cost [m], corr [m][3].
 * Per view: camera frame through E_v, front-facing test, projection and rounding as dfb_tsdf_update_projective, a one-pixel
 * border ring excluded, centre and 4-neighbour depths valid and within max_distance of each other, live point and normal
 * from the back-projected pixels, gates |l - c| <= max_distance and ln.g >= min_normal_dot |ln| |g|, cost |ln.(l - c)|
 * (smallest wins, ties to the lower view); corr = R_v^T (c - t_v) in the frame of the warped points (oracle/assoc.py). */
int dfb_corr_projective(const double* warped_pts, const double* warped_normals, int64_t m, const dfb_views* views,
                        double max_distance, double min_normal_dot, int32_t* view, double* cost, double* corr,
                        dfb_stream_t stream);
/* Z-buffer rasteriser (the reference's GL vertex-id / depth renderer, core/gl/glrender.py, without a GL context): the mesh
 * pts [n_pts][3] float64 (e.g. warped by dfb_warp_points) / faces [n_faces][3] int32 seen by the cameras of *views (K, E,
 * rows, cols; its depth[] pointers are ignored).  Per view v, each [rows][cols], pixel (r, c) sampled at x = c, y = r:
 * depth (negative depth, 0 = no face: the convention of every depth input here), face (id, -1 = none) and normal [..][3]
 * (the winning face's unit normal (Pb - Pa) x (Pc - Pa) in the frame of pts, float32; 0 = none or degenerate).  Faces with
 * an index outside [0, n_pts), a vertex at camera depth <= 0 or zero projected area are culled; edges are inclusive, depth
 * is perspective-correct, the nearest float32 depth wins and ties go to the lower face id (oracle/render.py).
 * workspace: dfb_render_workspace_words(n_faces, n_views, rows, cols) uint64 words (-1 for invalid arguments); after the
 * call workspace[0] holds the number of (face, view) pairs that went through the large-face kernel. */
int64_t dfb_render_workspace_words(int64_t n_faces, int n_views, int rows, int cols);
int dfb_render(const double* pts, int64_t n_pts, const int32_t* faces, int64_t n_faces, const dfb_views* views,
               uint64_t* workspace, int64_t workspace_words, float* depth, int32_t* face, float* normal, dfb_stream_t stream);
/* Rigid tracking of a depth frame against the whole fused FusionDM volume (nothing in the reference: compute_live_tsdf's
 * useICP branch, core/fusion_dm.py, needs a pose file).  Every pixel (r, c) with r % stride == 0 and c % stride == 0 and depth
 * z = -depth[r][c] > 0 is back-projected, x = Kinv [c z, r z, z], and moved to the world by the pose lw34 = [R|t]
 * (world -> camera, as in dfb_fuse_depth_rigid): p = R^T (x - t), grid coordinate g = (p - center) / scale + tsdf_res / 2.
 * It contributes when the 8 corners of its trilinear cell (0 <= floor(g) <= r - 2 on every axis) all have weight > 0 and
 * |tsdf| * scale < tdist.  Its residual is rho = scale * D, D the standard trilinear interpolant of the cell (along z, then y,
 * then x; not the swapped weights of interpolate_tsdf), its Jacobian J = [grad D, p x grad D] for the twist (tau, omega) acting
 * on world points as p + tau + omega x p, its Huber weight w = min(1, delta / |rho|) (oracle/track.py).
 * out29 (device): upper triangle of H = sum w J^T J (21, row-major), g = sum w J rho (6), the Huber cost, the pixel count.
 * residual (device, optional): [ceil(rows/stride)][ceil(cols/stride)] rho of every sampled pixel, NaN where it did not
 * contribute.  K is the matrix Kinv inverts (checked, not read).  workspace: dfb_track_workspace_doubles(rows, cols, stride)
 * doubles (-1 for invalid arguments).  A slab volume (x0 != 0 or x1 != rx) is refused.  No atomics: a call's sums are
 * identical run to run. */
int64_t dfb_track_workspace_doubles(int rows, int cols, int stride);
int dfb_track_normal_eq(const dfb_volume* vol, int tsdf_res, double scale, const double center[3], const float* depth, int rows,
                        int cols, const double K[9], const double Kinv[9], const double lw34[12], int stride, double tdist,
                        double delta, double* workspace, int64_t workspace_doubles, double* out29, double* residual,
                        dfb_stream_t stream);
/* Raycasting of the whole fused FusionDM volume (nothing in the reference, which can only extract the surface): depth and
 * normal maps of the model from every view of `views` (K is not read, Kinv is; E[v] = [R|t] world -> camera as in
 * dfb_fuse_depth_rigid, identity without extrinsics; depth pointers ignored).  Pixel (r, c) of view v samples its ray at
 * z_k = z_near + k step (camera z, world units) while z_k <= z_far, each sample back-projected and gated exactly as
 * dfb_track_normal_eq back-projects and gates a pixel of depth z_k (grid g = (p - center) / scale + tsdf_res / 2, all 8
 * corners observed with |tsdf| * scale < tdist, standard trilinear D).  The first pair of consecutive valid samples with
 * D_k > 0 >= D_k+1 is a hit, refined once, z* = z_k + step D_k / (D_k - D_k+1); D_k < 0 <= D_k+1 (a back face) ends the ray
 * with no hit.  depth [V][rows][cols] (device): -float(z*), 0 = no hit; normal [V][rows][cols][3] (device): grad D / |grad D| at
 * z* in the world frame, 0 = no hit or zero gradient.  The march is clipped to the volume's box (oracle/raycast.py).
 * A slab volume (x0 != 0 or x1 != rx) is refused.  Needs step > 0, 0 <= z_near < z_far (finite), (z_far - z_near) / step < 2^30.
 * One thread per ray, no atomics: identical run to run. */
int dfb_raycast(const dfb_volume* vol, int tsdf_res, double scale, const double center[3], const dfb_views* views, double tdist,
                double step, double z_near, double z_far, float* depth, float* normal, dfb_stream_t stream);
/* core/fusion.py:211-215: unsupported [m] = 1 where min over the k nearest nodes of |node - vert| / dg_w >= 1. */
int dfb_graph_unsupported(const float* verts, int64_t m, const int32_t* vert_knn, int k, const float* node_pos,
                          const float* node_w, uint8_t* unsupported, dfb_stream_t stream);
/* uniform_sample (core/util.py:27-47) over the points of *g (cell >= radius / 4 recommended): runs `rounds` rounds of
 * the parallel greedy selection on state [n] (0 undecided, 1 kept, 2 dropped; zero it before the first call);
 * *undecided = candidates still open after the last round (repeat until 0). */
int dfb_graph_sample_rounds(const dfb_point_grid* g, double radius, int rounds, uint8_t* state, int32_t* undecided,
                            dfb_stream_t stream);

/* ---- SURVEY 8f rank 3: surface extraction ------------------------------------------------------------------- */
/* Indexed level-set mesh of a device-resident float32 volume [rx][ry][rz]: the replacement of
 * skimage.measure.marching_cubes_lewiner(volume, step_size=step, allow_degenerate=False) as called by Fusion.marching_cubes /
 * write_canonical_mesh (core/fusion.py:554-568, 579; core/fusion_dm.py:341).  Cells span `step` voxels; one vertex per crossed
 * edge of the sampled grid (no welding pass), vertices in (x, y, z) voxel coordinates ordered by owning sample then axis, faces
 * ordered by cell; triangles with two vertices on one grid sample are dropped.  Call order: [dfb_mc_level] -> dfb_mc_count ->
 * read row_voff[rows] / row_toff[rows] (vertex / triangle totals) -> allocate -> dfb_mc_emit.
 * x_origin (count and emit, same value): sample index of the volume's first x-plane in the whole grid, 0 for a whole volume.  An
 * x-slab (SURVEY 8e) passed with its origin yields the coordinates AND the degenerate-triangle decisions of the whole grid, so the
 * slabs' meshes concatenate to the single-volume mesh bit for bit (dist.extract_surface_slab).  Rows of one x-plane are
 * contiguous: row_voff[i * ny] / row_toff[i * ny] are the first vertex / triangle of sample plane i. */
typedef struct dfb_mc_chunk {
    int32_t voff;  /* vertices of the row before this 32-sample chunk */
    uint32_t m[3]; /* per axis: bit l = the edge owned by sample 32*c + l crosses the level */
} dfb_mc_chunk;

/* level_out [3] (device) = {0.5 * (min + max), min, max}: the level skimage uses when none is passed, as the reference does.
 * scratch: dfb_mc_level_scratch_floats() floats. */
int64_t dfb_mc_level_scratch_floats(void);
int dfb_mc_level(const float* vol, int64_t n, float* scratch, float* level_out, dfb_stream_t stream);
/* rows = sampled (x, y) pairs; chunks = rows * ceil(samples_z / 32) */
int64_t dfb_mc_rows(int rx, int ry, int step);
int64_t dfb_mc_chunks(int rx, int ry, int rz, int step);
/* level: device pointer to one float.  Writes chunks [dfb_mc_chunks] and the exclusive vertex / triangle offsets of every
 * row, row_voff / row_toff [rows + 1] (slot [rows] = total). */
int dfb_mc_count(const float* vol, int rx, int ry, int rz, int step, int x_origin, const float* level, dfb_mc_chunk* chunks,
                 int32_t* row_voff, int32_t* row_toff, dfb_stream_t stream);
/* verts [nv][3], faces [nt][3] int32; normals [nv][3] (unit, along the +gradient) and values [nv] may be NULL. */
int dfb_mc_emit(const float* vol, int rx, int ry, int rz, int step, int x_origin, const float* level, const dfb_mc_chunk* chunks,
                const int32_t* row_voff, const int32_t* row_toff, float* verts, float* normals, float* values, int32_t* faces,
                dfb_stream_t stream);

/* ---- SURVEY 8b item 9 / 8e: collectives of the sharded path over NCCL -------------------------------------------
 * The reference is single-process (SURVEY 5 "Distributed communication backend: none"); these are what the slab-sharded
 * update and the residual-sharded solve need: per frame a root -> all broadcast of depth view(s) + node transforms +
 * global rigid dq, per Gauss-Newton iteration one sum of the flat [H | g | cost] buffer, and the neighbour exchange of
 * halo planes for surface extraction.  NCCL is bound at run time (dlopen libnccl.so.2); one communicator per GPU /
 * process, created from a unique id that the host distributes by its own means (file, socket, MPI, torch store). */
#define DFB_COMM_ID_BYTES 128
#define DFB_COMM_SUM 0
#define DFB_COMM_MAX 1
typedef struct dfb_comm dfb_comm;
int dfb_comm_available(void);                 /* 0 = NCCL could not be loaded, else its version code (or 1) */
int dfb_comm_unique_id(void* id_out);         /* host buffer of DFB_COMM_ID_BYTES; call on one rank, hand the bytes to all */
int dfb_comm_init(dfb_comm** out, const void* id, int world, int rank, int device);
int dfb_comm_destroy(dfb_comm* c);
int dfb_comm_rank(const dfb_comm* c);
int dfb_comm_world(const dfb_comm* c);
int dfb_comm_broadcast(dfb_comm* c, void* buf, int64_t bytes, int root, dfb_stream_t stream);
/* depths [n_depth] float32, node_dq [n_nodes][8] float32, lw [8] float64 (each optional), one grouped launch */
int dfb_comm_broadcast_frame(dfb_comm* c, float* depths, int64_t n_depth, float* node_dq, int n_nodes, double* lw, int root,
                             dfb_stream_t stream);
/* in-place reduction over ranks of n doubles: the flat normal-equation buffer [H (nnzb*64) | g (8N) | cost (2)] */
int dfb_comm_allreduce_f64(dfb_comm* c, double* buf, int64_t n, int op, dfb_stream_t stream);
/* grouped send to send_peer + receive from recv_peer (either side optional: peer < 0 or NULL buffer) */
int dfb_comm_sendrecv(dfb_comm* c, const void* send_buf, int64_t send_bytes, int send_peer, void* recv_buf, int64_t recv_bytes,
                      int recv_peer, dfb_stream_t stream);

/* ---- one frame of the a3 path as ONE CUDA-graph launch (the reference's per-frame `updateTSDF` call, test.py:129) ----
 * dfb_frame_step_run = [root: copy dq_src -> wf->node_dq] -> [broadcast wf->node_dq over io->comm] -> dfb_nodes_pack ->
 * dfb_tsdf_update_projective(DFB_MODE_HYBRID) -> [copy ws->counters -> counters_host], with the upload + broadcast of the next
 * frame's sensor data (prefetch_*) as a concurrent branch.  Captured on first use, replayed while the arguments stay
 * byte-identical, updated in place (cudaGraphExecUpdate) when they change.  `stream` must not be the legacy default
 * stream (then the launches are issued directly, un-captured).  Every field of dfb_frame_io is optional (NULL / 0). */
typedef struct dfb_frame_io {
    dfb_comm* comm;           /* transforms: root -> all at the head of the step */
    dfb_comm* comm_prefetch;  /* sensor data of the NEXT frame: root -> all, concurrent with the step (its own communicator) */
    int root;
    const float* dq_src;      /* root: this frame's node transforms [n_nodes][8] (pinned host or device), NULL = already in wf->node_dq */
    void* prefetch_dst;       /* device buffer the next frame's sensor data lands in (not the one this step reads) */
    const void* prefetch_src; /* root: its source (pinned host or device), NULL = already in prefetch_dst */
    int64_t prefetch_bytes;
    uint32_t* counters_host;  /* pinned host [8]: ws->counters after the step */
} dfb_frame_io;
typedef struct dfb_frame_step dfb_frame_step;
int dfb_frame_step_create(dfb_frame_step** out);
void dfb_frame_step_destroy(dfb_frame_step* st);
int dfb_frame_step_run(dfb_frame_step* st, const dfb_volume* vol, const dfb_warpfield* wf, const dfb_views* views, double tdist,
                       double wmax, const dfb_workspace* ws, const dfb_frame_io* io, dfb_stream_t stream);
/* out = {captures, in-place updates, replays, un-captured runs, nodes of the last captured graph} */
int dfb_frame_step_stats(const dfb_frame_step* st, int64_t out[5]);

#ifdef __cplusplus
}
#endif
#endif /* DFB_H_ */
