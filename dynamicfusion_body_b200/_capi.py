"""ctypes binding of include/dfb.h (libdfb_b200.so).

There is deliberately no fallback: if the CUDA library has not been built, importing this module
raises, and every product entry point fails with it.  Build with `python -m dynamicfusion_body_b200.build`
(or `__graft_entry__.build()`).
"""
import ctypes as C
import os

DFB_MAX_K = 8
DFB_MAX_VIEWS = 8
DFB_NODE_REC_FLOATS = 12
DFB_COMM_ID_BYTES = 128
MODE_HYBRID = 0
MODE_EXACT = 1
MODE_FAST_ONLY = 2
MODE_LIST_ONLY = 3
MODE_BRICK_CLASSIFY = 4
MODE_BRICK_STREAM = 5
MODE_BRICK_MIXED = 6
MODE_BRICK_UPDATE = 7

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DFB_LIB") or os.path.join(_PKG_DIR, "libdfb_b200.so")   # DFB_LIB: developer override (kernel variants)

c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
c_u8p = C.POINTER(C.c_uint8)
c_u16p = C.POINTER(C.c_uint16)
c_u32p = C.POINTER(C.c_uint32)
c_i32p = C.POINTER(C.c_int32)


class Volume(C.Structure):
    _fields_ = [("tsdf", C.c_void_p), ("weight", C.c_void_p),
                ("rx", C.c_int), ("ry", C.c_int), ("rz", C.c_int),
                ("x0", C.c_int), ("x1", C.c_int)]


class WarpField(C.Structure):
    _fields_ = [("node_rec", C.c_void_p), ("node_pos", C.c_void_p), ("node_dq", C.c_void_p),
                ("node_w", C.c_void_p), ("n_nodes", C.c_int), ("k", C.c_int), ("knn", C.c_void_p),
                ("has_lw", C.c_int), ("lw_is_f32", C.c_int), ("lw", C.c_double * 8),
                ("brick_nodes", C.c_void_p), ("brick_count", C.c_void_p), ("brick_pairs", C.c_void_p),
                ("region_nodes", C.c_void_p), ("region_count", C.c_void_p), ("region_pairs", C.c_void_p),
                ("region_rec", C.c_void_p)]


class Views(C.Structure):
    _fields_ = [("n_views", C.c_int), ("depth", C.c_void_p * DFB_MAX_VIEWS),
                ("rows", C.c_int), ("cols", C.c_int),
                ("K", C.c_double * 9), ("Kinv", C.c_double * 9),
                ("has_extrinsics", C.c_int), ("E", (C.c_double * 12) * DFB_MAX_VIEWS)]


class Workspace(C.Structure):
    _fields_ = [("list", C.c_void_p), ("capacity", C.c_uint32), ("counters", C.c_void_p),
                ("brick_cls", C.c_void_p), ("brick_lists", C.c_void_p), ("overflow_bits", C.c_void_p)]


class GNProblem(C.Structure):
    _fields_ = [("n_vert", C.c_int64), ("vertices", C.c_void_p), ("normals", C.c_void_p), ("corr", C.c_void_p),
                ("vert_knn", C.c_void_p), ("n_nodes", C.c_int), ("k", C.c_int), ("node_pos", C.c_void_p),
                ("node_w", C.c_void_p), ("node_nbr", C.c_void_p), ("lw", C.c_double * 8), ("lw_is_f32", C.c_int),
                ("rw", C.c_double), ("huber", C.c_int), ("f_scale", C.c_double), ("order", C.c_void_p)]


class FrameIO(C.Structure):
    _fields_ = [("comm", C.c_void_p), ("comm_prefetch", C.c_void_p), ("root", C.c_int), ("dq_src", C.c_void_p),
                ("prefetch_dst", C.c_void_p), ("prefetch_src", C.c_void_p), ("prefetch_bytes", C.c_int64),
                ("counters_host", C.c_void_p)]


class PointGrid(C.Structure):
    _fields_ = [("pts", C.c_void_p), ("n", C.c_int64), ("origin", C.c_double * 3), ("cell", C.c_double),
                ("dims", C.c_int * 3), ("cell_start", C.c_void_p), ("order", C.c_void_p)]


def declare(lib):
    """Attach argtypes/restype for every entry point of include/dfb.h present in `lib`."""
    vp = C.c_void_p
    sig = {
        "version": ([], C.c_int),
        "last_error": ([], C.c_char_p),
        "nodes_pack": ([vp, vp, vp, C.c_int, vp, vp], C.c_int),
        "knn_build_volume": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp], C.c_int),
        "knn_brick_count": ([C.c_int, C.c_int, C.c_int], C.c_int64),
        "knn_build_volume_radii": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp], C.c_int),
        "knn_update_volume": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp], C.c_int),
        "brick_nodes_update": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp], C.c_int),
        "region_update": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp], C.c_int),
        "brick_count": ([C.c_int, C.c_int, C.c_int], C.c_int64),
        "brick_nodes_build": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp], C.c_int),
        "region_count": ([C.c_int, C.c_int, C.c_int], C.c_int64),
        "region_build": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp], C.c_int),
        "knn_points": ([vp, C.c_int64, vp, C.c_int, C.c_int, vp, vp], C.c_int),
        "tsdf_update_projective": ([C.POINTER(Volume), C.POINTER(WarpField), C.POINTER(Views), C.c_double, C.c_double,
                                    C.c_int, C.POINTER(Workspace), vp, vp, vp], C.c_int),
        "fuse_depth_rigid": ([C.POINTER(Volume), C.c_int, vp, C.c_int, C.c_int, c_f64p, c_f64p, c_f64p, C.c_double,
                              c_f64p, C.c_double, C.c_double, C.c_int, C.POINTER(Workspace), vp, vp, vp], C.c_int),
        "tsdf_update_volume": ([C.POINTER(Volume), C.POINTER(WarpField), vp, C.c_int, C.c_int, C.c_int, C.c_double,
                                C.c_double, C.c_int, C.POINTER(Workspace), vp, vp], C.c_int),
        "warp_points": ([vp, vp, C.c_int64, vp, C.POINTER(WarpField), vp, vp, vp], C.c_int),
        "dq_blend_points": ([vp, C.c_int64, vp, C.POINTER(WarpField), vp, vp], C.c_int),
        "gn_residuals": ([C.POINTER(GNProblem), vp, C.c_int, vp, vp], C.c_int),
        "gn_residuals_lw": ([C.POINTER(GNProblem), vp, C.c_int, c_f64p, C.c_int, vp, vp], C.c_int),
        "gn_pattern_rows": ([C.POINTER(GNProblem), vp, vp, vp], C.c_int),
        "gn_pattern_cols": ([C.c_int, vp, vp, vp, vp], C.c_int),
        "gn_normal_eq": ([C.POINTER(GNProblem), vp, vp, vp, C.c_int64, vp, vp, vp, vp], C.c_int),
        "gn_lw_normal_eq": ([C.POINTER(GNProblem), vp, c_f64p, vp, vp, vp, vp], C.c_int),
        "gn_solve_workspace_doubles": ([C.c_int], C.c_int64),
        "point_grid_scratch_ints": ([C.c_int64], C.c_int64),
        "point_grid_build": ([C.POINTER(PointGrid), vp, vp, vp, vp], C.c_int),
        "point_grid_knn": ([C.POINTER(PointGrid), vp, C.c_int64, C.c_int, vp, vp, vp], C.c_int),
        "corr_select": ([vp, vp, C.c_int64, vp, vp, C.c_int, vp, vp, vp], C.c_int),
        "corr_projective": ([vp, vp, C.c_int64, C.POINTER(Views), C.c_double, C.c_double, vp, vp, vp, vp], C.c_int),
        "render_workspace_words": ([C.c_int64, C.c_int, C.c_int, C.c_int], C.c_int64),
        "render": ([vp, C.c_int64, vp, C.c_int64, C.POINTER(Views), vp, C.c_int64, vp, vp, vp, vp], C.c_int),
        "track_workspace_doubles": ([C.c_int, C.c_int, C.c_int], C.c_int64),
        "track_normal_eq": ([C.POINTER(Volume), C.c_int, C.c_double, c_f64p, vp, C.c_int, C.c_int, c_f64p, c_f64p, c_f64p, C.c_int,
                             C.c_double, C.c_double, vp, C.c_int64, vp, vp, vp], C.c_int),
        "raycast": ([C.POINTER(Volume), C.c_int, C.c_double, c_f64p, C.POINTER(Views), C.c_double, C.c_double, C.c_double,
                     C.c_double, vp, vp, vp], C.c_int),
        "graph_unsupported": ([vp, C.c_int64, vp, C.c_int, vp, vp, vp, vp], C.c_int),
        "graph_sample_rounds": ([C.POINTER(PointGrid), C.c_double, C.c_int, vp, vp, vp], C.c_int),
        "mc_level_scratch_floats": ([], C.c_int64),
        "mc_level": ([vp, C.c_int64, vp, vp, vp], C.c_int),
        "mc_rows": ([C.c_int, C.c_int, C.c_int], C.c_int64),
        "mc_chunks": ([C.c_int, C.c_int, C.c_int, C.c_int], C.c_int64),
        "mc_count": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp], C.c_int),
        "mc_emit": ([vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "gn_solve": ([C.c_int, vp, vp, vp, vp, C.c_double, C.c_int, C.c_double, vp, vp, vp, vp, vp], C.c_int),
        "comm_available": ([], C.c_int),
        "comm_unique_id": ([vp], C.c_int),
        "comm_init": ([C.POINTER(vp), vp, C.c_int, C.c_int, C.c_int], C.c_int),
        "comm_destroy": ([vp], C.c_int),
        "comm_rank": ([vp], C.c_int),
        "comm_world": ([vp], C.c_int),
        "comm_broadcast": ([vp, vp, C.c_int64, C.c_int, vp], C.c_int),
        "comm_broadcast_frame": ([vp, vp, C.c_int64, vp, C.c_int, vp, C.c_int, vp], C.c_int),
        "comm_allreduce_f64": ([vp, vp, C.c_int64, C.c_int, vp], C.c_int),
        "comm_sendrecv": ([vp, vp, C.c_int64, C.c_int, vp, C.c_int64, C.c_int, vp], C.c_int),
        "frame_step_create": ([C.POINTER(vp)], C.c_int),
        "frame_step_destroy": ([vp], None),
        "frame_step_run": ([vp, C.POINTER(Volume), C.POINTER(WarpField), C.POINTER(Views), C.c_double, C.c_double,
                            C.POINTER(Workspace), C.POINTER(FrameIO), vp], C.c_int),
        "frame_step_stats": ([vp, C.POINTER(C.c_int64)], C.c_int),
    }
    for name, (argtypes, restype) in sig.items():
        fn = getattr(lib, "dfb_" + name, None)
        if fn is None:
            continue
        fn.argtypes = argtypes
        fn.restype = restype
    return lib


_lib = None


def lib():
    """The CUDA library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ImportError(
                "libdfb_b200.so is not built (%s). There is no CPU fallback: run "
                "`python -m dynamicfusion_body_b200.build` (needs nvcc)." % LIB_PATH)
        _lib = declare(C.CDLL(LIB_PATH))
    return _lib


class DfbError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = lib().dfb_last_error()
        raise DfbError("libdfb_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))


EXPORTS = [
    "dfb_version", "dfb_last_error", "dfb_nodes_pack", "dfb_knn_build_volume", "dfb_knn_points", "dfb_brick_count", "dfb_brick_nodes_build", "dfb_region_count", "dfb_region_build",
    "dfb_tsdf_update_projective", "dfb_tsdf_update_volume", "dfb_fuse_depth_rigid", "dfb_warp_points", "dfb_dq_blend_points",
    "dfb_gn_residuals", "dfb_gn_residuals_lw", "dfb_gn_pattern_rows", "dfb_gn_pattern_cols", "dfb_gn_normal_eq",
    "dfb_gn_lw_normal_eq", "dfb_gn_solve_workspace_doubles", "dfb_gn_solve",
    "dfb_point_grid_scratch_ints", "dfb_point_grid_build", "dfb_point_grid_knn", "dfb_corr_select", "dfb_corr_projective", "dfb_render_workspace_words", "dfb_render",
    "dfb_track_workspace_doubles", "dfb_track_normal_eq", "dfb_raycast", "dfb_graph_unsupported", "dfb_graph_sample_rounds",
    "dfb_mc_level_scratch_floats", "dfb_mc_level", "dfb_mc_rows", "dfb_mc_chunks", "dfb_mc_count", "dfb_mc_emit",
    "dfb_knn_brick_count", "dfb_knn_build_volume_radii", "dfb_knn_update_volume", "dfb_brick_nodes_update", "dfb_region_update",
    "dfb_comm_available", "dfb_comm_unique_id", "dfb_comm_init", "dfb_comm_destroy", "dfb_comm_rank", "dfb_comm_world",
    "dfb_comm_broadcast", "dfb_comm_broadcast_frame", "dfb_comm_allreduce_f64", "dfb_comm_sendrecv",
    "dfb_frame_step_create", "dfb_frame_step_destroy", "dfb_frame_step_run", "dfb_frame_step_stats",
]
