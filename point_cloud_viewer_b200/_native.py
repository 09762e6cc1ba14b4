"""ctypes bindings of include/pcv.h (libpcv_b200.so).

The shared library is the product; this module is plumbing.  It fails loudly when the CUDA extension
has not been built (there is no CPU or pure-Python fallback)."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCV_B200_LIB") or os.path.join(_HERE, "libpcv_b200.so")  # env override: kernel-variant experiments only

PCV_OK = 0
ERR_NAMES = {
    -1: "PCV_ERR_INVALID",
    -2: "PCV_ERR_CUDA",
    -3: "PCV_ERR_IO",
    -4: "PCV_ERR_NOT_FOUND",
    -5: "PCV_ERR_CANCELLED",
    -6: "PCV_ERR_UNSUPPORTED",
    -7: "PCV_ERR_SINGULAR",
}


class PcvError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (ERR_NAMES.get(code, code), msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("max_points_per_node", C.c_uint64), ("levels_per_pass", C.c_uint32), ("reserved", C.c_uint32)]


class Points(C.Structure):
    _fields_ = [
        ("x", C.c_void_p),
        ("y", C.c_void_p),
        ("z", C.c_void_p),
        ("stride", C.c_uint64),
        ("rgb", C.c_void_p),
        ("intensity", C.c_void_p),
        ("n", C.c_uint64),
    ]


class NodeMeta(C.Structure):
    _fields_ = [
        ("id_high", C.c_uint64),
        ("id_low", C.c_uint64),
        ("num_points", C.c_int64),
        ("position_encoding", C.c_int32),
        ("level", C.c_int32),
        ("cube_min", C.c_double * 3),
        ("cube_edge", C.c_double),
        ("point_offset", C.c_uint64),
        ("xyz_byte_offset", C.c_uint64),
    ]


class Location(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("pad", C.c_int32),
        ("aabb_min", C.c_double * 3),
        ("aabb_max", C.c_double * 3),
        ("clip_from_query", C.c_double * 16),
        ("query_from_clip", C.c_double * 16),
        ("query_from_obb", C.c_double * 7),
        ("obb_from_query", C.c_double * 7),
        ("half_extent", C.c_double * 3),
    ]


class Interval(C.Structure):
    _fields_ = [("lo", C.c_double), ("hi", C.c_double)]


class Batch(C.Structure):
    _fields_ = [("n", C.c_uint64), ("xyz", C.c_void_p), ("rgb", C.c_void_p), ("intensity", C.c_void_p), ("src_index", C.c_void_p)]


BATCH_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(Batch))


class BuildStats(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_uint64),
        ("passes", C.c_uint32),
        ("deepest_level", C.c_uint32),
        ("num_nodes", C.c_uint64),
        ("algorithmic_bytes", C.c_uint64),
        ("ms_host_plan", C.c_float),
        ("ms_partition", C.c_float),
        ("ms_place", C.c_float),
        ("ms_total", C.c_float),
        ("ms_host_wait", C.c_float),
    ]


class QueryStats(C.Structure):
    """pcv_query_stats (include/pcv.h)."""

    _fields_ = [("ms_device", C.c_float), ("ms_select", C.c_float), ("ms_cull", C.c_float), ("kernel_launches", C.c_uint32), ("algorithmic_bytes", C.c_uint64),
                ("tested_points", C.c_uint64), ("returned_points", C.c_uint64), ("stored_points", C.c_uint64), ("visited_pairs", C.c_uint64)]


class QueryOut(C.Structure):
    """pcv_query_out (include/pcv.h): caller-owned device buffers for the survivors of pcv_query_batch_device."""

    _fields_ = [("xyz", C.c_void_p), ("rgb", C.c_void_p), ("intensity", C.c_void_p), ("src_index", C.c_void_p), ("loc", C.c_void_p),
                ("cap", C.c_uint64), ("stored", C.c_uint64)]


class XrayStats(C.Structure):
    """pcv_xray_stats (include/pcv.h)."""

    _fields_ = [("ms_device", C.c_float), ("kernel_launches", C.c_uint32), ("points", C.c_uint64), ("algorithmic_bytes", C.c_uint64)]


class XrayQuadtreeParams(C.Structure):
    """pcv_xray_quadtree_params (include/pcv.h)."""

    _fields_ = [("strategy", C.c_int32), ("p0", C.c_float), ("p1", C.c_float), ("colormap", C.c_int32), ("bin_size", C.c_double),
                ("has_query_from_global", C.c_int32), ("query_from_global", C.c_double * 7), ("background", C.c_uint8 * 4),
                ("tile_size_px", C.c_uint32), ("pixel_size_m", C.c_double), ("root_level", C.c_uint8), ("root_index", C.c_uint64)]


class XrayQuadtreeInfo(C.Structure):
    """pcv_xray_quadtree_info (include/pcv.h)."""

    _fields_ = [("rect_min_x", C.c_double), ("rect_min_y", C.c_double), ("rect_edge", C.c_double), ("deepest_level", C.c_uint8),
                ("tile_size_px", C.c_uint32), ("num_nodes", C.c_uint32), ("num_leaves", C.c_uint32), ("ms_leaves", C.c_float),
                ("ms_parents", C.c_float), ("kernel_launches", C.c_uint32), ("leaf_points", C.c_uint64)]


XRAY_TILE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint8, C.c_uint64, C.POINTER(C.c_uint8), C.c_uint32)


class KernelStat(C.Structure):
    _fields_ = [("name", C.c_char * 24), ("launches", C.c_uint64), ("algorithmic_bytes", C.c_uint64), ("ms", C.c_double)]


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.c_uint64)
ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p)
BARRIER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p)


class Comm(C.Structure):  # pcv_comm
    _fields_ = [("user", C.c_void_p), ("rank", C.c_int), ("world", C.c_int), ("allreduce_sum_u64", ALLREDUCE_FN), ("allgather", ALLGATHER_FN), ("barrier", BARRIER_FN)]


class PlyInfo(C.Structure):
    """pcv_ply_info (include/pcv.h)."""

    _fields_ = [("num_points", C.c_uint64), ("header_bytes", C.c_uint64), ("record_bytes", C.c_uint32), ("has_color", C.c_int32),
                ("has_intensity", C.c_int32), ("type_xyz", C.c_int32 * 3), ("off_xyz", C.c_uint32 * 3), ("off_rgb", C.c_uint32 * 3),
                ("off_intensity", C.c_uint32), ("offset", C.c_double * 3)]


# every symbol include/pcv.h declares: (name, restype, argtypes)
_dp = C.POINTER(C.c_double)
_u64p = C.POINTER(C.c_uint64)
SYMBOLS = [
    ("pcv_create", C.c_int, [C.c_int, C.POINTER(Config), C.POINTER(C.c_void_p)]),
    ("pcv_destroy", None, [C.c_void_p]),
    ("pcv_last_error", C.c_char_p, []),
    ("pcv_device_count", C.c_int, []),
    ("pcv_bbox", C.c_int, [C.c_void_p, C.POINTER(Points), _dp, _dp]),
    ("pcv_bbox_device", C.c_int, [C.c_void_p, C.POINTER(Points), _dp, _dp]),
    ("pcv_build_octree", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_double, _dp, _dp, C.POINTER(C.c_void_p)]),
    ("pcv_build_octree_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_double, _dp, _dp, C.POINTER(C.c_void_p)]),
    ("pcv_octree_free", None, [C.c_void_p]),
    ("pcv_octree_info", C.c_int, [C.c_void_p, _u64p, _u64p, _u64p, _dp, _dp, _dp, C.POINTER(C.c_int)]),
    ("pcv_octree_nodes", C.c_int, [C.c_void_p, C.POINTER(NodeMeta), C.c_uint64]),
    ("pcv_octree_node_data", C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_nodes_data_blob", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, _u64p]),
    ("pcv_octree_shuffle_nodes", C.c_int, [C.c_void_p, C.c_uint64]),
    ("pcv_lod_order", C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]),
    ("pcv_octree_download", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_octree_device_arrays", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    ("pcv_octree_write_dir", C.c_int, [C.c_void_p, C.c_char_p]),
    ("pcv_octree_load_dir", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    ("pcv_nodes_in_location", C.c_int, [C.c_void_p, C.POINTER(Location), C.c_void_p, C.c_uint64, _u64p]),
    ("pcv_visible_nodes", C.c_int, [C.c_void_p, _dp, C.c_void_p, C.c_uint64, _u64p]),
    ("pcv_query_points", C.c_int, [C.c_void_p, C.POINTER(Location), C.c_void_p, C.c_uint32, C.c_uint64, BATCH_CB, C.c_void_p]),
    ("pcv_query_batch_device", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(QueryOut)]),
    ("pcv_last_query_stats", C.c_int, [C.c_void_p, C.POINTER(QueryStats)]),
    ("pcv_last_xray_stats", C.c_int, [C.c_void_p, C.POINTER(XrayStats)]),
    ("pcv_xray_tile", C.c_int, [C.c_void_p, _dp, _dp, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    ("pcv_xray_tile_attr", C.c_int, [C.c_void_p, _dp, _dp, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    ("pcv_xray_tile_attr_binned", C.c_int, [C.c_void_p, _dp, _dp, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_double, C.c_void_p, C.POINTER(C.c_int)]),
    ("pcv_xray_assign_background", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    ("pcv_xray_build_parent", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]),
    ("pcv_xray_quadtree", C.c_int, [C.c_void_p, C.POINTER(XrayQuadtreeParams), XRAY_TILE_FN, C.c_void_p, C.POINTER(XrayQuadtreeInfo)]),
    ("pcv_xray_quadtree_write_dir", C.c_int, [C.c_void_p, C.POINTER(XrayQuadtreeParams), C.c_char_p, C.POINTER(XrayQuadtreeInfo)]),
    ("pcv_s2_cell_ids", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_uint32, C.c_void_p]),
    ("pcv_s2_build", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_uint32, C.POINTER(C.c_void_p)]),
    ("pcv_s2_build_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_uint32, C.POINTER(C.c_void_p)]),
    ("pcv_s2_free", None, [C.c_void_p]),
    ("pcv_s2_info", C.c_int, [C.c_void_p, _u64p, _u64p, C.POINTER(C.c_uint32), _dp, _dp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("pcv_s2_cells", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_s2_build_stats", C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint32), _u64p]),
    ("pcv_s2_cell_data", C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_s2_cells_in_union", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, _u64p]),
    ("pcv_s2_query_union", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, _u64p, _u64p]),
    ("pcv_s2_write_dir", C.c_int, [C.c_void_p, C.c_char_p]),
    ("pcv_s2_load_dir", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    ("pcv_s2_union_contains", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_void_p, C.c_uint32, C.c_void_p]),
    ("pcv_prefix_histogram_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_double, _dp, _dp, C.c_uint32, C.c_void_p]),
    ("pcv_prefix_histogram_bbox_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_double, _dp, _dp, C.c_uint32, C.c_void_p, _dp, _dp]),
    ("pcv_prefix_pack_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_void_p, C.c_uint64, C.c_double, _dp, _dp, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_prefix_pack_exchange_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_void_p, C.c_uint64, C.c_double, _dp, _dp, C.c_uint32, C.c_void_p, C.c_uint32,
                                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_unpack_colours_device", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    ("pcv_ipc_alloc", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.c_void_p]),
    ("pcv_ipc_free", C.c_int, [C.c_void_p, C.c_void_p]),
    ("pcv_ipc_open", C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("pcv_ipc_close", C.c_int, [C.c_void_p, C.c_void_p]),
    ("pcv_shard_ingest_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_double, _dp, _dp, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("pcv_shard_exchange_device", C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_shard_send_info", C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("pcv_shard_send_dest", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), _u64p]),
    ("pcv_shard_send_free", None, [C.c_void_p]),
    ("pcv_build_octree_from_records_device", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, _dp, _dp, C.c_uint32, C.c_void_p,
                                                       C.POINTER(C.c_void_p)]),
    ("pcv_build_octree_sharded", C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Points), C.c_double, _dp, _dp, C.c_uint32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                           C.POINTER(C.c_uint32), C.c_void_p, C.c_void_p, _u64p, C.POINTER(C.c_void_p)]),
    ("pcv_shard_pass_device", C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_build_octree_after_pass_device", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_double, _dp, _dp, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("pcv_shard_send_cells", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), _u64p]),
    ("pcv_sharded_release", C.c_int, [C.c_void_p, C.c_void_p]),
    ("pcv_release_cached_memory", C.c_int, [C.c_void_p]),
    ("pcv_sharded_phases", C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    ("pcv_build_octree_sharded_device", C.c_int, [C.c_void_p, C.POINTER(Points), C.c_double, _dp, _dp, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("pcv_octree_node_nsub", C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, _u64p]),
    ("pcv_octree_nsub_all", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    ("pcv_assemble_top", C.c_int, [C.c_void_p, C.c_double, _dp, _dp, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    ("pcv_ply_read_header", C.c_int, [C.c_char_p, C.POINTER(PlyInfo)]),
    ("pcv_ply_unpack_device", C.c_int, [C.c_void_p, C.POINTER(PlyInfo), C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _dp, _dp]),
    ("pcv_ply_load_device", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(PlyInfo), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, _dp, _dp]),
    ("pcv_build_octree_from_file", C.c_int, [C.c_void_p, C.c_char_p, C.c_double, C.c_int, C.POINTER(C.c_void_p)]),
    ("pcv_synth_points_device", C.c_int, [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_synth_points_host", C.c_int, [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("pcv_synth_bbox", C.c_int, [C.c_int, _dp, _dp, _dp]),
    ("pcv_device_alloc", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    ("pcv_device_free", C.c_int, [C.c_void_p, C.c_void_p]),
    ("pcv_last_build_stats", C.c_int, [C.c_void_p, C.POINTER(BuildStats)]),
    ("pcv_kernel_launch_count", C.c_uint64, [C.c_void_p]),
    ("pcv_set_profiling", C.c_int, [C.c_void_p, C.c_int]),
    ("pcv_kernel_stats", C.c_int, [C.c_void_p, C.POINTER(KernelStat), C.c_uint32, C.POINTER(C.c_uint32)]),
]

_lib = None


def lib():
    """Load libpcv_b200.so; raise (never fall back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "point_cloud_viewer_b200: %s is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH
            )
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != PCV_OK:
        raise PcvError(rc, lib().pcv_last_error().decode("utf-8", "replace"))
