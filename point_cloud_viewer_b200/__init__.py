"""point_cloud_viewer_b200 — B200-native octree builder + LOD / frustum point-query engine.

The product is the CUDA shared library behind include/pcv.h (csrc/).  This package is the thin host
layer used by tests and bench.py: it mirrors the names of the reference's interface for this path
(build_octree, Octree.get_visible_nodes / get_node_data / nodes_in_location, PointQuery streaming)
and never computes on the CPU — every call goes through the C ABI and fails loudly without a GPU.
"""
import ctypes as C
import os

import numpy as np

from . import _native as N
from . import geometry
from ._native import PcvError, Location  # noqa: F401

ENC_BYTES = {1: 1, 2: 2, 3: 4, 4: 8}
NODE_DTYPE = np.dtype([("id_high", "<u8"), ("id_low", "<u8"), ("num_points", "<i8"), ("enc", "<i4"), ("level", "<i4"), ("cube", "<f8", (4,)),
                       ("point_offset", "<u8"), ("xyz_byte_offset", "<u8")])
SYNTH_SLAB_ECEF, SYNTH_GAUSS_CLUSTERS = 1, 2


def _d3(v):
    return (C.c_double * 3)(*[float(x) for x in v])


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return a
    return a.ctypes.data


def node_name(hi, lo):
    """NodeId Display: 'r' + octal path (src/octree/node.rs:73-86)."""
    v = (int(hi) << 64) | int(lo)
    level = v >> 120
    return "r" + "".join(str((v >> (3 * i)) & 7) for i in range(level - 1, -1, -1))


def node_id_from_name(name):
    level = len(name) - 1
    idx = int(name[1:], 8) if level else 0
    v = (level << 120) | idx
    return v >> 64, v & 0xFFFFFFFFFFFFFFFF


def device_count():
    return N.lib().pcv_device_count()


XRAY_COLORED, XRAY_INTENSITY, XRAY_HEIGHT_STDDEV = 1, 2, 3


class Context:
    """One per GPU (pcv_ctx)."""

    def __init__(self, device=0, max_points_per_node=0, levels_per_pass=0):
        cfg = N.Config(max_points_per_node, levels_per_pass, 0)
        h = C.c_void_p()
        N.check(N.lib().pcv_create(device, C.byref(cfg), C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if self.h:
            N.lib().pcv_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- a1
    def bbox(self, x, y, z, stride=1, n=None, device=False):
        n = int(n if n is not None else (len(x) if stride == 1 else len(x) // 1))
        pts = N.Points(_p(x), _p(y), _p(z), stride, None, None, n)
        mn, mx = (C.c_double * 3)(), (C.c_double * 3)()
        fn = N.lib().pcv_bbox_device if device else N.lib().pcv_bbox
        N.check(fn(self.h, C.byref(pts), mn, mx))
        return np.array(mn), np.array(mx)

    # -- build_octree (generation.rs:289-295): returns an Octree resident in HBM
    def build_octree(self, x, y, z, rgb, resolution, bbox_min, bbox_max, intensity=None, stride=1, n=None, device=False):
        if n is None:
            n = len(rgb) // 3 if getattr(rgb, "ndim", 1) == 1 else rgb.shape[0]
        keep = (x, y, z, rgb, intensity)  # keep host arrays alive during the call
        pts = N.Points(_p(x), _p(y), _p(z), stride, _p(rgb), _p(intensity), int(n))
        out = C.c_void_p()
        fn = N.lib().pcv_build_octree_device if device else N.lib().pcv_build_octree
        N.check(fn(self.h, C.byref(pts), float(resolution), _d3(bbox_min), _d3(bbox_max), C.byref(out)))
        del keep
        return Octree(self, out)

    # -- S2-cell point cloud (src/read_write/s2.rs, src/s2_cells/mod.rs)
    def s2_cell_ids(self, x, y, z, level, stride=1, n=None):
        """CellID::from_point(p).parent(level) for host points."""
        n = int(n if n is not None else len(x) // (1 if stride == 1 else 1))
        pts = N.Points(_p(x), _p(y), _p(z), stride, None, None, n)
        out = np.zeros(n, np.uint64)
        N.check(N.lib().pcv_s2_cell_ids(self.h, C.byref(pts), int(level), _p(out)))
        return out

    def build_s2_cloud(self, x, y, z, rgb=None, intensity=None, split_level=20, stride=1, n=None, device=False):
        """S2Splitter::write over the whole cloud + get_meta (read_write/s2.rs:52-125,165-173): an S2Cloud resident in HBM."""
        if n is None:
            n = len(x)
        keep = (x, y, z, rgb, intensity)
        pts = N.Points(_p(x), _p(y), _p(z), stride, _p(rgb), _p(intensity), int(n))
        out = C.c_void_p()
        fn = N.lib().pcv_s2_build_device if device else N.lib().pcv_s2_build
        N.check(fn(self.h, C.byref(pts), int(split_level), C.byref(out)))
        del keep
        return S2Cloud(self, out)

    def load_s2_dir(self, directory):
        """S2Cells::from_data_provider over an on-disk S2 directory."""
        out = C.c_void_p()
        N.check(N.lib().pcv_s2_load_dir(self.h, os.fsencode(str(directory)), C.byref(out)))
        return S2Cloud(self, out)

    def s2_union_contains(self, x, y, z, union_ids, stride=1, n=None):
        """CellUnion as PointCulling (geometry/s2_cell_union.rs:27-31): boolean mask over host points."""
        n = int(n if n is not None else len(x))
        pts = N.Points(_p(x), _p(y), _p(z), stride, None, None, n)
        u = np.ascontiguousarray(union_ids, np.uint64)
        mask = np.zeros(n, np.uint8)
        N.check(N.lib().pcv_s2_union_contains(self.h, C.byref(pts), _p(u), len(u), _p(mask)))
        return mask.astype(bool)

    # -- PLY input (src/read_write/ply.rs, generation.rs:256-287)
    def load_ply(self, path):
        """PlyIterator + find_bounding_box in one pass: the file's points as device SoA arrays.  Returns a PlyPoints."""
        info = ply_read_header(path)
        return PlyPoints(self, path, info)

    def ply_unpack_device(self, info, records_ptr, n, x_ptr, y_ptr, z_ptr, rgb_ptr=None, intensity_ptr=None):
        mn, mx = (C.c_double * 3)(), (C.c_double * 3)()
        N.check(N.lib().pcv_ply_unpack_device(self.h, C.byref(info), records_ptr, int(n), x_ptr, y_ptr, z_ptr, rgb_ptr, intensity_ptr, mn, mx))
        return np.array(mn), np.array(mx)

    def build_octree_from_file(self, path, resolution, attributes=("color",)):
        """build_octree_from_file (generation.rs:272-287) without the directory: the octree stays resident in HBM."""
        out = C.c_void_p()
        N.check(N.lib().pcv_build_octree_from_file(self.h, os.fsencode(str(path)), float(resolution), 1 if "intensity" in attributes else 0, C.byref(out)))
        return Octree(self, out)

    def load_dir(self, directory):
        out = C.c_void_p()
        N.check(N.lib().pcv_octree_load_dir(self.h, str(directory).encode(), C.byref(out)))
        return Octree(self, out)

    def device_buffer(self, shape, typestr):
        """Device memory from the context's pool, viewable by torch through __cuda_array_interface__ (typestr e.g. '<f8')."""
        return DeviceBuffer(self, shape, typestr)

    def last_build_stats(self):
        s = N.BuildStats()
        N.check(N.lib().pcv_last_build_stats(self.h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in N.BuildStats._fields_}

    def set_profiling(self, on):
        N.check(N.lib().pcv_set_profiling(self.h, 1 if on else 0))

    def kernel_stats(self):
        arr = (N.KernelStat * 16)()
        n = C.c_uint32()
        N.check(N.lib().pcv_kernel_stats(self.h, arr, 16, C.byref(n)))
        return {arr[i].name.decode(): dict(launches=arr[i].launches, algorithmic_bytes=arr[i].algorithmic_bytes, ms=arr[i].ms) for i in range(n.value)}

    def kernel_launch_count(self):
        return int(N.lib().pcv_kernel_launch_count(self.h))

    def synth_points_device(self, kind, seed, first, n, x_ptr, y_ptr, z_ptr, rgb_ptr):
        N.check(N.lib().pcv_synth_points_device(self.h, kind, seed, first, n, x_ptr, y_ptr, z_ptr, rgb_ptr))

    def prefix_histogram_device(self, x, y, z, n, resolution, bbox_min, bbox_max, k, stride=1):
        pts = N.Points(_p(x), _p(y), _p(z), stride, None, None, int(n))
        counts = np.zeros(8 ** k, np.uint64)
        N.check(N.lib().pcv_prefix_histogram_device(self.h, C.byref(pts), float(resolution), _d3(bbox_min), _d3(bbox_max), k, _p(counts)))
        return counts

    def prefix_histogram_bbox_device(self, x, y, z, n, resolution, bbox_min, bbox_max, k, stride=1):
        """Level-k cell histogram of the local points + their bounding box, one pass over the positions."""
        pts = N.Points(_p(x), _p(y), _p(z), stride, None, None, int(n))
        counts = np.zeros(8 ** k, np.uint64)
        mn, mx = (C.c_double * 3)(), (C.c_double * 3)()
        N.check(N.lib().pcv_prefix_histogram_bbox_device(self.h, C.byref(pts), float(resolution), _d3(bbox_min), _d3(bbox_max), k, _p(counts), mn, mx))
        return counts, np.array(mn), np.array(mx)

    def prefix_pack_device(self, x, y, z, rgb, intensity, gidx, gidx_base, n, resolution, bbox_min, bbox_max, k, cell_to_rank, nranks, out_xyz,
                           out_rgb, out_intensity, out_idx, stride=1):
        pts = N.Points(_p(x), _p(y), _p(z), stride, _p(rgb), _p(intensity), int(n))
        c2r = np.ascontiguousarray(cell_to_rank, np.int32)
        counts = np.zeros(nranks, np.uint64)
        N.check(N.lib().pcv_prefix_pack_device(self.h, C.byref(pts), _p(gidx), int(gidx_base), float(resolution), _d3(bbox_min), _d3(bbox_max), k,
                                               _p(c2r), nranks, _p(out_xyz), _p(out_rgb), _p(out_intensity), _p(out_idx), _p(counts)))
        return counts

    def prefix_pack_exchange_device(self, x, y, z, rgb, intensity, gidx_base, n, resolution, bbox_min, bbox_max, k, cell_to_rank, nranks, dst_first,
                                    dst_x, dst_y, dst_z, dst_index, dst_intensity, dst_colour):
        """Fused pack + exchange (pcv.h): dst_* are lists of device pointers (one per rank, as mapped in this process)."""
        pts = N.Points(_p(x), _p(y), _p(z), 1, _p(rgb), _p(intensity), int(n))
        c2r = np.ascontiguousarray(cell_to_rank, np.int32)
        first = np.ascontiguousarray(dst_first, np.uint64)
        arr = lambda lst: (C.c_void_p * nranks)(*[int(v) if v else None for v in lst])
        ax, ay, az, ai, ac = arr(dst_x), arr(dst_y), arr(dst_z), arr(dst_index), arr(dst_colour)
        an = arr(dst_intensity) if dst_intensity is not None else None
        counts = np.zeros(nranks, np.uint64)
        N.check(N.lib().pcv_prefix_pack_exchange_device(self.h, C.byref(pts), None, int(gidx_base), float(resolution), _d3(bbox_min), _d3(bbox_max), k,
                                                        _p(c2r), nranks, _p(first), ax, ay, az, ai, an, ac, _p(counts)))
        return counts

    def unpack_colours_device(self, colour_ptr, n, rgb_ptr):
        N.check(N.lib().pcv_unpack_colours_device(self.h, colour_ptr, int(n), rgb_ptr))

    def ipc_alloc(self, nbytes):
        p, h = C.c_void_p(), (C.c_uint8 * 64)()
        N.check(N.lib().pcv_ipc_alloc(self.h, int(nbytes), C.byref(p), h))
        return p.value, bytes(h)

    def ipc_free(self, ptr):
        N.check(N.lib().pcv_ipc_free(self.h, ptr))

    def ipc_open(self, handle):
        p = C.c_void_p()
        hb = (C.c_uint8 * 64).from_buffer_copy(handle)
        N.check(N.lib().pcv_ipc_open(self.h, hb, C.byref(p)))
        return p.value

    def ipc_close(self, ptr):
        N.check(N.lib().pcv_ipc_close(self.h, ptr))

    # ---- exchange of ingested records (pcv.h: pcv_shard_*) ----
    def shard_ingest(self, x, y, z, rgb, intensity, n, resolution, bbox_min, bbox_max, k):
        """Ingest step + digit histogram of the local points: (level-k cell counts, send handle)."""
        pts = N.Points(_p(x), _p(y), _p(z), 1, _p(rgb), _p(intensity), int(n))
        counts = np.zeros(8 ** k, np.uint64)
        h = C.c_void_p()
        N.check(N.lib().pcv_shard_ingest_device(self.h, C.byref(pts), float(resolution), _d3(bbox_min), _d3(bbox_max), k, _p(counts), C.byref(h)))
        return counts, h

    def shard_exchange(self, send, k, cell_to_rank, nranks, dst_first, dst_rec, dst_col, dst_dig, dst_intensity=None):
        c2r = np.ascontiguousarray(cell_to_rank, np.int32)
        first = np.ascontiguousarray(dst_first, np.uint64)
        arr = lambda lst: (C.c_void_p * nranks)(*[int(v) if v else None for v in lst])
        counts = np.zeros(nranks, np.uint64)
        N.check(N.lib().pcv_shard_exchange_device(send, k, _p(c2r), nranks, _p(first), arr(dst_rec), arr(dst_col) if dst_col is not None else None, arr(dst_dig),
                                                  arr(dst_intensity) if dst_intensity is not None else None, _p(counts)))
        return counts

    def shard_send_info(self, send):
        w, g = C.c_int(), C.c_int()
        N.check(N.lib().pcv_shard_send_info(send, C.byref(w), C.byref(g)))
        return bool(w.value), g.value

    def shard_send_dest(self, send):
        p, n = C.c_void_p(), C.c_uint64()
        N.check(N.lib().pcv_shard_send_dest(send, C.byref(p), C.byref(n)))
        return p.value, n.value

    def shard_send_free(self, send):
        N.lib().pcv_shard_send_free(send)

    def build_octree_sharded(self, comm_struct, x_ptr, y_ptr, z_ptr, stride, rgb_ptr, intensity_ptr, n, resolution, bbox_min, bbox_max, prefix_levels=2, keep_send=True):
        """pcv_build_octree_sharded: the whole multi-GPU build in one C call per rank; `comm_struct` is a _native.Comm.
        Returns (local Octree, top Octree or None, k, cell_to_rank, unit_nsub, points owned, send handle or None)."""
        pts = N.Points(x_ptr, y_ptr, z_ptr, stride, rgb_ptr, intensity_ptr, int(n))
        local, top, send, k, nrecv = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_uint32(), C.c_uint64()
        c2r = np.zeros(8 ** prefix_levels, np.int32)
        un = np.zeros(8 ** prefix_levels, np.uint64)
        N.check(N.lib().pcv_build_octree_sharded(self.h, C.addressof(comm_struct), C.byref(pts), float(resolution), _d3(bbox_min), _d3(bbox_max), prefix_levels,
                                                 C.byref(local), C.byref(top), C.byref(k), _p(c2r), _p(un), C.byref(nrecv), C.byref(send) if keep_send else None))
        kk = int(k.value)
        return (Octree(self, local), Octree(self, top) if top.value else None, kk, c2r[: 8 ** kk].copy(), un[: 8 ** kk].copy(), int(nrecv.value),
                send if keep_send else None)

    def shard_send_cells(self, send):
        """(device pointer, n) of the per-point level-2 cells a fused exchange pass leaves with the handle; None if the handle went
        through the exchange of ingested records instead."""
        ptr, n = C.c_void_p(), C.c_uint64()
        if N.lib().pcv_shard_send_cells(send, C.byref(ptr), C.byref(n)) != 0:
            return None
        return (ptr.value or 0), int(n.value)

    def release_cached_memory(self):
        N.check(N.lib().pcv_release_cached_memory(self.h))

    def sharded_phases(self):
        """Per-phase wall-clock milliseconds of the last build_octree_sharded on this context."""
        out = (C.c_double * 6)()
        N.check(N.lib().pcv_sharded_phases(self.h, out))
        names = ("ingest + histogram", "all-reduce + plan", "exchange", "local build", "top assembly")
        d = {nm: float(out[i]) for i, nm in enumerate(names)}
        d["fused_exchange_pass"] = bool(out[5])
        return d

    def sharded_release(self, comm_struct):
        N.check(N.lib().pcv_sharded_release(self.h, C.addressof(comm_struct)))

    def build_octree_from_records(self, rec_ptr, col_ptr, dig_ptr, intensity_ptr, n, resolution, bbox_min, bbox_max, k, prefix_counts):
        """The owner's part of a sharded build over the records its peers stored into its slab."""
        pc = np.ascontiguousarray(prefix_counts, np.uint64)
        out = C.c_void_p()
        N.check(N.lib().pcv_build_octree_from_records_device(self.h, rec_ptr, col_ptr, dig_ptr, intensity_ptr, int(n), float(resolution), _d3(bbox_min), _d3(bbox_max),
                                                             k, _p(pc), C.byref(out)))
        return Octree(self, out)

    def build_octree_sharded_device_soa(self, x_ptr, y_ptr, z_ptr, rgb_ptr, intensity_ptr, n, resolution, bbox_min, bbox_max, k, prefix_counts):
        """Local part of a sharded build from SoA device arrays (the layout the fused exchange delivers)."""
        pts = N.Points(x_ptr, y_ptr, z_ptr, 1, rgb_ptr, intensity_ptr, int(n))
        pc = np.ascontiguousarray(prefix_counts, np.uint64)
        out = C.c_void_p()
        N.check(N.lib().pcv_build_octree_sharded_device(self.h, C.byref(pts), float(resolution), _d3(bbox_min), _d3(bbox_max), k, _p(pc), C.byref(out)))
        return Octree(self, out)

    def build_octree_sharded_device(self, xyz_ptr, rgb_ptr, intensity_ptr, n, resolution, bbox_min, bbox_max, k, prefix_counts):
        """Local part of a sharded build: AoS xyz (n*3 f64) device pointer; prefix_counts = global counts of levels 1..k."""
        pts = N.Points(xyz_ptr, xyz_ptr + 8, xyz_ptr + 16, 3, rgb_ptr, intensity_ptr, int(n))
        pc = np.ascontiguousarray(prefix_counts, np.uint64)
        out = C.c_void_p()
        N.check(N.lib().pcv_build_octree_sharded_device(self.h, C.byref(pts), float(resolution), _d3(bbox_min), _d3(bbox_max), k, _p(pc), C.byref(out)))
        return Octree(self, out)

    def assemble_top(self, resolution, bbox_min, bbox_max, k, prefix_counts, unit_nsub, xyz_codes, rgb, intensity):
        pc = np.ascontiguousarray(prefix_counts, np.uint64)
        un = np.ascontiguousarray(unit_nsub, np.uint64)
        npts = len(rgb) // 3
        out = C.c_void_p()
        N.check(N.lib().pcv_assemble_top(self.h, float(resolution), _d3(bbox_min), _d3(bbox_max), k, _p(pc), _p(un), _p(xyz_codes), _p(rgb), _p(intensity),
                                         npts, C.byref(out)))
        return Octree(self, out)


class DeviceBuffer:
    """A block of the context's stream-ordered pool exposed through __cuda_array_interface__ (zero-copy torch view)."""

    def __init__(self, ctx, shape, typestr):
        self.ctx = ctx
        self.shape = tuple(int(s) for s in shape)
        itemsize = int(typestr[2:])
        nbytes = itemsize
        for s in self.shape:
            nbytes *= s
        p = C.c_void_p()
        N.check(N.lib().pcv_device_alloc(ctx.h, max(nbytes, 16), C.byref(p)))
        self.ptr = p.value
        self.__cuda_array_interface__ = {"shape": self.shape, "typestr": typestr, "data": (self.ptr, False), "version": 2, "strides": None}

    def tensor(self):
        import torch

        t = torch.as_tensor(self, device="cuda:%d" % self.ctx.device)
        t._pcv_owner = self  # keep the block alive as long as the view
        return t

    def free(self):
        if self.ptr and self.ctx.h:
            N.lib().pcv_device_free(self.ctx.h, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def lod_order(seed, name, n):
    """new_order of node `name` with n points: shuffled[i] = original[new_order[i]] (reshuffle, node_drawer.rs:34-43)."""
    hi, lo = node_id_from_name(name)
    out = np.zeros(max(int(n), 1), np.uint64)
    N.check(N.lib().pcv_lod_order(int(seed), hi, lo, int(n), _p(out)))
    return out[: int(n)]


def synth_points_host(kind, seed, first, n):
    x, y, z = np.empty(n), np.empty(n), np.empty(n)
    rgb = np.empty(n * 3, np.uint8)
    N.check(N.lib().pcv_synth_points_host(kind, seed, first, n, _p(x), _p(y), _p(z), _p(rgb)))
    return x, y, z, rgb


def synth_bbox(kind):
    mn, mx, res = (C.c_double * 3)(), (C.c_double * 3)(), C.c_double()
    N.check(N.lib().pcv_synth_bbox(kind, mn, mx, C.byref(res)))
    return np.array(mn), np.array(mx), res.value


class Octree:
    """Mirror of point_viewer::octree::Octree (src/octree/mod.rs:141-358) over a pcv_octree."""

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self.h = handle
        nn, npts, xb, res = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_double()
        mn, mx, hi = (C.c_double * 3)(), (C.c_double * 3)(), C.c_int()
        N.check(N.lib().pcv_octree_info(self.h, C.byref(nn), C.byref(npts), C.byref(xb), C.byref(res), mn, mx, C.byref(hi)))
        self.num_points, self.xyz_bytes, self.resolution = npts.value, xb.value, res.value
        self.bbox_min, self.bbox_max, self.has_intensity = np.array(mn), np.array(mx), bool(hi.value)
        arr = (N.NodeMeta * max(nn.value, 1))()
        N.check(N.lib().pcv_octree_nodes(self.h, arr, nn.value))
        self.node_array = arr
        self.num_nodes = nn.value
        # structured numpy view of the node table (no per-node Python objects until someone asks for `nodes`)
        self.meta = np.frombuffer(arr, dtype=NODE_DTYPE, count=nn.value) if nn.value else np.zeros(0, NODE_DTYPE)
        self._nodes = None
        self._order = None

    @property
    def nodes(self):
        if self._nodes is None:
            self._nodes, self._order = {}, []
            for m in self.meta:
                name = node_name(m["id_high"], m["id_low"])
                self._order.append(name)
                self._nodes[name] = dict(
                    num_points=int(m["num_points"]),
                    enc=int(m["enc"]),
                    level=int(m["level"]),
                    cube=(float(m["cube"][0]), float(m["cube"][1]), float(m["cube"][2]), float(m["cube"][3])),
                    hi=int(m["id_high"]),
                    lo=int(m["id_low"]),
                    point_offset=int(m["point_offset"]),
                    xyz_byte_offset=int(m["xyz_byte_offset"]),
                )
        return self._nodes

    @property
    def order(self):
        self.nodes
        return self._order

    def nsub_all(self):
        out = np.zeros(max(self.num_nodes, 1), np.uint64)
        N.check(N.lib().pcv_octree_nsub_all(self.h, _p(out), self.num_nodes))
        return out[: self.num_nodes]

    def node_data_at(self, i):
        """node_data by position in the node table."""
        m = self.meta[i]
        n, bpc = int(m["num_points"]), ENC_BYTES[int(m["enc"])]
        xyz, rgb = np.zeros(n * 3 * bpc, np.uint8), np.zeros(n * 3, np.uint8)
        inten = np.zeros(n, np.float32) if self.has_intensity else None
        src = np.zeros(n, np.uint64)
        N.check(N.lib().pcv_octree_node_data(self.h, int(m["id_high"]), int(m["id_low"]), _p(xyz), _p(rgb), _p(inten), _p(src)))
        return xyz, rgb, inten, src

    def free(self):
        # pcv_octree_free works through the owning pcv_ctx, so it must not run once that context is destroyed (an octree that
        # outlives Context.close(), e.g. one collected at interpreter exit)
        if self.h and self.ctx.h:
            N.lib().pcv_octree_free(self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # Octree::get_node_data (octree/mod.rs:285-307) (+ provenance)
    def node_data(self, name):
        m = self.nodes[name]
        n, bpc = m["num_points"], ENC_BYTES[m["enc"]]
        xyz, rgb = np.zeros(n * 3 * bpc, np.uint8), np.zeros(n * 3, np.uint8)
        inten = np.zeros(n, np.float32) if self.has_intensity else None
        src = np.zeros(n, np.uint64)
        N.check(N.lib().pcv_octree_node_data(self.h, m["hi"], m["lo"], _p(xyz), _p(rgb), _p(inten), _p(src)))
        return xyz, rgb, inten, src

    def nodes_data_blob(self, names, out=None):
        """`/nodes_data` of the web viewer (octree_web_viewer/src/backend.rs:92-165): one binary reply for a list of node names,
        gathered on the GPU from the resident octree.  `out`: optional (pinned) uint8 array to receive the blob."""
        ids = np.zeros(2 * len(names), np.uint64)
        for k, nm in enumerate(names):
            ids[2 * k], ids[2 * k + 1] = node_id_from_name(nm)
        size = C.c_uint64()
        N.check(N.lib().pcv_nodes_data_blob(self.h, _p(ids), len(names), None, 0, C.byref(size)))
        if out is None:
            out = np.zeros(max(size.value, 1), np.uint8)
        N.check(N.lib().pcv_nodes_data_blob(self.h, _p(ids), len(names), _p(out), out.nbytes if hasattr(out, "nbytes") else len(out), C.byref(size)))
        return out[: size.value]

    def shuffle_nodes(self, seed):
        """Apply the viewers' random draw order to every node, once, on the GPU (node_drawer.rs:185-205; mod.rs:286-287)."""
        N.check(N.lib().pcv_octree_shuffle_nodes(self.h, int(seed)))

    def node_nsub(self, name):
        m = self.nodes[name]
        v = C.c_uint64()
        N.check(N.lib().pcv_octree_node_nsub(self.h, m["hi"], m["lo"], C.byref(v)))
        return v.value

    def download(self, xyz=None, rgb=None, intensity=None, src=None, want_src=True):
        xyz = np.zeros(max(self.xyz_bytes, 1), np.uint8) if xyz is None else xyz
        rgb = np.zeros(max(self.num_points * 3, 1), np.uint8) if rgb is None else rgb
        if intensity is None and self.has_intensity:
            intensity = np.zeros(self.num_points, np.float32)
        if src is None and want_src:
            src = np.zeros(max(self.num_points, 1), np.uint64)
        N.check(N.lib().pcv_octree_download(self.h, _p(xyz), _p(rgb), _p(intensity), _p(src)))
        return xyz, rgb, intensity, src

    def write_dir(self, directory):
        N.check(N.lib().pcv_octree_write_dir(self.h, str(directory).encode()))

    # PointCloud::nodes_in_location (octree/mod.rs:329-331)
    def nodes_in_location(self, loc):
        cap = len(self.nodes) + 1
        out = np.zeros(2 * cap, np.uint64)
        n = C.c_uint64()
        N.check(N.lib().pcv_nodes_in_location(self.h, C.byref(loc), _p(out), cap, C.byref(n)))
        return [node_name(out[2 * i], out[2 * i + 1]) for i in range(n.value)]

    # Octree::get_visible_nodes (octree/mod.rs:228)
    def get_visible_nodes(self, clip_from_world):
        m = np.asarray(clip_from_world, np.float64)
        flat = m.T.reshape(-1) if m.ndim == 2 else m
        cap = len(self.nodes) + 1
        out = np.zeros(2 * cap, np.uint64)
        n = C.c_uint64()
        N.check(N.lib().pcv_visible_nodes(self.h, (C.c_double * 16)(*[float(v) for v in flat]), _p(out), cap, C.byref(n)))
        return [node_name(out[2 * i], out[2 * i + 1]) for i in range(n.value)]

    # ParallelIterator::try_for_each_batch semantics (iterator.rs:255-333) on the caller's thread
    def query_points(self, loc, callback=None, filters=(), batch_size=500000):
        """Streams batches dict(xyz (n,3) f64, rgb (n,3), intensity, src).  A callback returning a truthy
        value cancels the stream (ErrorKind::Channel); without a callback the batches are returned."""
        f = np.asarray(filters, np.float64).reshape(-1)
        nf = len(f) // 2
        got = []

        def tramp(_user, bp):
            b = bp.contents
            n = b.n
            d = dict(
                xyz=np.ctypeslib.as_array(C.cast(b.xyz, C.POINTER(C.c_double)), (n, 3)).copy() if n else np.zeros((0, 3)),
                rgb=np.ctypeslib.as_array(C.cast(b.rgb, C.POINTER(C.c_uint8)), (n, 3)).copy() if n else np.zeros((0, 3), np.uint8),
                intensity=np.ctypeslib.as_array(C.cast(b.intensity, C.POINTER(C.c_float)), (n,)).copy() if (n and b.intensity) else None,
                src=np.ctypeslib.as_array(C.cast(b.src_index, C.POINTER(C.c_uint64)), (n,)).copy() if n else np.zeros(0, np.uint64),
            )
            if callback is None:
                got.append(d)
                return 0
            return 1 if callback(d) else 0

        cb = N.BATCH_CB(tramp)
        rc = N.lib().pcv_query_points(self.h, C.byref(loc), _p(f) if nf else None, nf, int(batch_size), cb, None)
        if rc == -5:
            raise PcvError(rc, "cancelled by callback")
        N.check(rc)
        return got

    def query_batch_device(self, locs, filters=(), points=False, cap=None):
        """Per-location survivor and tested counts of a batch of locations.  points=True also returns the survivors, copied to
        the host: dict(loc, src (u32), xyz (n,3) f64, rgb (n,3), intensity or None, stored), in no particular order.  They land
        in device buffers of `cap` points; cap=None sizes them to the survivor total with a first, counting call."""
        arr = (N.Location * len(locs))(*locs)
        f = np.asarray(filters, np.float64).reshape(-1)
        nf = len(f) // 2
        counts, tested = np.zeros(len(locs), np.uint64), np.zeros(len(locs), np.uint64)
        if not points:
            N.check(N.lib().pcv_query_batch_device(self.h, arr, len(locs), _p(f) if nf else None, nf, _p(counts), _p(tested), None))
            return counts, tested
        if cap is None:
            cap = int(self.query_batch_device(locs, filters)[0].sum())
        cap = int(cap)
        ctx, rows = self.ctx, max(cap, 1)
        bufs = dict(xyz=ctx.device_buffer((rows, 3), "<f8"), rgb=ctx.device_buffer((rows, 3), "|u1"), src=ctx.device_buffer((rows,), "<i4"),
                    loc=ctx.device_buffer((rows,), "<i4"))
        if self.has_intensity:
            bufs["intensity"] = ctx.device_buffer((rows,), "<f4")
        try:
            out = N.QueryOut(bufs["xyz"].ptr, bufs["rgb"].ptr, bufs["intensity"].ptr if self.has_intensity else None, bufs["src"].ptr, bufs["loc"].ptr, cap, 0)
            N.check(N.lib().pcv_query_batch_device(self.h, arr, len(locs), _p(f) if nf else None, nf, _p(counts), _p(tested), C.byref(out)))
            n = int(out.stored)
            got = {k: b.tensor()[:n].cpu().numpy() for k, b in bufs.items()}  # the call has synchronised the context's stream
        finally:
            for b in bufs.values():
                b.free()
        got["src"], got["loc"] = got["src"].view(np.uint32), got["loc"].view(np.uint32)
        got.setdefault("intensity", None)
        got["stored"] = n
        return counts, tested, got

    def last_query_stats(self):
        """Timing / traffic of the last query_batch_device call (pcv_query_stats)."""
        st = N.QueryStats()
        N.check(N.lib().pcv_last_query_stats(self.ctx.h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in N.QueryStats._fields_}

    def last_xray_stats(self):
        st = N.XrayStats()
        N.check(N.lib().pcv_last_xray_stats(self.ctx.h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in N.XrayStats._fields_}

    def xray_tile(self, tile_min, tile_max, w, h, query_from_global=None, want_bits=False):
        rgba = np.zeros((h, w, 4), np.uint8)
        zb = np.zeros((h, w, 32), np.uint32) if want_bits else None
        anyp = C.c_int()
        q = (C.c_double * 7)(*[float(v) for v in query_from_global]) if query_from_global is not None else None
        N.check(N.lib().pcv_xray_tile(self.h, _d3(tile_min), _d3(tile_max), w, h, q, _p(rgba), _p(zb), C.byref(anyp)))
        return bool(anyp.value), rgba, zb

    def xray_tile_attr(self, tile_min, tile_max, w, h, strategy, p0=0.0, p1=0.0, colormap=0, query_from_global=None):
        """strategy: XRAY_COLORED / XRAY_INTENSITY (p0 = min, p1 = max) / XRAY_HEIGHT_STDDEV (p0 = max_stddev, colormap 0 Jet, 1 Purplish)."""
        rgba = np.zeros((h, w, 4), np.uint8)
        anyp = C.c_int()
        q = (C.c_double * 7)(*[float(v) for v in query_from_global]) if query_from_global is not None else None
        N.check(N.lib().pcv_xray_tile_attr(self.h, _d3(tile_min), _d3(tile_max), w, h, q, int(strategy), float(p0), float(p1), int(colormap), _p(rgba),
                                           C.byref(anyp)))
        return bool(anyp.value), rgba


    def xray_tile_attr_binned(self, tile_min, tile_max, w, h, strategy, bin_size, p0=0.0, p1=0.0, query_from_global=None):
        """XRAY_COLORED / XRAY_INTENSITY with Binning = Some(("intensity", bin_size)) (xray/src/generation.rs:129-157)."""
        rgba = np.zeros((h, w, 4), np.uint8)
        anyp = C.c_int()
        q = (C.c_double * 7)(*[float(v) for v in query_from_global]) if query_from_global is not None else None
        N.check(N.lib().pcv_xray_tile_attr_binned(self.h, _d3(tile_min), _d3(tile_max), w, h, q, int(strategy), float(p0), float(p1), float(bin_size),
                                                  _p(rgba), C.byref(anyp)))
        return bool(anyp.value), rgba

    def xray_quadtree(self, tile_size_px, pixel_size_m, strategy=0, p0=0.0, p1=0.0, colormap=0, bin_size=0.0, query_from_global=None,
                      background=(255, 255, 255, 255), root=(0, 0), on_tile=None, keep_tiles=True):
        """build_xray_quadtree (xray/src/generation.rs:560-622) on the GPU: returns (info dict, {(level, index): RGBA array}).
        `on_tile(level, index, rgba)` is called for every finished tile (return a true value to cancel)."""
        pr = N.XrayQuadtreeParams()
        pr.strategy, pr.p0, pr.p1, pr.colormap, pr.bin_size = int(strategy), float(p0), float(p1), int(colormap), float(bin_size)
        pr.has_query_from_global = 0 if query_from_global is None else 1
        if query_from_global is not None:
            pr.query_from_global = (C.c_double * 7)(*[float(v) for v in query_from_global])
        pr.background = (C.c_uint8 * 4)(*[int(v) for v in background])
        pr.tile_size_px, pr.pixel_size_m = int(tile_size_px), float(pixel_size_m)
        pr.root_level, pr.root_index = int(root[0]), int(root[1])
        tiles = {}

        def cb(_user, level, index, ptr, tpx):
            img = np.ctypeslib.as_array(ptr, shape=(tpx, tpx, 4))
            if keep_tiles:
                tiles[(int(level), int(index))] = img.copy()
            return 1 if (on_tile is not None and on_tile(int(level), int(index), img)) else 0

        info = N.XrayQuadtreeInfo()
        N.check(N.lib().pcv_xray_quadtree(self.h, C.byref(pr), N.XRAY_TILE_FN(cb), None, C.byref(info)))
        return {k: getattr(info, k) for k, _ in N.XrayQuadtreeInfo._fields_}, tiles

    def xray_quadtree_write_dir(self, directory, tile_size_px, pixel_size_m, strategy=0, p0=0.0, p1=0.0, colormap=0, bin_size=0.0, query_from_global=None,
                                background=(255, 255, 255, 255), root=(0, 0)):
        """build_xray_quadtree with the reference's outputs: <directory>/<node id>.png + the quadtree's meta file."""
        pr = _xray_params(tile_size_px, pixel_size_m, strategy, p0, p1, colormap, bin_size, query_from_global, background, root)
        info = N.XrayQuadtreeInfo()
        N.check(N.lib().pcv_xray_quadtree_write_dir(self.h, C.byref(pr), os.fsencode(str(directory)), C.byref(info)))
        return {k: getattr(info, k) for k, _ in N.XrayQuadtreeInfo._fields_}


class S2Cloud:
    """pcv_s2cloud: the S2-cell point cloud (S2Cells / S2Meta of src/s2_cells/mod.rs) resident in HBM."""

    def __init__(self, ctx, handle):
        self.ctx, self.h = ctx, handle
        nc, npnt, lvl = C.c_uint64(), C.c_uint64(), C.c_uint32()
        mn, mx = (C.c_double * 3)(), (C.c_double * 3)()
        hc, hi = C.c_int(), C.c_int()
        N.check(N.lib().pcv_s2_info(self.h, C.byref(nc), C.byref(npnt), C.byref(lvl), mn, mx, C.byref(hc), C.byref(hi)))
        self.num_cells, self.num_points, self.split_level = nc.value, npnt.value, lvl.value
        self.bbox_min, self.bbox_max = np.array(mn), np.array(mx)
        self.has_color, self.has_intensity = bool(hc.value), bool(hi.value)
        self.cell_ids = np.zeros(self.num_cells, np.uint64)
        self.cell_counts = np.zeros(self.num_cells, np.uint64)
        N.check(N.lib().pcv_s2_cells(self.h, _p(self.cell_ids), _p(self.cell_counts)))

    def free(self):
        if self.h and self.ctx.h:  # as Octree.free: pcv_s2_free needs the owning pcv_ctx alive
            N.lib().pcv_s2_free(self.h)
        self.h = None

    def write_dir(self, directory):
        """<token>.xyz / .rgb / .intensity per cell + meta.pb, as S2Splitter<RawNodeWriter> leaves them."""
        N.check(N.lib().pcv_s2_write_dir(self.h, os.fsencode(str(directory))))

    def build_stats(self):
        ms, l, b = C.c_float(), C.c_uint32(), C.c_uint64()
        N.check(N.lib().pcv_s2_build_stats(self.h, C.byref(ms), C.byref(l), C.byref(b)))
        return dict(ms_device=ms.value, kernel_launches=l.value, algorithmic_bytes=b.value)

    def cell_data(self, cell_id):
        """points_in_node: (xyz f64 (n, 3), rgb or None, intensity or None, source index)."""
        k = int(np.searchsorted(self.cell_ids, np.uint64(cell_id)))
        n = int(self.cell_counts[k]) if k < self.num_cells and int(self.cell_ids[k]) == int(cell_id) else 0
        xyz = np.zeros((n, 3), np.float64)
        rgb = np.zeros((n, 3), np.uint8) if self.has_color else None
        inten = np.zeros(n, np.float32) if self.has_intensity else None
        src = np.zeros(n, np.uint64)
        N.check(N.lib().pcv_s2_cell_data(self.h, int(cell_id), _p(xyz), _p(rgb), _p(inten), _p(src)))
        return xyz, rgb, inten, src

    def cells_in_union(self, union_ids=None):
        """nodes_in_location for AllPoints (None) / S2Cells(CellUnion)."""
        u = None if union_ids is None else np.ascontiguousarray(union_ids, np.uint64)
        out = np.zeros(self.num_cells, np.uint64)
        n = C.c_uint64()
        N.check(N.lib().pcv_s2_cells_in_union(self.h, _p(u), 0 if u is None else len(u), _p(out), len(out), C.byref(n)))
        return out[: n.value]

    def query_union(self, union_ids=None, cap=None):
        """The filtered point stream of the location: dict(xyz, rgb, intensity, src, tested)."""
        u = None if union_ids is None else np.ascontiguousarray(union_ids, np.uint64)
        nu = 0 if u is None else len(u)
        n, tested = C.c_uint64(), C.c_uint64()
        if cap is None:
            N.check(N.lib().pcv_s2_query_union(self.h, _p(u), nu, None, None, None, None, 0, C.byref(n), C.byref(tested)))
            cap = n.value
        xyz = np.zeros((cap, 3), np.float64)
        rgb = np.zeros((cap, 3), np.uint8) if self.has_color else None
        inten = np.zeros(cap, np.float32) if self.has_intensity else None
        src = np.zeros(cap, np.uint64)
        N.check(N.lib().pcv_s2_query_union(self.h, _p(u), nu, _p(xyz), _p(rgb), _p(inten), _p(src), cap, C.byref(n), C.byref(tested)))
        m = min(cap, n.value)
        return dict(xyz=xyz[:m], rgb=None if rgb is None else rgb[:m], intensity=None if inten is None else inten[:m], src=src[:m], total=n.value, tested=tested.value)


def s2_token(cell_id):
    """CellID::to_token: the per-cell file stem of the reference's S2 directory layout."""
    if int(cell_id) == 0:
        return "X"
    return ("%016x" % int(cell_id)).rstrip("0")


def xray_node_name(level, index):
    """quadtree NodeId -> its name / PNG stem ("r", "r0", "r123323"; quadtree/src/lib.rs:216-233)."""
    return "r" + "".join(str((int(index) >> (2 * l)) & 3) for l in reversed(range(int(level))))


def xray_node_id(name):
    """NodeId::from_str (quadtree/src/lib.rs:201-213): (level, index)."""
    level = len(name) - 1
    return level, (int(name[1:], 4) if level > 0 else 0)


def _xray_params(tile_size_px, pixel_size_m, strategy, p0, p1, colormap, bin_size, query_from_global, background, root):
    pr = N.XrayQuadtreeParams()
    pr.strategy, pr.p0, pr.p1, pr.colormap, pr.bin_size = int(strategy), float(p0), float(p1), int(colormap), float(bin_size)
    pr.has_query_from_global = 0 if query_from_global is None else 1
    if query_from_global is not None:
        pr.query_from_global = (C.c_double * 7)(*[float(v) for v in query_from_global])
    pr.background = (C.c_uint8 * 4)(*[int(v) for v in background])
    pr.tile_size_px, pr.pixel_size_m = int(tile_size_px), float(pixel_size_m)
    pr.root_level, pr.root_index = int(root[0]), int(root[1])
    return pr


def xray_assign_background(ctx, rgba, background):
    """assign_background (xray/src/generation.rs:695-720) in place on a C-contiguous (..., 4) uint8 array."""
    bg = np.asarray(background, np.uint8)
    assert rgba.dtype == np.uint8 and rgba.flags.c_contiguous and rgba.shape[-1] == 4 and bg.shape == (4,)
    N.check(N.lib().pcv_xray_assign_background(ctx.h, _p(rgba), rgba.size // 4, _p(bg)))
    return rgba


def xray_build_parent(ctx, children, background, tile_px):
    """build_parent + Lanczos3 reduction (xray/src/generation.rs:410-451, 722-759).  children: 4 x (N, N, 4) uint8 or None."""
    child_px = next(c.shape[0] for c in children if c is not None)
    keep = [np.ascontiguousarray(c, np.uint8) if c is not None else None for c in children]
    for c in keep:
        assert c is None or c.shape == (child_px, child_px, 4)
    ptrs = (C.c_void_p * 4)(*[_p(c) for c in keep])
    bg = np.asarray(background, np.uint8)
    out = np.zeros((tile_px, tile_px, 4), np.uint8)
    N.check(N.lib().pcv_xray_build_parent(ctx.h, ptrs, child_px, _p(bg), tile_px, _p(out)))
    return out


def ply_read_header(path):
    """parse_header + the property checks of PlyIterator::from_file (ply.rs:126-229, 327-450) -> pcv_ply_info."""
    info = N.PlyInfo()
    N.check(N.lib().pcv_ply_read_header(os.fsencode(str(path)), C.byref(info)))
    return info


class PlyPoints:
    """The points of a PLY file on the device: x, y, z (f64, header offset added), rgb (n*3 u8), intensity (f32) as
    DeviceBuffers, plus the bounding box the reference's find_bounding_box pass would return."""

    def __init__(self, ctx, path, info):
        self.ctx, self.info, self.n = ctx, info, int(info.num_points)
        n = self.n
        self.x, self.y, self.z = (ctx.device_buffer((max(n, 1),), "<f8") for _ in range(3))
        self.rgb = ctx.device_buffer((max(3 * n, 1),), "|u1") if info.has_color else None
        self.intensity = ctx.device_buffer((max(n, 1),), "<f4") if info.has_intensity else None
        mn, mx = (C.c_double * 3)(), (C.c_double * 3)()
        N.check(N.lib().pcv_ply_load_device(ctx.h, os.fsencode(str(path)), C.byref(info), self.x.ptr, self.y.ptr, self.z.ptr,
                                            self.rgb.ptr if self.rgb else None, self.intensity.ptr if self.intensity else None, mn, mx))
        self.bbox_min, self.bbox_max = np.array(mn), np.array(mx)

    def batches(self, batch_size):
        """The PointsBatch stream of PlyIterator (ply.rs:522-556): ceil(n / batch_size) host batches, the last one short."""
        x, y, z = (b.tensor()[: self.n].cpu().numpy() for b in (self.x, self.y, self.z))
        rgb = self.rgb.tensor()[: 3 * self.n].cpu().numpy().reshape(-1, 3) if self.rgb else None
        inten = self.intensity.tensor()[: self.n].cpu().numpy() if self.intensity else None
        for first in range(0, self.n, batch_size):
            sl = slice(first, min(first + batch_size, self.n))
            b = {"position": np.stack([x[sl], y[sl], z[sl]], 1)}
            if rgb is not None:
                b["color"] = rgb[sl]
            if inten is not None:
                b["intensity"] = inten[sl]
            yield b

    def build_octree(self, resolution, with_intensity=False):
        return self.ctx.build_octree(self.x.ptr, self.y.ptr, self.z.ptr, self.rgb.ptr if self.rgb else None, resolution, self.bbox_min, self.bbox_max,
                                     intensity=self.intensity.ptr if (with_intensity and self.intensity) else None, n=self.n, device=True)

    def free(self):
        for b in (self.x, self.y, self.z, self.rgb, self.intensity):
            if b is not None:
                b.free()


def build_octree_from_file(output_directory, resolution, filename, attributes=("color",), device=0, ctx=None):
    """Drop-in shape of point_viewer::octree::build_octree_from_file (src/octree/generation.rs:272-287)."""
    own = ctx is None
    ctx = ctx or Context(device)
    tree = ctx.build_octree_from_file(filename, resolution, attributes)
    tree.write_dir(output_directory)
    if own:
        tree.free()
        ctx.close()
        return None
    return tree


def build_octree(output_directory, resolution, bounding_box, batches, attributes=("color",), device=0, ctx=None):
    """Drop-in shape of point_viewer::octree::build_octree (src/octree/generation.rs:289-295):
    drains `batches` (iterable of dict(position (n,3) f64, color (n,3) u8[, intensity (n,) f32])), builds on
    the GPU, writes the reference's directory layout.  bounding_box = (min3, max3)."""
    pos, col, inten = [], [], []
    for b in batches:
        pos.append(np.ascontiguousarray(b["position"], np.float64).reshape(-1, 3))
        col.append(np.ascontiguousarray(b["color"], np.uint8).reshape(-1, 3))
        if "intensity" in b and "intensity" in attributes:
            inten.append(np.ascontiguousarray(b["intensity"], np.float32).reshape(-1))
    P = np.concatenate(pos) if pos else np.zeros((0, 3))
    Cc = np.concatenate(col) if col else np.zeros((0, 3), np.uint8)
    I = np.concatenate(inten) if inten else None
    own = ctx is None
    ctx = ctx or Context(device)
    flat = P.reshape(-1)
    tree = ctx.build_octree(flat[0:], flat[1:], flat[2:], Cc.reshape(-1), resolution, bounding_box[0], bounding_box[1], intensity=I, stride=3, n=len(P))
    tree.write_dir(output_directory)
    if own:
        tree.free()
        ctx.close()
        return None
    return tree
