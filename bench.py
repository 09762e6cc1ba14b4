#!/usr/bin/env python
"""bench.py — build_octree (+ frustum query, X-ray tiles) throughput on B200, one JSON line on rank 0.

  python bench.py --gpus N --steps K --warmup W          the CUDA path (this repo)
  python bench.py --impl reference --gpus N ...           the reference's CPU algorithm (oracle port) on the host cores
  python bench.py --gpus 1 ... --dump-outputs DIR         also write the last timed step's octree as DIR/*.npy (see dump_outputs)

A step = one build_octree over one batch of synthetic points (BASELINE.json config 2: Gaussian clusters in a 1024 m cube,
resolution 1024/2^20 -> depth 20, 1e9 points per GPU).  At N > 1 every rank owns the same number of points of one global index
space (weak scaling; config 4 = 8e9 points on 8 GPUs): the points shard by level-2 octree prefix and move once to their owners
over NVLink (one fused rank + peer-store kernel, CUDA-IPC mapped receive slabs; NCCL carries only the small all-reduces).
`value` = points / device time of the step (a CUDA event pair around the call, host planning included, max over ranks) with the
inputs resident in HBM; `e2e` = the same build through the C-ABI host entry point: pinned host buffers -> H2D -> build -> D2H
of the node arrays, all inside the timed region.  Next to it (N = 1): per-kernel roofline from CUDA events on the library's
stream, the frustum query and X-ray tile workloads (configs 3 and 5) with their own rooflines and CPU baselines, the reference's
own bench sizes (config 1), a parity verdict of the GPU octree against the oracle on a sample of the same generator, and - last,
in a child process (scripts/xray_pyramid_bench.py) - the whole X-ray quadtree and the S2-cell split (SURVEY 8 f3 / f4), each
with device time, HBM fraction, CPU port and parity verdict.  N > 1 lines carry parity and full-size checks, the phase
breakdown and the whole-build roofline per GPU.

The reference arm never loads the CUDA library: generator, in-memory and file-backed ("faithful") builds all come from oracle/.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 1
METRIC = "build_octree Mpoints/sec"
UNIT = "Mpoints/s"
SLAB_SEED = 80293751232  # point_cloud_test/src/lib.rs:46


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp"

    def __init__(self, index=0):
        self.p = None
        self.index = index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def window(self, t0, t1):
        """Only samples taken inside [t0, t1] (time.time()) count: the sampler is started before the warm-up so that nvidia-smi's
        own start-up (it initialises NVML and takes driver locks for hundreds of milliseconds) stays out of the timed steps."""
        self.t0, self.t1 = t0, t1

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        import datetime

        t0, t1 = getattr(self, "t0", None), getattr(self, "t1", None)
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            if t0 is not None and len(f) >= 7:
                try:
                    ts = datetime.datetime.strptime(f[6], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    if ts < t0 - 0.05 or ts > t1 + 0.05:
                        continue
                except ValueError:
                    pass
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm and t0 is not None:  # a timed region shorter than the sampling period: fall back to every sample of the run
            self.t0 = self.t1 = None
            self.p = type("Done", (), {"terminate": lambda s: None, "communicate": lambda s, timeout=None: (out, ""), "kill": lambda s: None})()
            return self.stop()
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def workload_config(n, world, args):
    """The `config` object of the JSON line - shared by both arms so that the reference arm names the same workload."""
    return {
        "workload": "build_octree on %d synthetic Gaussian-cluster points per GPU (BASELINE config %d), resolution 1024/2^20 (depth 20), XYZ f64 SoA + RGB" % (n, 2 if world == 1 else 4),
        "points_per_gpu": n, "levels_per_pass": 2, "max_points_per_node": 100000,
        "l2": "inputs (%.1f GB per GPU) are larger than L2; no flush needed" % (27.0 * n / 1e9),
        "parallelism": "single GPU" if world == 1 else "points shard by level-%d octree prefix; one fused rank + peer-store kernel moves every point into its owner's memory over NVLink (CUDA IPC), NCCL only for the small all-reduces" % args.prefix_levels,
    }


def _shm_dir():
    d = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else tempfile.gettempdir()
    return tempfile.mkdtemp(prefix="pcv_bench_", dir=d)


def cpu_build_times(O, x, y, z, rgb3, res, bmin, bmax, cores, steps_mem, steps_faithful):
    """Oracle build_octree, both variants (BASELINE.md 2): in memory and with the reference's file round trips (/dev/shm)."""
    tm, tf = [], []
    for _ in range(steps_mem):
        t0 = time.perf_counter()
        o = O.build(x, y, z, rgb3, res, bmin, bmax, num_threads=cores)
        tm.append(time.perf_counter() - t0)
        del o
    for _ in range(steps_faithful):
        d = _shm_dir()
        try:
            t0 = time.perf_counter()
            O.build_faithful(x, y, z, rgb3, res, bmin, bmax, d, num_threads=cores)
            tf.append(time.perf_counter() - t0)
        finally:
            shutil.rmtree(d, ignore_errors=True)
    return tm, tf


def config1_cpu(O, cores):
    """The reference's own bench shapes (point_cloud_test/benches/main.rs:10-19, src/lib.rs:42-61): 1e5 and 1e6 slab points,
    resolution 0.001, on the oracle (both variants)."""
    out = {}
    bmin, bmax, res = O.synth_bbox(O.SYNTH_SLAB_ECEF)
    th = min(cores, 10)  # build_octree's default: 10 rayon threads (src/bin/build_octree.rs:37)
    for n in (100_000, 1_000_000):
        x, y, z, rgb = O.synth_points(O.SYNTH_SLAB_ECEF, SLAB_SEED, 0, n, num_threads=cores)
        tm, tf = cpu_build_times(O, x, y, z, rgb.reshape(-1, 3), res, bmin, bmax, th, 3, 2)
        out[str(n)] = {"in_memory_ms": min(tm) * 1e3, "faithful_ms": min(tf) * 1e3, "Mpoints_per_s": n / min(min(tm), min(tf)) / 1e6, "threads": th}
    return out


def run_reference(args):
    """The reference's own algorithm on the host cores: the oracle (C++ restatement of build_octree with the reference's task
    structure: serial root split, one task per split node, per-level parallel subsampling), in memory and file-backed.  Each
    step builds a bounded sample (default 1e8 points) of the N = 1 workload; the line's value is the faster variant."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_api as O

    n = int(args.ref_points)
    cores = os.cpu_count() or 1
    x, y, z, rgb = O.synth_points(O.SYNTH_GAUSS_CLUSTERS, SEED, 0, n, num_threads=cores)
    bmin, bmax, res = O.synth_bbox(O.SYNTH_GAUSS_CLUSTERS)
    rgb3 = rgb.reshape(-1, 3)
    cpu_build_times(O, x, y, z, rgb3, res, bmin, bmax, cores, min(args.warmup, 1), 0)
    tm, tf = cpu_build_times(O, x, y, z, rgb3, res, bmin, bmax, cores, args.steps, min(args.steps, 3))
    ms_mem, ms_f = sum(tm) / len(tm) * 1e3, sum(tf) / len(tf) * 1e3
    ms = min(ms_mem, ms_f)
    v = n / (ms * 1e3)
    full = int(args.points)
    sample = "first %d points of the same generator per step, %d threads; in-memory %.0f ms (%d steps), faithful (/dev/shm node files) %.0f ms (%d steps); value = the faster" % (
        n, cores, ms_mem, len(tm), ms_f, len(tf))
    cfg = workload_config(full, args.gpus, args)
    cfg.update(sample_points_per_step=n, same_config=(n == full),
               note="the reference's CPU algorithm (oracle port) timed on a bounded sample of this workload: the ratio to the GPU arm extrapolates the per-point rate")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "variants": {"in_memory_Mpoints_per_s": n / (ms_mem * 1e3), "faithful_Mpoints_per_s": n / (ms_f * 1e3)},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    try:
        line["config1"] = config1_cpu(O, cores)
    except Exception as e:
        line["config1"] = {"error": str(e)[:200]}
    print(json.dumps(line))


def make_frusta(G, bmin, bmax, count, far, seed=7):
    """SURVEY 8d config 3: eye uniform in the bbox, orientation = normalised 4-vector of Irwin-Hall variates,
    Perspective3(aspect 1.0, fovy 1.2, near 0.1, far) as in point_cloud_test/src/queries.rs:38-44."""
    import numpy as np

    rng = np.random.default_rng(seed)
    locs = []
    persp = G.Perspective.new_fov(1.0, 1.2, 0.1, far)
    for _ in range(count):
        eye = bmin + rng.random(3) * (bmax - bmin)
        q = rng.random((4, 12)).sum(1) - 6.0
        q /= np.linalg.norm(q)
        locs.append(G.frustum(G.Isometry(eye, q), persp))
    return locs


def bench_ply(ctx, pcv, n, peak):
    """build_octree_from_file's input side on a synthetic xyz-f32 + rgb-u8 PLY (15-byte records, page-cache resident)."""
    import numpy as np

    d = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
    path = os.path.join(d, "pcv_bench_%d_%d.ply" % (os.getpid(), n))
    rec = np.zeros(n, dtype=np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("red", "u1"), ("green", "u1"), ("blue", "u1")]))
    rng = np.random.default_rng(0)
    for k, scale in (("x", 200.0), ("y", 200.0), ("z", 20.0)):
        rec[k] = rng.random(n, dtype=np.float32) * scale
    rec["red"] = np.arange(n, dtype=np.uint32) & 255
    try:
        with open(path, "wb") as f:
            f.write(("ply\nformat binary_little_endian 1.0\ncomment offset: 4100000 660000 4700000\nelement vertex %d\nproperty float x\nproperty float y\n"
                     "property float z\nproperty uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n" % n).encode())
            rec.tofile(f)
        del rec
        fbytes = os.path.getsize(path)
        ctx.load_ply(path).free()  # warm-up: pinned ring, pool
        ctx.set_profiling(True)
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            pp = ctx.load_ply(path)
            times.append((time.perf_counter() - t0) * 1e3)
            pp.free()
        ks = ctx.kernel_stats()["k_ply_unpack"]
        ctx.set_profiling(False)
        ms = sorted(times)[1]
        t0 = time.perf_counter()
        tree = ctx.build_octree_from_file(path, 0.001)
        bms = (time.perf_counter() - t0) * 1e3
        nodes = int(tree.num_nodes)
        tree.free()
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_api as O

        m = min(n, 5_000_000)
        t0 = time.perf_counter()
        O.ply_read(path, 0, m)
        cms = (time.perf_counter() - t0) * 1e3
        kg = ks["algorithmic_bytes"] / (ks["ms"] * 1e-3) / 1e9 if ks["ms"] > 0 else 0.0
        return {"workload": "%d-point binary PLY (x,y,z float + r,g,b uchar, %d-byte records), page-cache resident" % (n, fbytes // max(1, n)),
                "load_ms": ms, "Mpoints_per_s": n / (ms * 1e3), "file_GB_per_s": fbytes / (ms * 1e-3) / 1e9, "h2d_bytes": fbytes,
                "kernel": {"name": "k_ply_unpack", "launches": ks["launches"], "ms": ks["ms"], "achieved_GBps": kg, "frac_of_hbm_peak": kg / peak,
                           "algorithmic_bytes": ks["algorithmic_bytes"]},
                "build_octree_from_file_ms": bms, "build_octree_from_file_Mpoints_per_s": n / (bms * 1e3), "octree_nodes": nodes,
                "cpu_baseline": {"value": m / (cms * 1e3), "unit": "Mpoints/s", "cores": 1, "kind": "port",
                                 "sample": "first %d points through the oracle restatement of PlyIterator (single thread, as the reference)" % m}}
    finally:
        if os.path.exists(path):
            os.remove(path)


def bench_config1(ctx, pcv, torch, O, cores):
    """BASELINE config 1 on the GPU: the reference's bench shapes (1e5 and 1e6 slab points) through the host entry point
    (pageable numpy arrays in, octree resident) and device resident, next to the oracle on the host cores."""
    out = {}
    bmin, bmax, res = pcv.synth_bbox(pcv.SYNTH_SLAB_ECEF)
    cpu = config1_cpu(O, cores)
    for n in (100_000, 1_000_000):
        x, y, z, rgb = O.synth_points(O.SYNTH_SLAB_ECEF, SLAB_SEED, 0, n, num_threads=cores)
        dx, dy, dz = [torch.from_numpy(a).cuda() for a in (x, y, z)]
        drgb = torch.from_numpy(rgb).cuda()
        host_ms, dev_ms = [], []
        nodes = 0
        for i in range(6):
            t0 = time.perf_counter()
            t = ctx.build_octree(x, y, z, rgb, res, bmin, bmax)
            host_ms.append((time.perf_counter() - t0) * 1e3)
            nodes = int(t.num_nodes)
            t.free()
            t0 = time.perf_counter()
            t = ctx.build_octree(dx.data_ptr(), dy.data_ptr(), dz.data_ptr(), drgb.data_ptr(), res, bmin, bmax, n=n, device=True)
            dev_ms.append((time.perf_counter() - t0) * 1e3)
            t.free()
        h, d = min(host_ms[1:]), min(dev_ms[1:])
        c = cpu[str(n)]
        out[str(n)] = {"gpu_host_api_ms": h, "gpu_device_resident_ms": d, "gpu_Mpoints_per_s_host_api": n / (h * 1e3), "gpu_Mpoints_per_s_device": n / (d * 1e3),
                       "octree_nodes": nodes, "cpu": c, "speedup_host_api_vs_cpu": min(c["in_memory_ms"], c["faithful_ms"]) / h}
    return out


def sharded_builder(D):
    """The multi-GPU build: one C call per rank (pcv_build_octree_sharded; torch.distributed only lends its collectives).
    PCV_PY_ORCH=1 runs the same steps orchestrated from Python instead (exchange of ingested records, no fused pass)."""
    return D.build_octree_sharded if os.environ.get("PCV_PY_ORCH") else D.build_octree_sharded_native


def multi_gpu_parity_check(ctx, pcv, D, torch, dist, world, rank, dev, n_global, res, bmin, bmax, k):
    """Inside the measured multi-GPU run: the sharded build of this run's N ranks == the single-GPU build == the oracle, bit for bit
    (node set, counts, encodings, cubes, per-slot global source index, colours, position codes), on n_global points of the
    benchmark generator (they include the identical-point blocks that reach level 20)."""
    import numpy as np

    kind = pcv.SYNTH_GAUSS_CLUSTERS
    n = n_global // world
    xs = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(3)]
    c = torch.empty(n * 3, dtype=torch.uint8, device=dev)
    ctx.synth_points_device(kind, SEED, rank * n, n, xs[0].data_ptr(), xs[1].data_ptr(), xs[2].data_ptr(), c.data_ptr())
    comm = D.TorchComm(dev)
    tree = sharded_builder(D)(ctx, xs[0], xs[1], xs[2], c, None, rank * n, res, bmin, bmax, prefix_levels=k)
    merged = tree.gather_all(comm)  # collective; rank 0 receives every final node
    kk = tree.k
    tree.free()
    verdict = {}
    if rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_api as O

        N = n * world
        X, Y, Z, RGB = O.synth_points(O.SYNTH_GAUSS_CLUSTERS, SEED, 0, N)
        single = ctx.build_octree(X, Y, Z, RGB, res, bmin, bmax)
        ref = O.build(X, Y, Z, RGB.reshape(-1, 3), res, bmin, bmax)
        try:
            from parity import compare_trees

            compare_trees(ref, single)  # single GPU == oracle
            assert set(single.nodes) == set(merged), "node sets differ: %s" % sorted(set(single.nodes) ^ set(merged))[:6]
            for name, m in single.nodes.items():  # sharded == single GPU
                g = merged[name]
                assert (g["num_points"], g["enc"], tuple(g["cube"])) == (m["num_points"], m["enc"], tuple(m["cube"])), name
                if m["num_points"]:
                    sx, sc, si, ss = single.node_data(name)
                    assert np.array_equal(ss, g["src"]), (name, "src index order")
                    assert np.array_equal(sx, g["xyz"]) and np.array_equal(sc, g["rgb"]), (name, "codes / colours")
            verdict = {"n": N, "ranks": world, "prefix_levels": kk, "equal": True, "nodes": len(merged), "deepest_level": max(len(nm) - 1 for nm in merged),
                       "what": "sharded build over this run's ranks == single-GPU build == oracle: node set, counts, encodings, cubes, per-slot global source index, colours, position codes"}
        except AssertionError as e:
            verdict = {"n": N, "ranks": world, "equal": False, "error": str(e)[:300]}
        single.free()
    dist.barrier()
    return verdict


def _final_node_bytes(pcv, tree):
    """Sum over the final nodes this rank holds of n (3 bpc + 3): local nodes at level >= k, plus the assembled top on rank 0."""

    def part(octree, min_level):
        return sum(int(m["num_points"]) * (3 * pcv.ENC_BYTES[int(m["enc"])] + 3) for name, m in octree.nodes.items() if len(name) - 1 >= min_level)

    total = part(tree.local, tree.k)
    if getattr(tree, "top", None) is not None:
        total += part(tree.top, 0)
    return total


def full_size_check(tree, D, torch, dist, world, n, dev):
    """Size-independent invariants of the full-size sharded result, all-reduced over the ranks: every input point appears
    exactly once in the final nodes (count, sum and sum of squares of the global source indices, mod 2^64)."""
    import ctypes as C
    import numpy as np

    import point_cloud_viewer_b200 as pcv
    from point_cloud_viewer_b200 import _native as N

    comm = D.TorchComm(dev)
    r_idx = tree.resolve_provenance(comm).to(torch.int64)  # collective

    def sums(octree, index, min_level):
        meta = octree.meta
        if octree.num_points == 0 or len(meta) == 0:
            return 0, 0, 0
        p = [C.c_void_p() for _ in range(4)]
        N.check(N.lib().pcv_octree_device_arrays(octree.h, *[C.byref(v) for v in p]))
        src = torch.as_tensor(D._RawCuda(p[3].value, (octree.num_points,), "<i4"), device=dev).to(torch.int64)
        order = np.argsort(meta["point_offset"], kind="stable")
        lev = torch.from_numpy(meta["level"][order].astype(np.int64)).to(dev)
        cnt = torch.from_numpy(meta["num_points"][order].astype(np.int64)).to(dev)
        keep = torch.repeat_interleave(lev >= min_level, cnt)
        g = index[src[keep]]
        return int(keep.sum()), int(g.sum()), int((g * g).sum())  # int64 wrap-around arithmetic

    c0, s0, q0 = sums(tree.local, r_idx, tree.k)
    if tree.top is not None:
        ti = torch.from_numpy(np.asarray(tree.top_index, np.uint64).astype(np.int64)).to(dev)
        c1, s1, q1 = sums(tree.top, ti, 0)
        c0, s0, q0 = c0 + c1, s0 + s1, q0 + q1
    wrap = lambda v: ((v + 2 ** 63) % 2 ** 64) - 2 ** 63
    t = torch.tensor([c0, wrap(s0), wrap(q0)], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    NT = world * n
    want = [NT, wrap(NT * (NT - 1) // 2), wrap((NT - 1) * NT * (2 * NT - 1) // 6)]
    got = [int(v) for v in t]
    return {"ok": got == want, "points": got[0], "expected_points": NT, "sum_idx_ok": got[1] == want[1], "sum_idx_sq_ok": got[2] == want[2]}


DUMP_BYTES = 64_000_000
DUMP_SEED = 20240917


def dump_outputs(tree, directory):
    """What the timed build hands its caller, for output-for-output comparison of two builds on the same seeded input:
    the whole node table (nodes.npy, one row per node in (id_high, id_low) order: level, the two 64-bit id words as 32-bit
    halves, num_points, position encoding, cube min xyz, edge) and, for a seeded sample of whole nodes that fits the 64 MB
    budget, every point of those nodes in slot order (sample_*.npy: node row, position code as stored, colour, source index)."""
    import numpy as np

    m = tree.meta
    rows = np.lexsort((m["id_low"], m["id_high"]))
    half = lambda v: [(v >> np.uint64(32)).astype(np.float64), (v & np.uint64(0xFFFFFFFF)).astype(np.float64)]
    nodes = np.stack([m["level"][rows].astype(np.float64)] + half(m["id_high"][rows]) + half(m["id_low"][rows])
                     + [m["num_points"][rows].astype(np.float64), m["enc"][rows].astype(np.float64)]
                     + [m["cube"][rows, k] for k in range(4)], 1)
    per_point = 8 + 3 * 8 + 3 * 4 + 8
    budget = (DUMP_BYTES - nodes.nbytes) // per_point
    picked, total = [], 0
    for r in np.random.default_rng(DUMP_SEED).permutation(len(rows)):
        k = int(m["num_points"][rows[r]])
        if k and total + k <= budget:
            picked.append(int(r))
            total += k
    node_of, code, rgb, src = [], [], [], []
    for r in sorted(picked):
        xyz, c, _, s = tree.node_data_at(int(rows[r]))
        dt = {1: "<u1", 2: "<u2", 3: "<f4", 4: "<f8"}[int(m["enc"][rows[r]])]
        code.append(np.frombuffer(xyz.tobytes(), dt).reshape(-1, 3).astype(np.float64))
        rgb.append(c.reshape(-1, 3).astype(np.float32))
        src.append(s.astype(np.float64))
        node_of.append(np.full(len(s), r, np.float64))
    out = {"nodes": nodes, "sample_node": np.concatenate(node_of or [np.zeros(0)]), "sample_position_code": np.concatenate(code or [np.zeros((0, 3))]),
           "sample_rgb": np.concatenate(rgb or [np.zeros((0, 3), np.float32)]), "sample_source_index": np.concatenate(src or [np.zeros(0)])}
    assert sum(a.nbytes for a in out.values()) <= DUMP_BYTES
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import point_cloud_viewer_b200 as pcv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = int(args.points)
    kind = pcv.SYNTH_GAUSS_CLUSTERS
    bmin, bmax, res = pcv.synth_bbox(kind)
    ctx = pcv.Context(local)

    def make_input(count, first):
        xs = [torch.empty(count, dtype=torch.float64, device=dev) for _ in range(3)]
        c = torch.empty(count * 3, dtype=torch.uint8, device=dev)
        ctx.synth_points_device(kind, SEED, first, count, xs[0].data_ptr(), xs[1].data_ptr(), xs[2].data_ptr(), c.data_ptr())
        return xs[0], xs[1], xs[2], c

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    out_extra = {}
    if world > 1:
        from point_cloud_viewer_b200 import distributed as D

        # ---- multi-GPU parity, inside the measured run (VERDICT r1): sharded vs single-GPU vs oracle on a small global sample ----
        try:
            out_extra["parity_check"] = multi_gpu_parity_check(ctx, pcv, D, torch, dist, world, rank, dev, int(args.parity_points), res, bmin, bmax, args.prefix_levels)
        except Exception as e:
            out_extra["parity_check"] = {"equal": False, "error": str(e)[:300]}

    x, y, z, rgb = make_input(n, rank * n + int(float(os.environ.get("PCV_FIRST_INDEX", "0"))))  # (diagnostic: another slice of the generator)

    if world > 1:

        def step():
            return sharded_builder(D)(ctx, x, y, z, rgb, None, rank * n, res, bmin, bmax, prefix_levels=args.prefix_levels)
    else:

        def step():
            return ctx.build_octree(x.data_ptr(), y.data_ptr(), z.data_ptr(), rgb.data_ptr(), res, bmin, bmax, n=n, device=True)

    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("PCV_NO_SAMPLER"):  # (diagnostic switch: the clocks line is part of the contract)
        sampler.start()  # before the warm-up: see ClockSampler.window
    for w in range(args.warmup):
        t = step()
        t.free()
    launches0 = ctx.kernel_launch_count()
    barrier()
    t_region0 = time.time()
    dev_ms = 0.0
    wall_ms = 0.0
    lib_ms = 0.0
    last = None
    for _ in range(args.steps):
        if last is not None:
            last.free()
        barrier()
        # The library works on its own stream and every step ends in a host-visible synchronisation, so an event pair on the
        # current stream brackets exactly the device timeline of the step, host planning gaps included (same clock at every N).
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        w0 = time.perf_counter()
        last = step()
        torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        wall_ms += (time.perf_counter() - w0) * 1e3
        dev_ms += e0.elapsed_time(e1)
        if world == 1:
            lib_ms += ctx.last_build_stats()["ms_total"]
        barrier()
    if os.environ.get("PCV_RANK_KSTATS"):  # diagnostic: per-rank kernel times of one extra step
        ctx.set_profiling(True)
        t = step()
        t.free()
        ks = ctx.kernel_stats()
        ctx.set_profiling(False)
        print("[kstats r%d] " % rank + "  ".join("%s %.2f" % (k, v["ms"]) for k, v in ks.items() if v["ms"] > 0), file=sys.stderr, flush=True)
    sampler.window(t_region0, time.time())
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.kernel_launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(last, args.dump_outputs)
    tm = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    dev_ms, wall_ms = float(tm[0]), float(tm[1])
    ms_per_step = dev_ms / args.steps
    value = world * n / (ms_per_step * 1e3)
    stats = ctx.last_build_stats() if world == 1 else last.stats
    nodes = int(last.num_nodes)

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(n, world, args),
        "wall_ms_per_step": wall_ms / args.steps, "gpu_launches": int(launches), "octree_nodes": nodes, "deepest_level": int(stats.get("deepest_level", 0)),
        "clocks": clocks,
    }
    out.update(out_extra)
    if world == 1:
        out["library_event_ms_per_step"] = lib_ms / args.steps
    if world > 1:
        # full-size invariants of the sharded result, all-reduced: every point exactly once (count, sum and sum of squares of the
        # global source indices), and the per-phase breakdown of the last step
        try:
            ctx.release_cached_memory()  # the library's recycled work buffers: the check below needs tens of GB for its own tensors
            out["full_size_check"] = full_size_check(last, D, torch, dist, world, n, dev)
        except Exception as e:
            out["full_size_check"] = {"ok": False, "error": str(e)[:300]}
        out["phases_ms"] = getattr(last, "phases_ms", None)
        # whole-build HBM roofline of the sharded job (SURVEY 8d bytes: 27 per input point + every point once in its final
        # encoding), per GPU.  One unconditional all-reduce: a rank whose local sum fails contributes a flag instead of hanging.
        try:
            final_bytes = float(_final_node_bytes(pcv, last))
            bad = 0.0
        except Exception:
            final_bytes, bad = 0.0, 1.0
        tb = torch.tensor([final_bytes, bad], dtype=torch.float64, device=dev)
        dist.all_reduce(tb)
        if float(tb[1]) == 0.0:
            peak, peak_src = _peaks()
            algo = 27.0 * n * world + float(tb[0])
            per_gpu = algo / world / (ms_per_step * 1e-3) / 1e9
            out["roofline"] = {"bound": "hbm", "kernel": "whole sharded build (per GPU; every kernel + the exchange)", "achieved": per_gpu, "peak": peak, "unit": "GB/s",
                               "frac": per_gpu / peak, "traffic": None, "peak_source": peak_src,
                               "whole_build": {"algorithmic_bytes": int(algo), "achieved": per_gpu, "frac": per_gpu / peak},
                               "note": "per-kernel rooflines are reported by the N = 1 run (same kernels); the exchange phase moves 17 B per point over NVLink (phases_ms.exchange)"}

    if world == 1 and not args.no_extras:
        peak, peak_src = _peaks()
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_api as O

        cores = os.cpu_count() or 1
        # ---- roofline of the dominant kernel: one extra build with CUDA events around every launch ----
        ctx.set_profiling(True)
        t = step()
        t.free()
        ks = ctx.kernel_stats()
        ctx.set_profiling(False)
        top = max(ks.items(), key=lambda kv: kv[1]["ms"])
        tname, tst = top
        achieved = tst["algorithmic_bytes"] / (tst["ms"] * 1e-3) / 1e9 if tst["ms"] > 0 else 0.0
        traffic = None
        try:  # DRAM bytes per launch from the committed `ncu --set full` capture (ratio to algorithmic bytes at N = 1e8)
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f)[tname]["ratio"] * tst["algorithmic_bytes"] / max(1, tst["launches"])
        except Exception:
            pass
        out["roofline"] = {
            "bound": "hbm", "kernel": tname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "peak_source": peak_src, "launches": tst["launches"], "avg_launch_ms": tst["ms"] / max(1, tst["launches"]),
            "algorithmic_bytes_per_launch": tst["algorithmic_bytes"] / max(1, tst["launches"]),
            "note": "per-kernel bytes are the pass-local reads + writes (records 16 B + colour 4 B + digit 1 B per point and pass); whole_build uses the SURVEY 8(d) compulsory bytes: 27 N + sum over nodes of n (3 bpc + 3)",
            "whole_build": {"algorithmic_bytes": int(stats["algorithmic_bytes"]), "achieved": stats["algorithmic_bytes"] / (ms_per_step * 1e-3) / 1e9,
                            "frac": stats["algorithmic_bytes"] / (ms_per_step * 1e-3) / 1e9 / peak},
            "kernels": {k: {"launches": v["launches"], "ms": v["ms"], "GBps": (v["algorithmic_bytes"] / (v["ms"] * 1e-3) / 1e9 if v["ms"] > 0 else 0.0)} for k, v in ks.items()},
        }

        if args.roofline_only:
            print(json.dumps(out))
            return
        # ---- BASELINE config 3: frustum-culled point query over the resident octree ----
        try:
            out["frustum_query"] = bench_query(ctx, pcv, torch, O, last, args, bmin, bmax, peak, cores, res)
        except Exception as e:  # never lose the build line
            out["frustum_query"] = {"error": str(e)[:300]}
        # ---- BASELINE config 5: X-ray leaf tiles over the resident octree ----
        try:
            out["xray"] = bench_xray(ctx, pcv, torch, O, last, args, bmin, bmax, peak, cores, res)
        except Exception as e:
            out["xray"] = {"error": str(e)[:300]}

        # ---- e2e: the reference-facing call with HOST buffers (H2D + build + D2H inside the timed region) ----
        last.free()
        last = None
        ne = n
        try:
            hx, hy, hz = [torch.empty(ne, dtype=torch.float64, pin_memory=True) for _ in range(3)]
            hrgb = torch.empty(ne * 3, dtype=torch.uint8, pin_memory=True)
            hx.copy_(x[:ne])
            hy.copy_(y[:ne])
            hz.copy_(z[:ne])
            hrgb.copy_(rgb[: 3 * ne])
            del x, y, z, rgb
            torch.cuda.empty_cache()
            oxyz = torch.empty(int(ne * 12 + (1 << 24)), dtype=torch.uint8, pin_memory=True)
            orgb = torch.empty(ne * 3, dtype=torch.uint8, pin_memory=True)

            def e2e_step():
                t = ctx.build_octree(hx.data_ptr(), hy.data_ptr(), hz.data_ptr(), hrgb.data_ptr(), res, bmin, bmax, n=ne)
                assert t.xyz_bytes <= oxyz.numel()
                t.download(xyz=oxyz.data_ptr(), rgb=orgb.data_ptr(), want_src=False)  # what build_octree leaves on disk: .xyz + .rgb + meta
                b = (t.xyz_bytes + ne * 3 + 80 * t.num_nodes, t.num_nodes)
                t.free()
                return b

            e2e_step()  # two warm-up calls: the stream-ordered pool grows to hold the 27 GB staging copy
            e2e_step()
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            esteps = max(1, min(args.steps, 3))
            for _ in range(esteps):
                d2h, _ = e2e_step()
            torch.cuda.synchronize()
            ems = (time.perf_counter() - w0) * 1e3 / esteps
            out["e2e"] = {"value": ne / (ems * 1e3), "unit": UNIT, "h2d_bytes_per_step": int(27 * ne), "d2h_bytes_per_step": int(d2h), "ms_per_step": ems, "steps": esteps,
                          "note": "pcv_build_octree(host SoA, pinned) + pcv_octree_download(pinned): node table, .xyz codes and .rgb of every node"}
            del hx, hy, hz, hrgb, oxyz, orgb
        except Exception as e:
            out["e2e"] = {"value": None, "unit": UNIT, "h2d_bytes_per_step": None, "d2h_bytes_per_step": None, "error": str(e)[:200]}

        # ---- CPU baseline: the oracle port on this box's host cores, bounded sample; and the parity verdict on that sample ----
        try:
            nc = int(args.cpu_points)
            cx, cy, cz, crgb = O.synth_points(O.SYNTH_GAUSS_CLUSTERS, SEED, 0, nc, num_threads=cores)
            t0 = time.perf_counter()
            o = O.build(cx, cy, cz, crgb.reshape(-1, 3), res, bmin, bmax, num_threads=cores)
            ct = time.perf_counter() - t0
            d = _shm_dir()
            try:
                ft, _ = O.build_faithful(cx, cy, cz, crgb.reshape(-1, 3), res, bmin, bmax, d, num_threads=cores)
            finally:
                shutil.rmtree(d, ignore_errors=True)
            best = min(ct, ft)
            out["cpu_baseline"] = {"value": nc / best / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": "first %d points of the same generator, one build per variant (oracle port of build_octree, %d threads): in-memory %.2f s, faithful (/dev/shm node files) %.2f s; value = the faster" % (nc, cores, ct, ft)}
            try:
                from parity import compare_trees

                gt = ctx.build_octree(cx, cy, cz, crgb, res, bmin, bmax)
                compare_trees(o, gt)
                deep = max(len(nm) - 1 for nm in o.nodes)
                out["parity_check"] = {"n": nc, "equal": True, "nodes": len(o.nodes), "deepest_level": deep,
                                       "what": "GPU octree of the first n points of the benchmark generator == oracle: node set, counts, encodings, cubes, per-slot source index, colours, position codes"}
                gt.free()
            except AssertionError as e:
                out["parity_check"] = {"n": nc, "equal": False, "error": str(e)[:300]}
            del o
        except Exception as e:
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": "failed: " + str(e)[:160]}

        # ---- BASELINE config 1: the reference's own bench sizes on both sides ----
        try:
            out["config1"] = bench_config1(ctx, pcv, torch, O, cores)
        except Exception as e:
            out["config1"] = {"error": str(e)[:300]}

        # ---- PLY input path (SURVEY 8f rank 1): file -> pinned ring -> H2D -> k_ply_unpack (+ fused bounding box) ----
        try:
            out["ply_ingest"] = bench_ply(ctx, pcv, int(args.ply_points), peak)
        except Exception as e:
            out["ply_ingest"] = {"error": str(e)[:200]}

        # ---- SURVEY 8(f3, f4): the whole X-ray quadtree (leaves, background, Lanczos3 parents) and the S2-cell cloud split - in a child process, last ----
        try:
            ctx.release_cached_memory()
            torch.cuda.empty_cache()
            r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "xray_pyramid_bench.py"), "--points", str(int(args.cpu_points)), "--tile-px", str(int(args.xray_px)),
                                "--peak", str(peak)], capture_output=True, text=True, timeout=420)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")]
            extra = json.loads(line[-1]) if line else {"xray_quadtree": {"error": ("rc %d: " % r.returncode) + (r.stderr or r.stdout)[-300:]}}
            out["xray_quadtree"] = extra.get("xray_quadtree")
            out["s2_cloud"] = extra.get("s2_cloud")
        except Exception as e:
            out["xray_quadtree"] = {"error": str(e)[:300]}
    else:
        out["e2e"] = {"value": None, "unit": UNIT, "h2d_bytes_per_step": None, "d2h_bytes_per_step": None, "note": "e2e is measured at N=1 (without --no-extras)"}
        if last is not None:
            last.free()

    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def bench_query(ctx, pcv, torch, O, tree, args, bmin, bmax, peak, cores, res):
    """Config 3: 1000 random frusta (two far planes) over the resident 1e9-point octree.  Device time from the library's CUDA
    events; bytes = B_query of SURVEY 8(d) (decode read of every tested point + 27 B per survivor).  CPU baseline: the oracle's
    ParallelIterator port (cores - 1 threads, point_cloud_client/src/lib.rs:67) over an octree of the first --cpu-points points."""
    G = pcv.geometry
    fq = {}
    sets = (("far10", 10.0, args.frusta), ("far0.1E", 102.4, args.frusta))
    for label, far, count in sets:
        locs = make_frusta(G, bmin, bmax, count, far)
        tree.query_batch_device(locs[:8])  # warm-up (tables, pool)
        torch.cuda.synchronize()
        best = None
        for _ in range(3):
            q0 = time.perf_counter()
            counts, tested = tree.query_batch_device(locs)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - q0) * 1e3
            qs = tree.last_query_stats()
            if best is None or qs["ms_device"] < best[0]["ms_device"]:
                best = (qs, wall, counts, tested)
        qs, wall, counts, tested = best
        gbps = qs["algorithmic_bytes"] / (qs["ms_device"] * 1e-3) / 1e9 if qs["ms_device"] > 0 else 0.0
        fq[label] = {"frusta": len(locs), "tested_points": int(tested.sum()), "returned_points": int(counts.sum()), "ms_device": qs["ms_device"], "ms_wall": wall,
                     "Mpoints_per_s_tested": float(tested.sum()) / (qs["ms_device"] * 1e3), "gpu_launches": int(qs["kernel_launches"]),
                     "roofline": {"bound": "hbm", "kernel": "k_cull", "achieved": gbps, "peak": peak, "unit": "GB/s", "frac": gbps / peak,
                                  "algorithmic_bytes": int(qs["algorithmic_bytes"]), "cull_kernel_ms": qs["ms_cull"]}}
    # CPU baseline on a sample octree (the oracle cannot hold 1e9 points in this run's time budget)
    nc = int(args.cpu_points)
    cx, cy, cz, crgb = O.synth_points(O.SYNTH_GAUSS_CLUSTERS, SEED, 0, nc, num_threads=cores)
    o = O.build(cx, cy, cz, crgb.reshape(-1, 3), res, bmin, bmax, num_threads=cores)
    gt = ctx.build_octree(cx, cy, cz, crgb, res, bmin, bmax)
    for label, far, count in sets:
        locs = make_frusta(G, bmin, bmax, min(count, 200), far)
        r = o.query_batch_timed(locs, max(1, cores - 1))
        gc, gtst = gt.query_batch_device(locs)
        qs = gt.last_query_stats()
        fq[label]["cpu_baseline"] = {"value": r["tested"] / r["seconds"] / 1e6 if r["seconds"] > 0 else None, "unit": "Mpoints/s tested", "cores": max(1, cores - 1), "kind": "port",
                                     "sample": "%d frusta over the octree of the first %d points (oracle ParallelIterator port)" % (len(locs), nc),
                                     "tested_points": r["tested"], "returned_points": r["returned"], "seconds": r["seconds"],
                                     "gpu_same_sample": {"tested_points": int(gtst.sum()), "returned_points": int(gc.sum()), "ms_device": qs["ms_device"],
                                                         "equal_counts": bool(int(gtst.sum()) == r["tested"] and int(gc.sum()) == r["returned"])}}
    gt.free()
    return fq


def bench_xray(ctx, pcv, torch, O, tree, args, bmin, bmax, peak, cores, res):
    """Config 5: the 16 leaf tiles (4 x 4 tiles of 256 m, 4096 x 4096 px of 0.0625 m) of the X-ray quadtree over the resident
    octree (xray/src/generation.rs:515-548,618-654), XRay colouring; bytes = B_xray of SURVEY 8(d)."""
    tile_px = int(args.xray_px)
    e = float(bmax[0] - bmin[0])
    nt = 4
    ts = e / nt
    ms, pts, byts, nonempty = 0.0, 0, 0, 0
    for iy in range(nt):
        for ix in range(nt):
            tmin = (bmin[0] + ix * ts, bmin[1] + iy * ts, bmin[2])
            tmax = (bmin[0] + (ix + 1) * ts, bmin[1] + (iy + 1) * ts, bmax[2])
            anyp, _rgba, _ = tree.xray_tile(tmin, tmax, tile_px, tile_px, None, want_bits=False)
            xs = tree.last_xray_stats()
            ms += xs["ms_device"]
            pts += xs["points"]
            byts += xs["algorithmic_bytes"]
            nonempty += 1 if anyp else 0
    gbps = byts / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
    out = {"tiles": nt * nt, "tile_px": tile_px, "non_empty_tiles": nonempty, "points": int(pts), "ms_device": ms, "Mpoints_per_s": pts / (ms * 1e3) if ms > 0 else None,
           "roofline": {"bound": "hbm", "kernel": "k_xray_*", "achieved": gbps, "peak": peak, "unit": "GB/s", "frac": gbps / peak, "algorithmic_bytes": int(byts)}}
    # CPU baseline: the oracle's xray_from_points on a sample octree, one tile per core like the reference's rayon tile loop
    nc = int(args.cpu_points)
    cx, cy, cz, crgb = O.synth_points(O.SYNTH_GAUSS_CLUSTERS, SEED, 0, nc, num_threads=cores)
    o = O.build(cx, cy, cz, crgb.reshape(-1, 3), res, bmin, bmax, num_threads=cores)
    px = min(tile_px, 1024)
    t0 = time.perf_counter()
    tmin, tmax = (bmin[0], bmin[1], bmin[2]), (bmin[0] + ts, bmin[1] + ts, bmax[2])
    o.xray_tile(tmin, tmax, px, px)
    ct = time.perf_counter() - t0
    loc = pcv.geometry.aabb(tmin, tmax)
    ol = O.Location()
    for f, _ in O.Location._fields_:
        setattr(ol, f, getattr(loc, f))
    npts = len(o.query(ol)["src"])
    out["cpu_baseline"] = {"value": npts / ct / 1e6 if ct > 0 else None, "unit": "Mpoints/s", "cores": 1, "kind": "port",
                           "sample": "one %d x %d leaf tile over the octree of the first %d points (%d points in the tile, %.2f s; the reference runs one tile per core)" % (px, px, nc, npts, ct)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--points", type=float, default=1e9, help="points per GPU per step (the same at every N)")
    ap.add_argument("--levels-per-pass", type=int, default=2, help="(accepted for compatibility: the split phase resolves two levels per pass)")
    ap.add_argument("--prefix-levels", type=int, default=2)
    ap.add_argument("--frusta", type=int, default=1000)
    ap.add_argument("--xray-px", type=int, default=4096)
    ap.add_argument("--cpu-points", type=float, default=2e7)
    ap.add_argument("--parity-points", type=float, default=1.6e7, help="global sample of the N > 1 parity check (sharded vs single GPU vs oracle)")
    ap.add_argument("--ply-points", type=float, default=1e8, help="points of the synthetic PLY file for the ingest measurement")
    ap.add_argument("--ref-points", type=float, default=1e8, help="points of the bounded sample each --impl reference step builds")
    ap.add_argument("--no-extras", action="store_true", help="profiling runs: only the timed build steps (no roofline / query / e2e / CPU legs)")
    ap.add_argument("--roofline-only", action="store_true", help="development runs: timed steps + per-kernel roofline, none of the other legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's octree (node table + a seeded sample of its points) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the single-GPU build (--impl ours, one process)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
