"""The C-ABI library loads and exports every symbol include/pcv.h declares; no compute without a GPU."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_exports_every_declared_symbol():
    from point_cloud_viewer_b200 import _native

    L = _native.lib()
    header = open(os.path.join(ROOT, "include", "pcv.h")).read()
    declared = set(re.findall(r"\b(pcv_[a-z0-9_]+)\s*\(", header)) - {"pcv_batch_cb"}
    bound = {name for name, _, _ in _native.SYMBOLS}
    assert declared == bound, (declared ^ bound)
    for name in declared:
        assert getattr(L, name) is not None


def test_struct_layouts_match_header():
    from point_cloud_viewer_b200 import _native as N

    assert C.sizeof(N.NodeMeta) == 80 and C.sizeof(N.Points) == 56 and C.sizeof(N.Location) == 8 + 8 * (6 + 32 + 14 + 3)
    assert C.sizeof(N.Config) == 16 and C.sizeof(N.Interval) == 16 and C.sizeof(N.Batch) == 40
    assert C.sizeof(N.PlyInfo) == 96 and N.PlyInfo.offset.offset == 72 and N.PlyInfo.off_intensity.offset == 64


def test_xray_quadtree_structs_match_the_c_compiler(tmp_path):
    """pcv_xray_quadtree_params / _info and pcv_query_out: ctypes sizes and field offsets equal gcc's for include/pcv.h."""
    import subprocess

    from point_cloud_viewer_b200 import _native as N

    structs = (("pcv_xray_quadtree_params", N.XrayQuadtreeParams), ("pcv_xray_quadtree_info", N.XrayQuadtreeInfo), ("pcv_query_out", N.QueryOut))
    fields = {st: [f for f, _ in cls._fields_] for st, cls in structs}
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "pcv.h"', "int main(void) {"]
    for st, fs in fields.items():
        src.append('printf("%s %%zu" "\\n", sizeof(%s));' % (st, st))
        for f in fs:
            src.append('printf("%s.%s %%zu" "\\n", offsetof(%s, %s));' % (st, f, st, f))
    src.append("return 0; }")
    c = tmp_path / "layout.c"
    c.write_text(chr(10).join(src))
    exe = str(tmp_path / "layout")
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, str(c)])
    got = dict(l.split() for l in subprocess.check_output([exe], text=True).splitlines())
    for st, cls in structs:
        assert int(got[st]) == C.sizeof(cls)
        for f, _ in cls._fields_:
            assert int(got["%s.%s" % (st, f)]) == getattr(cls, f).offset, (st, f)


def test_no_cpu_fallback():
    """Without a CUDA device the library refuses to create a context (there is no CPU path to fall back to)."""
    from point_cloud_viewer_b200 import _native as N
    import point_cloud_viewer_b200 as pcv

    if pcv.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(N.PcvError) as e:
        pcv.Context(0)
    assert e.value.code == -2


def test_product_sources_do_not_reference_the_oracle():
    """oracle/ is test infrastructure: nothing in the package or in include/ may include, import or link it."""
    pkg = os.path.join(ROOT, "point_cloud_viewer_b200")
    for base in (pkg, os.path.join(ROOT, "include")):
        for r, _, fs in os.walk(base):
            for f in fs:
                if f.endswith((".so", ".pyc")):
                    continue
                s = open(os.path.join(r, f), errors="ignore").read()
                assert not re.search(r'#include\s+"[^"]*oracle|import\s+oracle|liboracle|oracle_api', s), os.path.join(r, f)


def test_synth_generators_host():
    import numpy as np
    import point_cloud_viewer_b200 as pcv

    x, y, z, rgb = pcv.synth_points_host(pcv.SYNTH_SLAB_ECEF, 80293751232, 0, 50000)
    mn, mx, res = pcv.synth_bbox(pcv.SYNTH_SLAB_ECEF)
    P = np.stack([x, y, z], 1)
    assert res == 0.001 and (P >= mn).all() and (P <= mx).all()
    assert 240 < (mx - mn).max() < 245  # root edge of the rotated 200 x 200 x 20 slab
    assert np.array_equal(rgb.reshape(-1, 3)[:, 2], (np.arange(50000) & 255).astype(np.uint8))  # index encoded in colour
    x, y, z, rgb = pcv.synth_points_host(pcv.SYNTH_GAUSS_CLUSTERS, 1, (1 << 20) - 10, 150020)
    mn, mx, res = pcv.synth_bbox(pcv.SYNTH_GAUSS_CLUSTERS)
    P = np.stack([x, y, z], 1)
    assert res == 1024.0 / 2 ** 20 and (P >= mn).all() and (P <= mx).all()
    assert (P[10:150010] == P[10]).all() and not (P[:10] == P[10]).all()  # one block of 150 000 identical points


def test_cpp_mirror_compiles_against_the_library():
    """include/pcv.hpp (header-only C++ mirror of the crate's names) and its test program build and link against the
    library; running them needs a GPU (tests/test_cpp_host_gpu.py)."""
    import subprocess
    import tempfile

    from point_cloud_viewer_b200 import _native

    lib_dir = os.path.dirname(_native.LIB_PATH)
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "test_octree")
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", os.path.join(ROOT, "tests", "cpp", "test_octree.cpp"), "-o", exe, "-L" + lib_dir,
                               "-l:libpcv_b200.so", "-Wl,-rpath," + lib_dir])
        assert os.path.exists(exe)
