"""The reference's own integration tests for its two point clouds (point_cloud_test/tests/main.rs:10-58, 87-204) restated over the
GPU octree and the GPU S2-cell cloud: the same 1e6 synthetic ECEF points (SyntheticData of Arguments::default, restated in
reference_synthetic.py; index encoded in the colour), split level 20, resolution 0.001; AllPoints and the cell-union query
(queries.rs:49-53) must return the same indexed points up to the reference's own tolerance (distance <= 2 sqrt(3) resolution,
at most 1 % of the points on one side only).  The octree side of the cell-union query filters every octree point with the
CellUnion's PointCulling (the reference additionally pre-selects nodes through the s2 crate's latitude / longitude rectangles,
which is not built here and does not change which points pass the point test).
The tolerance depends on the data's bounding cube, not only on the resolution: every split and subsample pass decodes a node's
positions and re-encodes them truncated in the next node, so the error grows with the step of the coarsest fixed-point node a
point passes through.  The reference's slab frame (lat -84.4, lon -44.9) has a 283.5 m root cube, Float32 down to level 2 and a
largest drift of 1.87 mm; the product's own slab generator (PCV_SYNTH_SLAB_ECEF) has a 243.2 m root cube, Uint16 at level 2
with a 0.93 mm step and drifts by up to 4.78 mm, which the reference's 3.46 mm bound was never meant to cover.
(Sorts last: added after the round's last GPU session.)"""
import numpy as np
import pytest

import s2_api as S
from reference_synthetic import synthetic_data

pytestmark = pytest.mark.gpu


def _indexed(xyz, rgb):
    idx = (rgb[:, 0].astype(np.int64) << 16) + (rgb[:, 1].astype(np.int64) << 8) + rgb[:, 2].astype(np.int64)  # main.rs:139-140
    o = np.argsort(idx, kind="stable")
    return idx[o], xyz[o]


def _assert_points_equal(a, b, resolution):  # main.rs:160-204
    ia, pa = a
    ib, pb = b
    assert len(ia) and len(ib), "The query returned no points (using streaming)"
    common, ka, kb = np.intersect1d(ia, ib, return_indices=True)
    skipped = (len(ia) - len(common)) + (len(ib) - len(common))
    assert skipped <= -(-min(len(ia), len(ib)) // 100), (skipped, len(ia), len(ib))
    dist = np.linalg.norm(pa[ka] - pb[kb], axis=1)
    assert dist.max() <= np.sqrt(3.0) * 2.0 * resolution, dist.max()


def test_s2_and_octree_queries_agree(ctx):
    import point_cloud_viewer_b200 as pcv

    n = 1_000_000
    data = synthetic_data(n)
    x, y, z = (np.ascontiguousarray(data["xyz"][:, k]) for k in range(3))
    rgb = np.ascontiguousarray(data["rgb"].reshape(-1))
    bmin, bmax, res = data["bbox_min"], data["bbox_max"], 0.001
    tree = ctx.build_octree(x, y, z, rgb, res, bmin, bmax)
    cloud = ctx.build_s2_cloud(x, y, z, rgb, None, split_level=20)  # S2_LEVEL, point_cloud_test/src/lib.rs:21
    # num_points_in_octree_meta / num_points_in_s2_meta
    assert sum(m["num_points"] for m in tree.nodes.values()) == n and int(cloud.cell_counts.sum()) == n
    # check_all_query_equality
    oct_b = tree.query_points(pcv.geometry.all_points(), batch_size=5000 * 40)
    oct_xyz = np.concatenate([b["xyz"] for b in oct_b])
    oct_rgb = np.concatenate([b["rgb"] for b in oct_b])
    s2_all = cloud.query_union(None)
    _assert_points_equal(_indexed(s2_all["xyz"], s2_all["rgb"]), _indexed(oct_xyz, oct_rgb), res)
    assert len(s2_all["xyz"]) == len(oct_xyz) == n
    # check_cell_union_query_equality: the cell of the slab's origin at level 20 and its successor
    centre = data["origin"][None, :]  # ecef_from_local.translation
    cell = int(S.oracle_cell_ids(centre, 20)[0])
    u = np.array([cell, S.orc().orc_s2_next(cell)], np.uint64)
    s2_q = cloud.query_union(u)
    keep = ctx.s2_union_contains(np.ascontiguousarray(oct_xyz[:, 0]), np.ascontiguousarray(oct_xyz[:, 1]), np.ascontiguousarray(oct_xyz[:, 2]), u)
    assert 0 < keep.sum() < n and 0 < s2_q["total"] < n
    _assert_points_equal(_indexed(s2_q["xyz"], s2_q["rgb"]), _indexed(oct_xyz[keep], oct_rgb[keep]), res)
    cloud.free()
    tree.free()
