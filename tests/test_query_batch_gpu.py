"""The survivors of the batched device query (pcv_query_batch_device, k_cull_fused) against the oracle, point by point.

Two octrees of one mixed cloud cover every position encoding: fixture A (resolution 1 mm, 300 points per node) holds
Uint8 and Uint16 nodes, fixture B (resolution 2e-7, 500 points per node) Float32 and Float64 nodes as well.  Every
location's survivors, sorted by source index, must equal the oracle's query: source index, the decoded f64 position
bit for bit, colour and intensity.  Also checked: the interval filters, an output capacity that cuts a round of
survivors, points exactly on the faces of an Aabb and inside the one-ulp band of the frustum test where loc_contains
falls back to the divisions (through the streaming query too), a shuffled octree and one loaded from disk."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_api as O
from parity import compare_trees

pytestmark = pytest.mark.gpu

N_POINTS = 200_000
FIXTURES = {"A": (1e-3, 300), "B": (2e-7, 500)}  # resolution, max points per node
ENC_NAMES = {1: "Uint8", 2: "Uint16", 3: "Float32", 4: "Float64"}


def _mixed(rng, n):  # wide clusters -> U16/F32 nodes, 2 cm clusters -> U8 nodes with distinct points, one identical block
    cen = rng.random((20, 3)) * [200, 200, 20]
    k = rng.integers(0, 20, n)
    sig = np.where(k < 10, 3.0 * rng.random(20)[k], 0.02)
    P = cen[k] + rng.normal(0, 1, (n, 3)) * sig[:, None]
    P[: n // 20] = P[0]
    return P + (4.1e6, 6.6e5, 4.7e6)


def _cloud():
    rng = np.random.default_rng(5)
    P = _mixed(rng, N_POINTS)
    rgb = rng.integers(0, 256, (N_POINTS, 3), dtype=np.uint8)
    inten = (rng.random(N_POINTS) * 1000.0).astype(np.float32)
    x, y, z = (np.ascontiguousarray(P[:, a]) for a in range(3))
    b = O.bbox(x, y, z)
    return x, y, z, rgb, inten, np.array(b[:3]), np.array(b[3:])


def _oracle_tree(cloud, name):
    x, y, z, rgb, inten, bmin, bmax = cloud
    res, mppn = FIXTURES[name]
    return O.build(x, y, z, rgb, res, bmin, bmax, intensity=inten, max_points_per_node=mppn)


def _copy_loc(loc):
    o = O.Location()
    for f, _ in O.Location._fields_:
        setattr(o, f, getattr(loc, f))
    return o


def _locations(G, cloud):
    """47 locations: the query shapes of test_query_gpu._locations around the cloud's centre, seeded random frusta (near
    0.1, far 10 and 300), OBBs and AABBs around points of the cloud, one location outside the bounding box and one that
    appears twice."""
    x, y, z, _, _, bmin, bmax = cloud
    d = bmax - bmin
    q = G.quat_mul(G.quat_from_axis_angle([0, 0, 1], 0.7), G.quat_from_axis_angle([0, 1, 0], -0.9))
    frame = G.Isometry((bmin + bmax) * 0.5, q)
    locs = [
        G.all_points(),
        G.aabb(bmin + 0.2 * d, bmin + 0.8 * d),
        G.aabb(bmin + 0.45 * d, bmin + 0.5 * d),
        G.obb(frame, (50.0, 50.0, 5.0)),
        G.frustum(frame, G.Perspective.new_fov(1.0, 1.2, 0.1, 10.0)),
        G.frustum(frame * G.Isometry((0, 0, 0), G.quat_from_axis_angle([1, 0.3, 0], 1.3)), G.Perspective.new_fov(1.3, 0.9, 0.5, 150.0)),
        G.obb(frame * G.Isometry((10, -20, 1), G.quat_from_axis_angle([0.2, 0.5, -0.7], 0.523)), (30.0, 12.0, 4.0)),
    ]
    rng = np.random.default_rng(17)

    def near_point():
        i = rng.integers(0, len(x))
        return np.array([x[i], y[i], z[i]])

    def rotation():
        r = rng.normal(size=4)
        return r / np.linalg.norm(r)

    for i in range(14):  # the camera (looking down its -z) has a point of the cloud on its axis
        far = 10.0 if i % 2 else 300.0
        q = rotation()
        eye = near_point() - G.quat_rotate(q, (0.0, 0.0, -far * (0.1 + 0.5 * rng.random())))
        locs.append(G.frustum(G.Isometry(eye, q), G.Perspective.new_fov(0.7 + rng.random(), 0.6 + rng.random(), 0.1, far)))
    for _ in range(12):
        locs.append(G.obb(G.Isometry(near_point(), rotation()), 0.5 + rng.random(3) * 30.0))
    for _ in range(12):
        c, h = near_point(), 0.3 + rng.random(3) * 40.0
        locs.append(G.aabb(c - h, c + h))
    locs.append(G.aabb(bmax + 10.0, bmax + 20.0))  # outside the bounding box
    locs.append(locs[9])  # the same frustum twice
    return locs


OUTSIDE, DUPLICATE, DUPLICATED = 45, 46, 9


def _records(xyz, rgb, inten, src):
    """Survivor records as one structured array (xyz compared as bit patterns)."""
    r = np.zeros(len(src), [("src", "<u8"), ("x", "<u8"), ("y", "<u8"), ("z", "<u8"), ("r", "u1"), ("g", "u1"), ("b", "u1"), ("i", "<u4")])
    r["src"] = src
    bits = np.ascontiguousarray(xyz, np.float64).reshape(-1, 3).view(np.uint64)
    r["x"], r["y"], r["z"] = bits[:, 0], bits[:, 1], bits[:, 2]
    rgb = np.asarray(rgb).reshape(-1, 3)
    r["r"], r["g"], r["b"] = rgb[:, 0], rgb[:, 1], rgb[:, 2]
    r["i"] = np.ascontiguousarray(inten, np.float32).view(np.uint32)
    return r


def _by_src(r):
    return r[np.argsort(r["src"], kind="stable")]


def _by_value(r):
    """Sorted on everything but the source index (an octree loaded from disk has none)."""
    return np.sort(r, order=["x", "y", "z", "r", "g", "b", "i"])


def _oracle_sets(ref, locs, filters=()):
    out = []
    for loc in locs:
        w = ref.query(_copy_loc(loc), filters=filters, with_intensity=True)
        out.append((_records(w["xyz"], w["rgb"], w["intensity"], w["src"]), w["tested"]))
    return out


def _split(got, nloc):
    """The batched output grouped by location: list of record arrays."""
    rec = _records(got["xyz"], got["rgb"], got["intensity"], got["src"].astype(np.uint64))
    loc = got["loc"].astype(np.int64)
    assert (loc < nloc).all()
    order = np.argsort(loc, kind="stable")
    bounds = np.searchsorted(loc[order], np.arange(nloc + 1))
    return [rec[order[bounds[i]:bounds[i + 1]]] for i in range(nloc)]


def _check_against_oracle(counts, tested, got, want, key=_by_src, what=""):
    nloc = len(want)
    parts = _split(got, nloc)
    for i, (part, (w, wt)) in enumerate(zip(parts, want)):
        assert int(counts[i]) == len(w), (what, i, int(counts[i]), len(w))
        assert int(tested[i]) == wt, (what, i, int(tested[i]), wt)
        g, e = key(part), key(w)
        assert len(g) == len(e), (what, i, len(g), len(e))
        for f in ("src", "x", "y", "z", "r", "g", "b", "i"):
            if key is _by_value and f == "src":
                continue
            bad = np.flatnonzero(g[f] != e[f])
            assert len(bad) == 0, (what, "location %d: %d survivors differ in %s, first at %d" % (i, len(bad), f, bad[0]))
    assert got["stored"] == int(np.sum(counts)) == len(got["src"]), (what, got["stored"], int(np.sum(counts)))
    return parts


# ---- boundary locations (built from the oracle's decoded points; checked on the host first) ---------------------------
ONE_MINUS_2M52 = 0.99999999999999977795539507496869  # 1 - 2^-52, the kernel's threshold factor


def _most_common(v):
    vals, cnt = np.unique(v, return_counts=True)
    return vals[np.argmax(cnt)], int(cnt.max())


def _boundary_aabbs(G, xyz):
    """Two boxes whose faces pass through decoded coordinates that many points share: the shared point lies on the
    inclusive min faces of the first box and on the exclusive max faces of the second (aabb.rs:46-48)."""
    c = np.array([_most_common(xyz[:, a])[0] for a in range(3)])
    return [G.aabb(c, c + 25.0), G.aabb(c - 25.0, c)], c


def _band_frusta(G, xyz):
    """Frusta whose x row puts the points with the most common decoded x exactly at |r| = 1.75: inside the band
    fl(|w| (1 - 2^-52)) < |r| < |w| with w = nextafter(1.75, 2) (from below and, mirrored, from above), and on |r| == |w| with
    w = 1.75.  x near 4.1e6 has a spacing of 2^-31, so c = x_p -+ 1.75 and every x - c are exact."""
    xp = _most_common(xyz[:, 0])[0]
    cy, cz = float(np.median(xyz[:, 1])), float(np.median(xyz[:, 2]))
    s = 2.0 ** -12
    W = np.nextafter(1.75, 2.0)
    out = []
    for sign, w in ((1.0, W), (-1.0, W), (1.0, 1.75)):
        c = xp - sign * 1.75
        assert sign * (xp - c) == 1.75 and (xp - c) + c == xp
        M = np.array([[sign, 0, 0, -sign * c], [0, s, 0, -s * cy], [0, 0, s, -s * cz], [0, 0, 0, w]])
        out.append(G.frustum_from_matrix4(M))
    return out, xp


def _frustum_terms(loc, xyz):
    """r and w of loc_contains in the kernel's operation order (f64 multiply, then add; no fused multiply-add)."""
    m = np.array(loc.clip_from_query[:])
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    n = m[3] * x
    n = n + m[7] * y
    n = n + m[11] * z
    n = n + m[15]
    r = []
    for i in range(3):
        a = m[i] * x
        a = m[4 + i] * y + a
        a = m[8 + i] * z + a
        r.append(a + m[12 + i])
    return np.stack(r, 1), n


def _frustum_inside(loc, xyz):
    """frustum.rs:120-125 in numpy: the divided coordinates strictly inside (-1, 1); plus the band and tie masks."""
    r, n = _frustum_terms(loc, xyz)
    an, ar = np.abs(n), np.abs(r)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(n[:, None] != 0.0, r / n[:, None], r)
    inside = (q.min(1) > -1.0) & (q.max(1) < 1.0)
    T = an * ONE_MINUS_2M52
    band = ((ar > T[:, None]) & (ar < an[:, None])).any(1)
    tie = (ar == an[:, None]).any(1)
    return inside, band, tie


def boundary_cases(G, ref):
    """The boundary locations of one fixture with the checks that need no GPU: the cases really put >= 100 points on the
    faces / in the band / on the tie, and the oracle's own culling agrees with the numpy restatement."""
    every = ref.query(_copy_loc(G.all_points()), with_intensity=True)
    xyz = every["xyz"]
    boxes, c = _boundary_aabbs(G, xyz)
    for k, box in enumerate(boxes):
        lo, hi = np.array(box.aabb_min[:]), np.array(box.aabb_max[:])
        keep = ((xyz >= lo) & (xyz < hi)).all(1)
        closed = ((xyz >= lo) & (xyz <= hi)).all(1)
        on_face = (closed & (xyz == (lo if k == 0 else hi)).any(1)).sum()  # inside through the min face / outside through the max face
        assert on_face >= 100, ("aabb", k, int(on_face))
        w = ref.query(_copy_loc(box))
        assert np.array_equal(np.sort(w["src"]), np.sort(every["src"][keep])), ("aabb", k)
    frusta, xp = _band_frusta(G, xyz)
    lib = O.lib()
    for k, fr in enumerate(frusta):
        inside, band, tie = _frustum_inside(fr, xyz)
        at_xp = xyz[:, 0] == xp
        if k < 2:
            assert band[at_xp].all() and at_xp.sum() >= 100 and inside[at_xp].all(), ("band", k, int(at_xp.sum()))
            assert band.sum() >= 100
        else:
            assert tie[at_xp].all() and tie.sum() >= 100 and not inside[at_xp].any(), ("tie", int(tie.sum()))
        sample = np.flatnonzero(band | tie)[:200]
        sample = np.concatenate([sample, np.flatnonzero(inside)[:100], np.flatnonzero(~inside)[:100]])
        ofr = _copy_loc(fr)
        for i in sample:
            assert bool(lib.orc_location_contains(C.byref(ofr), O._d(xyz[i]))) == bool(inside[i]), ("orc_location_contains", k, int(i))
        w = ref.query(ofr)
        assert np.array_equal(np.sort(w["src"]), np.sort(every["src"][inside])), ("frustum", k)
    return boxes + frusta


# ---- fixtures -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cloud():
    return _cloud()


def _gpu_tree(pcv, cloud, name):
    x, y, z, rgb, inten, bmin, bmax = cloud
    res, mppn = FIXTURES[name]
    ctx = pcv.Context(0, max_points_per_node=mppn)
    return ctx, ctx.build_octree(x, y, z, rgb.reshape(-1), res, bmin, bmax, intensity=inten)


@pytest.fixture(scope="module")
def fixtures(cloud):
    import point_cloud_viewer_b200 as pcv

    G = pcv.geometry
    locs = _locations(G, cloud)
    out = {}
    for name in FIXTURES:
        ref = _oracle_tree(cloud, name)
        ctx, tree = _gpu_tree(pcv, cloud, name)
        compare_trees(ref, tree)
        out[name] = dict(ref=ref, ctx=ctx, tree=tree, want=_oracle_sets(ref, locs))
    yield dict(pcv=pcv, G=G, locs=locs, fx=out)
    for f in out.values():
        f["tree"].free()
        f["ctx"].close()


def _encoding_of_src(tree):
    """Position encoding of the node holding each source index."""
    _, _, _, src = tree.download()
    enc = np.zeros(len(src), np.int64)
    for m in tree.meta:
        enc[int(m["point_offset"]):int(m["point_offset"]) + int(m["num_points"])] = int(m["enc"])
    out = np.zeros(int(src.max()) + 1, np.int64)
    out[src.astype(np.int64)] = enc
    return out


# ---- (a) every location's survivors ------------------------------------------------------------------------------------
def test_survivors_equal_the_oracle_per_location(fixtures):
    locs = fixtures["locs"]
    per_enc = {e: 0 for e in ENC_NAMES}
    for name, f in fixtures["fx"].items():
        counts, tested, got = f["tree"].query_batch_device(locs, points=True)
        parts = _check_against_oracle(counts, tested, got, f["want"], what=name)
        assert len(parts[OUTSIDE]) == 0 and int(counts[OUTSIDE]) == 0, name
        assert len(parts[DUPLICATED]) > 0 and np.array_equal(_by_src(parts[DUPLICATE]), _by_src(parts[DUPLICATED])), name
        assert sum(1 for p in parts if len(p)) >= 35, (name, "locations with survivors")
        enc_of = _encoding_of_src(f["tree"])
        e, k = np.unique(enc_of[got["src"].astype(np.int64)], return_counts=True)
        for ee, kk in zip(e, k):
            per_enc[int(ee)] += int(kk)
    # the location set reaches every position encoding through k_cull_fused's staged (U8/U16/F32) and unstaged (F64) decodes
    assert all(v >= 1000 for v in per_enc.values()), {ENC_NAMES[e]: v for e, v in per_enc.items()}


# ---- (b) interval filters ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("filters", [[100.0, 400.0], [100.0, 400.0, 250.0, 900.0], [500.0, 200.0]], ids=["one", "two", "empty"])
def test_interval_filters(fixtures, filters):
    locs = fixtures["locs"]
    for name, f in fixtures["fx"].items():
        counts, tested, got = f["tree"].query_batch_device(locs, filters=filters, points=True)
        want = _oracle_sets(f["ref"], locs, filters)
        _check_against_oracle(counts, tested, got, want, what=(name, filters))
        lo, hi = max(filters[0::2]), min(filters[1::2])
        assert ((got["intensity"] >= lo) & (got["intensity"] <= hi)).all()
        if lo > hi:
            assert got["stored"] == 0 and int(counts.sum()) == 0
        else:
            assert got["stored"] > 1000


# ---- (c) output capacity ----------------------------------------------------------------------------------------------
def test_capacity_cuts_the_stored_survivors(fixtures):
    locs = fixtures["locs"]
    f = fixtures["fx"]["A"]
    counts, tested = f["tree"].query_batch_device(locs)
    total = int(counts.sum())
    keyed = []
    for i, (w, _) in enumerate(f["want"]):
        k = w.copy()
        k["src"] |= np.uint64(i) << np.uint64(32)
        keyed.append(k)
    allw = _by_src(np.concatenate(keyed))
    for cap in (total - 1, total // 3 + 7, 0):
        c2, t2, got = f["tree"].query_batch_device(locs, points=True, cap=cap)
        assert got["stored"] == min(cap, total) == len(got["src"]), (cap, got["stored"])
        assert np.array_equal(c2, counts) and np.array_equal(t2, tested), cap
        rec = _records(got["xyz"], got["rgb"], got["intensity"], got["src"].astype(np.uint64) | (got["loc"].astype(np.uint64) << np.uint64(32)))
        assert len(np.unique(rec["src"])) == len(rec), (cap, "a (location, source index) pair stored twice")
        at = np.searchsorted(allw["src"], rec["src"])
        at = np.minimum(at, len(allw) - 1)
        assert (allw["src"][at] == rec["src"]).all(), (cap, "stored survivor outside its location's oracle set")
        assert np.array_equal(allw[at], rec), (cap, "stored survivor differs from the oracle's point")


# ---- (d) points on the boundaries, batched and streaming ------------------------------------------------------------
def test_points_on_aabb_faces_and_in_the_frustum_band(fixtures):
    G = fixtures["G"]
    for name, f in fixtures["fx"].items():
        cases = boundary_cases(G, f["ref"])
        want = _oracle_sets(f["ref"], cases)
        counts, tested, got = f["tree"].query_batch_device(cases, points=True)
        _check_against_oracle(counts, tested, got, want, what=(name, "boundaries"))
        for k, loc in enumerate(cases):
            w = f["ref"].query(_copy_loc(loc), with_intensity=True)
            batches = f["tree"].query_points(loc, batch_size=1 << 20)
            cat = lambda key, empty: np.concatenate([b[key] for b in batches]) if batches else empty
            assert np.array_equal(cat("src", np.zeros(0, np.uint64)), w["src"]), (name, k)
            assert np.array_equal(cat("xyz", np.zeros((0, 3))).view(np.uint64), w["xyz"].view(np.uint64)), (name, k)
            assert np.array_equal(cat("rgb", np.zeros((0, 3), np.uint8)), w["rgb"]), (name, k)
            assert np.array_equal(cat("intensity", np.zeros(0, np.float32)), w["intensity"]), (name, k)


# ---- (e) other octrees the batched query reads -------------------------------------------------------------------------
def test_shuffled_and_loaded_octrees(fixtures, cloud, tmp_path):
    pcv, locs = fixtures["pcv"], fixtures["locs"]
    f = fixtures["fx"]["A"]
    ctx, tree = _gpu_tree(pcv, cloud, "A")
    try:
        tree.shuffle_nodes(12345)
        counts, tested, got = tree.query_batch_device(locs, points=True)
        _check_against_oracle(counts, tested, got, f["want"], what="shuffled")
    finally:
        tree.free()
    d = str(tmp_path / "oracle_dir")
    os.makedirs(d)
    f["ref"].write_dir(d)
    loaded = ctx.load_dir(d)
    try:
        counts, tested, got = loaded.query_batch_device(locs, points=True)
        _check_against_oracle(counts, tested, got, f["want"], key=_by_value, what="loaded")
    finally:
        loaded.free()
        ctx.close()
