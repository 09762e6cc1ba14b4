"""The numpy restatement of point_cloud_test's SyntheticData (reference_synthetic.py) that the S2-vs-octree GPU test runs on."""
import numpy as np

from reference_synthetic import chacha20_u64, synthetic_data


def test_chacha20_keystream():
    # RFC 8439 A.1 test vector 1 (all-zero key, nonce and counter), read as rand_core's little-endian next_u64 pairs
    assert [int(v) for v in chacha20_u64([0] * 8, 4)] == [0x903DF1A0ADE0B876, 0x28BD8653E56A5D40, 0x1AED8DA0B819D2BD, 0xC70D778BCCEF36A8]


def test_synthetic_data_shape():
    d = synthetic_data(1000)
    half = np.array([100.0, 100.0, 10.0])
    assert d["xyz"].shape == (1000, 3) and np.all(d["xyz"] >= d["bbox_min"] - 1e-6) and np.all(d["xyz"] <= d["bbox_max"] + 1e-6)
    assert np.isclose(np.linalg.norm(d["origin"]), 6.36e6, rtol=2e-3)  # on the ellipsoid
    assert np.allclose(np.linalg.norm(d["xyz"] - d["origin"], axis=1).max(), np.linalg.norm(half), rtol=0.05)
    idx = (d["rgb"][:, 0].astype(np.int64) << 16) + (d["rgb"][:, 1].astype(np.int64) << 8) + d["rgb"][:, 2]
    assert np.array_equal(idx, np.arange(1000))
    assert np.array_equal(synthetic_data(1000)["xyz"], d["xyz"])  # seeded: the same points every run
