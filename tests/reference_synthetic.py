"""point_cloud_test's SyntheticData (point_cloud_test/src/synthetic_data.rs:22-78) restated in numpy, so that a test can run on
the very points the reference's integration tests use: rand 0.7's StdRng (ChaCha20, seeded from a u64 through PCG32 as
rand_core 0.5's seed_from_u64 does), gen_range for f64 as UniformFloat::sample_single ([1, 2) mantissa draw minus one, times
the span, plus the low end), the slab's frame from the first two draws (math/mod.rs:167-183 local_frame_from_lat_lng, WGS84 to
ECEF), then three draws per point.  The frame is composed in numpy, so coordinates may differ from the reference's in the last
bits; the draws themselves are exact."""
import numpy as np

_M32 = np.uint64(0xFFFFFFFF)


def _pcg32_seed(state):
    mul, inc, m64 = 6364136223846793005, 11634580027462260723, (1 << 64) - 1
    words = []
    for _ in range(8):
        state = (state * mul + inc) & m64
        xs = (((state >> 18) ^ state) >> 27) & 0xFFFFFFFF
        rot = state >> 59
        words.append(((xs >> rot) | (xs << ((32 - rot) & 31))) & 0xFFFFFFFF)
    return words


def chacha20_u64(key_words, count):
    """The first `count` next_u64() of rand_chacha's ChaCha20Rng with this key (nonce 0, block counter from 0)."""
    nblocks = (2 * count + 15) // 16
    ctr = np.arange(nblocks, dtype=np.uint64)
    init = [np.full(nblocks, w, np.uint32) for w in (0x61707865, 0x3320646E, 0x79622D32, 0x6B206574)]
    init += [np.full(nblocks, w, np.uint32) for w in key_words]
    init += [(ctr & _M32).astype(np.uint32), (ctr >> np.uint64(32)).astype(np.uint32), np.zeros(nblocks, np.uint32), np.zeros(nblocks, np.uint32)]
    x = [w.copy() for w in init]

    def rotl(v, c):
        return (v << np.uint32(c)) | (v >> np.uint32(32 - c))

    def qr(a, b, c, d):
        x[a] += x[b]
        x[d] = rotl(x[d] ^ x[a], 16)
        x[c] += x[d]
        x[b] = rotl(x[b] ^ x[c], 12)
        x[a] += x[b]
        x[d] = rotl(x[d] ^ x[a], 8)
        x[c] += x[d]
        x[b] = rotl(x[b] ^ x[c], 7)

    with np.errstate(over="ignore"):
        for _ in range(10):
            qr(0, 4, 8, 12), qr(1, 5, 9, 13), qr(2, 6, 10, 14), qr(3, 7, 11, 15)
            qr(0, 5, 10, 15), qr(1, 6, 11, 12), qr(2, 7, 8, 13), qr(3, 4, 9, 14)
        words = np.stack([x[i] + init[i] for i in range(16)], 1).reshape(-1)[: 2 * count].astype(np.uint64)
    return words[0::2] | (words[1::2] << np.uint64(32))


def _quat(axis, angle):
    return np.array([np.cos(angle / 2)] + list(np.sin(angle / 2) * np.asarray(axis, np.float64)))


def _quat_mul(a, b):
    w1, x1, y1, z1 = a
    w2, x2, y2, z2 = b
    return np.array([w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2, w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                     w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2, w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2])


def _quat_matrix(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def synthetic_data(num_points, seed=80_293_751_232, width=200.0, height=20.0):
    """SyntheticData::new(width, height, num_points, seed) (Arguments::default, point_cloud_test/src/lib.rs:42-61), drained.
    Returns dict(xyz (n, 3) f64, rgb (n, 3) u8 with the index in the colour, bbox_min, bbox_max (SyntheticData::bbox),
    origin (ecef_from_local's translation))."""
    u = chacha20_u64(_pcg32_seed(seed), 2 + 3 * num_points)
    unit = ((u >> np.uint64(12)) | np.uint64(0x3FF0000000000000)).view(np.float64) - 1.0
    lat = np.radians(unit[0] * 180.0 - 90.0)
    lon = np.radians(unit[1] * 360.0 - 180.0)
    a, f = 6378137.0, 1.0 / 298.257223563
    e2 = f * (2.0 - f)
    nrad = a / np.sqrt(1.0 - e2 * np.sin(lat) ** 2)
    origin = np.array([nrad * np.cos(lat) * np.cos(lon), nrad * np.cos(lat) * np.sin(lon), nrad * (1.0 - e2) * np.sin(lat)])
    local_from_ecef = _quat_mul(_quat_mul(_quat([0, 0, 1], -np.pi / 2), _quat([0, 1, 0], lat - np.pi / 2)), _quat([0, 0, 1], -lon))
    rot = _quat_matrix(local_from_ecef).T
    half = np.array([width / 2, width / 2, height / 2])
    local = unit[2:].reshape(num_points, 3) * (2.0 * half) - half
    corners = np.array([[sx, sy, sz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)]) * half
    i = np.arange(num_points)
    rgb = np.stack([(i >> 16) & 255, (i >> 8) & 255, i & 255], 1).astype(np.uint8)
    return dict(xyz=local @ rot.T + origin, rgb=rgb, bbox_min=(corners @ rot.T + origin).min(0), bbox_max=(corners @ rot.T + origin).max(0), origin=origin)
