"""Seeded clouds for the wide VoxelGrid tests (tests/test_map_export_reference.py, tests/test_gpu_map_export.py): grids just
either side of INT32_MAX cells, far-apart clusters with 33- to 63-bit keys, and the refusal limits of the wide grid at both
edges.  Each returns (N, 4) float32 [x, y, z, intensity]."""
import numpy as np

INT32_MAX = 2 ** 31 - 1
# 2^63 - 1 = 4547599 * 6769801 * 299593, every factor below 2^24: the corners of such a box are exact floats at a 1 m leaf
DIV_AT_INT64_MAX = (4547599, 6769801, 299593)


def cube(side, n=200_000, seed=1):
    """Points in a cube of exactly `side` cells per axis at leaf 1.0 (div_b = side^3), corners included."""
    rng = np.random.default_rng(seed)
    p = np.empty((n, 4), np.float32)
    p[:, :3] = rng.uniform(0.0, side - 0.5, (n, 3)).astype(np.float32)
    p[:, 3] = rng.uniform(0, 255, n).astype(np.float32)
    p[0, :3] = 0.0
    p[1, :3] = side - 0.5
    return p


def clusters(extent, n=120_000, spread=0.5, seed=2, dirty=True):
    """Blobs at the corners of a box of `extent` metres (x, y, z): a grid of 2^33 to 2^48 cells at a centimetre-scale leaf
    that holds few occupied ones.  dirty: NaN / Inf rows and runs of exactly repeated points (many members per voxel)."""
    rng = np.random.default_rng(seed)
    ext = np.asarray(extent, np.float64)
    corners = np.array([[0, 0, 0], [1, 1, 1], [1, 0, 0], [0, 1, 1], [0.5, 0.25, 0.75]], np.float64) * ext
    c = corners[rng.integers(0, len(corners), n)]
    p = np.empty((n, 4), np.float32)
    p[:, :3] = (c + rng.normal(0.0, spread, (n, 3))).astype(np.float32)
    p[:, 3] = rng.uniform(0, 255, n).astype(np.float32)
    if dirty:
        rows = rng.choice(n, 300, replace=False)
        p[rows[:100], 0] = np.nan
        p[rows[100:200], 1] = np.inf
        p[rows[200:], 2] = -np.inf
        dup = rng.choice(n, 2000, replace=False)
        p[dup] = p[dup[0]]
        p[rng.choice(n, 500, replace=False), :3] = p[5, :3]
    return p


def far_from_origin(n=80_000, seed=3):
    """A cluster 20 km out at a 1 mm leaf: 2e7 leaf units, beyond 2^24, where PCL's f32 cell index merges cells."""
    rng = np.random.default_rng(seed)
    p = np.empty((n, 4), np.float32)
    base = np.where(rng.random(n) < 0.5, 0.0, 20000.0)[:, None] * np.array([1.0, 0.0, 0.0])
    p[:, :3] = (base + rng.uniform(0.0, 1.0, (n, 3))).astype(np.float32)
    p[:, 3] = rng.uniform(0, 255, n).astype(np.float32)
    return p


def key63(over, n=50_000, seed=4):
    """A 1 mm leaf over a cube of just under (over=False) or just over (over=True) 2^21 cells per axis: 63-bit keys below,
    a cell product beyond 2^63 - 1 above."""
    rng = np.random.default_rng(seed)
    side = (2 ** 21 + 2 if over else 2 ** 21 - 4) * 0.001
    p = np.empty((n, 4), np.float32)
    p[:, :3] = rng.uniform(0.0, side, (n, 3)).astype(np.float32)
    p[:, 3] = rng.uniform(0, 255, n).astype(np.float32)
    p[0, :3] = 0.0
    p[1, :3] = np.float32(side)
    return p


def two_points(a, b):
    p = np.zeros((2, 4), np.float32)
    p[0, :3], p[1, :3] = a, b
    p[:, 3] = (1.0, 2.0)
    return p


def refusal_edges():
    """(name, cloud, leaf, refused) at both sides of each limit of the wide grid."""
    e30 = 2.0 ** 30
    d0, d1, d2 = DIV_AT_INT64_MAX
    s21 = 2 ** 21
    return [
        ("extent_below", two_points((-e30, 0, 0), (e30 - 128, 0, 0)), 1.0, False),   # (mx - mn) * inv = 2^31 - 128
        ("extent_at", two_points((-e30, 0, 0), (e30, 0, 0)), 1.0, True),             # = 2^31
        ("min_b_fits", two_points((-2.0 ** 31, 0, 0), (-2.0 ** 31, 0, 0)), 1.0, False),
        ("min_b_below_int32", two_points((-2.0 ** 31 - 256, 0, 0), (-2.0 ** 31 - 256, 0, 0)), 1.0, True),
        ("max_b_fits", two_points((2.0 ** 31 - 128, 0, 0), (2.0 ** 31 - 128, 0, 0)), 1.0, False),
        ("max_b_above_int32", two_points((2.0 ** 31, 0, 0), (2.0 ** 31, 0, 0)), 1.0, True),
        ("cells_int64_max", two_points((0, 0, 0), (d0 - 1, d1 - 1, d2 - 1)), 1.0, False),  # product = 2^63 - 1
        ("cells_over_int64_max", two_points((0, 0, 0), (d0 - 1, d1 - 1, d2)), 1.0, True),
        ("cells_2_63", two_points((0, 0, 0), (s21 - 1, s21 - 1, s21 - 1)), 1.0, True),
        ("cells_2_63_minus", two_points((0, 0, 0), (s21 - 1, s21 - 1, s21 - 2)), 1.0, False),
    ]


def restate_wide(pts, leaf):
    """Independent numpy restatement of the wide grid (no crop, no min_pts) for clouds it does not refuse: per-axis index
    with np.float32 ops, int64 keys, stable argsort.  Returns keys per input point (-1 if not finite), centroids, counts and
    the membership rank per input point."""
    pts = np.asarray(pts, np.float32)
    finite = np.isfinite(pts[:, :3]).all(axis=1)
    kept = np.nonzero(finite)[0]
    p = pts[kept]
    inv = np.float32(1.0) / np.float32(leaf)
    fmin = np.floor(p[:, :3].min(axis=0) * inv)
    fmax = np.floor(p[:, :3].max(axis=0) * inv)
    div = fmax.astype(np.int64) - fmin.astype(np.int64) + 1
    ijk = (np.floor(p[:, :3] * inv) - fmin).astype(np.int64)
    key = ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * (div[0] * div[1])
    order = np.argsort(key, kind="stable")
    sk = key[order]
    heads = np.nonzero(np.r_[True, sk[1:] != sk[:-1]])[0]
    counts = np.diff(np.r_[heads, len(sk)])
    # sequential f32 sums in ascending point index (np.cumsum adds left to right)
    ps = p[order]
    cent = ps[heads].copy()
    for v in np.nonzero(counts > 1)[0]:
        b = heads[v]
        cent[v] = np.cumsum(ps[b:b + counts[v]], axis=0, dtype=np.float32)[-1] / np.float32(counts[v])
    rank_sorted = np.repeat(np.arange(len(heads)), counts)
    keys = np.full(len(pts), -1, np.int64)
    keys[kept] = key
    rank = np.full(len(pts), -1, np.int32)
    rank[kept[order]] = rank_sorted
    return dict(keys=keys, out_idx=sk[heads], centroids=cent, counts=counts, member_rank=rank, min_b=fmin.astype(np.int64),
                div_b=div)
