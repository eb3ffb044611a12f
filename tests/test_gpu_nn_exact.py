"""Exactness of the nearest-neighbour index (csrc/nn.cuh, nn.cu) against brute force (nn_bruteforce.py), through every
consumer: lgs_knn, the seeded and unseeded 1-NN of the correspondence searches, the statistical outlier filter, FastGICP's
lazy target covariances and getFitnessScore.

nn.cuh promises the exact neighbours with ties going to the smaller original index, so every comparison here is on
indices and on the bits of the f32 squared distances; only getFitnessScore, a sum in another order, gets a tolerance.
The clouds sit on the index's structural edges (leaf and node boundaries, the largest 3-level tree and the smallest
6-level one, the grid-stride loop of the query kernel) and on its numerical ones (lattices and duplicates full of ties,
zero extents, coordinates where f32 distances collapse, subnormal and overflowing squares).  Non-finite points are not
defined for the search and are left out."""
import zlib

import numpy as np
import pytest

from nn_bruteforce import bf_knn, cloud, lattice, lattice_queries, sor_distances_from_knn, sor_threshold, transform_pcl

pytestmark = pytest.mark.gpu

KS = (1, 2, 5, 6, 7, 20, 31, 32)
INT32_MAX = 2 ** 31 - 1
DBL_MAX = float(np.finfo(np.float64).max)
BIG_SHAPE = (128, 128, 64)  # 2^20 points: the largest cloud of a 3-level tree, with a full top node


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _assert_rows(gi, gd, ri, rd, what):
    assert gi.shape == ri.shape, what
    bad = np.nonzero((gi != ri).any(axis=1) | (_bits(gd) != _bits(rd)).any(axis=1))[0]
    assert bad.size == 0, "%s: %d rows differ, first %d: got %s / %s, want %s / %s" % (
        what, bad.size, bad[0], gi[bad[0]], gd[bad[0]], ri[bad[0]], rd[bad[0]])


def _check_knn(api, pts, q, ks=KS, what=""):
    ri, rd = bf_knn(pts, q, max(ks))  # the k-NN rows are prefixes of the 32-NN rows
    for k in ks:
        gi, gd = api.knn(pts, q, k)
        _assert_rows(gi, gd, ri[:, :k], rd[:, :k], "%s k=%d" % (what, k))


def _uniform(rng, n, lo=-50.0, hi=50.0):
    return cloud(rng.uniform(lo, hi, (n, 3)))


def _mixed_queries(rng, pts, m=200, lo=-55.0, hi=55.0):
    """random queries around the cloud, some indexed points and a few queries 10 km outside the bounding box"""
    far = rng.normal(size=(8, 3))
    far = far / np.linalg.norm(far, axis=1, keepdims=True) * 1e4
    parts = [rng.uniform(lo, hi, (m, 3)), pts[rng.integers(0, len(pts), min(50, len(pts))), :3], far]
    return cloud(np.concatenate(parts))


# ---- geometries -----------------------------------------------------------------------------------------------------

def _geometry(name):
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    if name == "uniform":
        p = _uniform(rng, 5000)
        return p, _mixed_queries(rng, p)
    if name == "lattice":
        shape = (12, 11, 10)
        return lattice(shape, rng), lattice_queries(shape, rng, 600)
    if name == "repeated_point":  # 100 copies of one point among others: they span several leaves
        p = _uniform(rng, 3000)
        p[rng.choice(3000, 100, replace=False), :3] = p[0, :3]
        q = _mixed_queries(rng, p)
        q = np.concatenate([q, cloud(p[[0] * 3, :3] + np.float32([[0, 0, 0], [0.01, 0, 0], [0, 0.3, -0.2]]))])
        return p, q
    if name == "identical":
        p = cloud(np.repeat(np.float32([[3.25, -1.5, 0.75]]), 500, axis=0))
        return p, cloud(np.concatenate([p[:1, :3], rng.uniform(-5, 5, (100, 3))]))
    if name == "plane":  # zero extent in z
        p = _uniform(rng, 3000)
        p[:, 2] = 0
        return p, _mixed_queries(rng, p)
    if name == "line":  # zero extent in y and z
        p = _uniform(rng, 3000)
        p[:, 1:3] = 0
        return p, _mixed_queries(rng, p)
    if name == "offset_1e5":  # f32 spacing 2^-7 m: distances collapse onto few values; 20 points appear twice
        p = cloud(rng.uniform(-50, 50, (3000, 3)).astype(np.float32) + np.float32(1e5))
        p = np.concatenate([p, p[:20]])
        return p, np.concatenate([cloud(rng.uniform(-55, 55, (300, 3)).astype(np.float32) + np.float32(1e5)), p[:20]])
    if name == "scale_1e-22":  # squares are f32 subnormals: any flush-to-zero shows
        p = cloud(rng.uniform(-50, 50, (3000, 3)).astype(np.float32) * np.float32(1e-22))
        return p, cloud(rng.uniform(-55, 55, (300, 3)).astype(np.float32) * np.float32(1e-22))
    if name == "scale_1e20":  # most squares overflow to +inf: ties at +inf go to the smaller index
        p = cloud(rng.uniform(-50, 50, (3000, 3)).astype(np.float32) * np.float32(1e20))
        return p, cloud(rng.uniform(-55, 55, (300, 3)).astype(np.float32) * np.float32(1e20))
    raise KeyError(name)


GEOMETRIES = ["uniform", "lattice", "repeated_point", "identical", "plane", "line", "offset_1e5", "scale_1e-22", "scale_1e20"]


@pytest.mark.parametrize("name", GEOMETRIES)
def test_knn_geometries(api, name):
    pts, q = _geometry(name)
    _check_knn(api, pts, q, what=name)


def test_knn_velodyne(api, oracle, velodyne_pair):
    pts = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    q = np.concatenate([oracle.voxel_grid(velodyne_pair["source"], 0.4)["points"], pts[::50]])
    _check_knn(api, pts, q, what="velodyne")


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 1023, 1024, 1025, 32768, 32769])
def test_knn_sizes(api, n):
    rng = np.random.default_rng(n)
    pts = _uniform(rng, n)
    _check_knn(api, pts, _mixed_queries(rng, pts), what="n=%d" % n)


@pytest.mark.parametrize("n", [0, 1, 5, 31])
def test_knn_pads_rows_beyond_the_cloud(api, n):
    rng = np.random.default_rng(100 + n)
    pts = _uniform(rng, n)
    q = _mixed_queries(rng, pts, m=40) if n else _uniform(rng, 40)
    gi, gd = api.knn(pts, q, 32)
    assert (gi[:, n:] == -1).all() and (_bits(gd[:, n:]) == 0).all()
    ri, rd = bf_knn(pts, q, 32)
    _assert_rows(gi, gd, ri, rd, "n=%d k=32" % n)


def test_knn_grid_stride(api):
    # 200 003 queries: more warps than one launch of nn_knn_kernel has (148 SMs x 64 CTAs x 8 warps = 75 776)
    rng = np.random.default_rng(5)
    pts = _uniform(rng, 1000)
    q = _uniform(rng, 200003, -60, 60)
    _check_knn(api, pts, q, ks=(7, 32), what="m=200003")


# ---- the 3-level / 6-level boundary ---------------------------------------------------------------------------------

@pytest.fixture(scope="module", params=[0, 1], ids=["n=1048576", "n=1048577"])
def big(request):
    """A 128 x 128 x 64 lattice (2^20 points, the largest 3-level tree) and, for the second parameter, the same lattice
    plus a duplicate of one of its points (the smallest 6-level tree), with about 1 000 queries on lattice points, cell
    and face centres and the duplicated point, and their brute-force 32-NN."""
    rng = np.random.default_rng(2020)
    pts = lattice(BIG_SHAPE, rng)
    dup = 123457
    if request.param:
        pts = np.concatenate([pts, pts[dup:dup + 1]])  # the copy has the larger index: queries there must return dup
    q = np.concatenate([lattice_queries(BIG_SHAPE, rng, 900), pts[[dup] * 4], cloud(rng.uniform(-3, 130, (96, 3)))])
    ri, rd, far = bf_knn(pts, q, 32, farthest=True)
    return dict(pts=pts, q=q, ri=ri, rd=rd, far=far, dup=dup)


def test_knn_largest_3_level_and_smallest_6_level_tree(api, big):
    pts, q = big["pts"], big["q"]
    for k in KS:
        gi, gd = api.knn(pts, q, k)
        _assert_rows(gi, gd, big["ri"][:, :k], big["rd"][:, :k], "n=%d k=%d" % (len(pts), k))
    assert (big["ri"][-100:-96, 0] == big["dup"]).all()


# ---- seeded 1-NN ----------------------------------------------------------------------------------------------------

def _seed_sets(rng, n, ri, rd, far):
    """the seeds every query is run with: the true answer, a tie partner (an equally near point with a larger index, or the
    answer where there is none), a random point, the farthest point, and three that mean 'no seed'"""
    tie = ri[:, 0].copy()
    for j in range(1, ri.shape[1]):
        same = (ri[:, j] >= 0) & (_bits(rd[:, j]) == _bits(rd[:, 0]))
        tie[same] = ri[same, j]
    m = len(ri)
    return {
        "answer": ri[:, 0], "tie_partner": tie, "random": rng.integers(0, n, m).astype(np.int32), "farthest": far.astype(np.int32),
        "minus_one": np.full(m, -1, np.int32), "n": np.full(m, n, np.int32), "int32_max": np.full(m, INT32_MAX, np.int32),
    }


def _check_search1(api, pts, q, ri, rd, far, what):
    sets = _seed_sets(np.random.default_rng(len(pts)), len(pts), ri, rd, far)
    assert (sets["tie_partner"] != sets["answer"]).any(), "%s: no query with a tied neighbour" % what
    runs = [("none", None)] + sorted(sets.items())
    for name, seeds in runs:
        gi, gd = api.nn_search1(pts, q, seeds)
        _assert_rows(gi[:, None], gd[:, None], ri[:, :1], rd[:, :1], "%s seed=%s" % (what, name))


@pytest.mark.parametrize("name", ["lattice", "repeated_point", "offset_1e5"])
def test_search1_seeded(api, name):
    pts, q = _geometry(name)
    ri, rd, far = bf_knn(pts, q, 32, farthest=True)
    _check_search1(api, pts, q, ri, rd, far, name)


def test_search1_seeded_big(api, big):
    _check_search1(api, big["pts"], big["q"], big["ri"], big["rd"], big["far"], "n=%d" % len(big["pts"]))


def test_search1_empty_cloud(api):
    q = _uniform(np.random.default_rng(1), 10)
    for seeds in (None, np.zeros(10, np.int32)):
        gi, gd = api.nn_search1(np.zeros((0, 4), np.float32), q, seeds)
        assert (gi == -1).all() and np.isinf(gd).all() and (gd > 0).all()


# ---- statistical outlier filter (nn_self_knn) -----------------------------------------------------------------------

SOR_CLOUDS = ["uniform", "lattice", "repeated_point", "identical", "plane", "offset_1e5", "scale_1e-22"]


@pytest.mark.parametrize("mean_k", [1, 5, 30, 31])
@pytest.mark.parametrize("name", SOR_CLOUDS)
def test_sor(api, name, mean_k):
    pts, _ = _geometry(name)
    ri, rd = bf_knn(pts, pts, mean_k + 1)
    dist = sor_distances_from_knn(ri, rd, mean_k)
    s = api.StatisticalOutlierRemoval()
    s.setMeanK(mean_k)
    s.setStddevMulThresh(1.0)
    s.setInputCloud(pts)
    out = s.filter()
    assert np.array_equal(_bits(s.distances), _bits(dist))
    thr = sor_threshold(dist, 1.0)
    # the kernel sums the distances in a tree order, the restatement serially: equal up to the f64 rounding of the sums
    assert np.isnan(s.info.threshold) == np.isnan(thr)
    if not np.isnan(thr):
        assert s.info.threshold == pytest.approx(thr, rel=1e-12, abs=1e-300)
    keep = ~(dist > s.info.threshold)
    assert np.array_equal(s.keep, keep)
    clear = np.isnan(thr) | (np.abs(dist.astype(np.float64) - thr) > 1e-9 * abs(thr))
    assert np.array_equal(s.keep[clear], ~(dist[clear] > thr))
    assert np.array_equal(out, pts[keep])


def test_sor_distances_6_level_tree(api):
    rng = np.random.default_rng(77)
    pts = lattice(BIG_SHAPE, rng)
    pts = np.concatenate([pts, pts[:1]])  # 2^20 + 1 points
    rows = rng.choice(len(pts), 2000, replace=False)
    rows[0] = 0
    rows[1] = len(pts) - 1  # the duplicated point and its copy
    ri, rd = bf_knn(pts, pts[rows], 32)
    for mean_k in (1, 5, 30, 31):
        s = api.StatisticalOutlierRemoval()
        s.setMeanK(mean_k)
        s.setInputCloud(pts)
        s.filter()
        assert np.array_equal(_bits(s.distances[rows]), _bits(sor_distances_from_knn(ri, rd, mean_k))), "mean_k=%d" % mean_k


# ---- FastGICP: lazy (nn_knn_list) against eager (nn_self_knn) target covariances ------------------------------------

def _pose(rx, ry, rz, tx, ty, tz):
    cx, sx, cy, sy, cz, sz = np.cos(rx), np.sin(rx), np.cos(ry), np.sin(ry), np.cos(rz), np.sin(rz)
    R = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]]) @ np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    T = np.eye(4)
    T[:3, :3], T[:3, 3] = R, (tx, ty, tz)
    return T


@pytest.mark.parametrize("k", [10, 20, 32])
def test_gicp_lazy_target_covariances_match_eager(api, k):
    # The target has more than 3/2 of the source's points, so FastGICP computes target covariances lazily, for the matched
    # points only (nn_knn_list); asking for them first (covariances(1)) makes it compute all of them up front
    # (nn_self_knn).  Both must give the same neighbour lists, hence bitwise the same linearisation.  (The lazy path is
    # the default; LGS_GICP_LAZY_TARGET=0 would turn it off.)
    rng = np.random.default_rng(k)
    tgt = lattice((20, 20, 8), rng, spacing=0.5)
    tgt[:, :3] += rng.integers(-1, 2, (len(tgt), 3)).astype(np.float32) * np.float32(0.125)  # lattice-like, still tied
    src = tgt[rng.choice(len(tgt), 1000, replace=False)].copy()
    src[:, :3] += rng.uniform(-0.2, 0.2, (1000, 3)).astype(np.float32)
    objs = []
    for eager in (False, True):
        g = api.FastGICP()
        g.setCorrespondenceRandomness(k)
        g.setMaxCorrespondenceDistance(1e6)
        g.setInputTarget(tgt)
        g.setInputSource(src)
        if eager:
            g.covariances(1)
        objs.append(g)
    poses = [np.eye(4), _pose(0.02, -0.01, 0.05, 0.1, -0.2, 0.05), _pose(-0.1, 0.05, 0.3, 1.0, 0.5, -0.25), _pose(0, 0, -0.2, -0.4, 0, 0)]
    for i, T in enumerate(poses):
        a, b = objs[0].linearize(T), objs[1].linearize(T)
        for x, y, what in zip(a, b, ("cost", "H", "b", "correspondences")):
            assert np.array_equal(np.asarray(x), np.asarray(y)), "pose %d: %s differs" % (i, what)
    # at the identity the queries are the source points themselves: the correspondences are their exact 1-NN
    ri, _ = bf_knn(tgt, src, 1)
    assert np.array_equal(objs[0].linearize(np.eye(4))[3], ri[:, 0])
    assert np.array_equal(objs[1].linearize(np.eye(4))[3], ri[:, 0])


# ---- getFitnessScore (nn_fitness_kernel) ----------------------------------------------------------------------------

def _fitness_ref(d2, max_range):
    d = d2.astype(np.float64)
    sel = d <= max_range
    return float(np.sum(d[sel])) / int(sel.sum()) if sel.any() else DBL_MAX


def test_fitness(api, oracle, velodyne_pair):
    tgt = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    src = oracle.voxel_grid(velodyne_pair["source"], 0.4)["points"]
    icp = api.IterativeClosestPoint()
    icp.setMaximumIterations(5)
    icp.setMaxCorrespondenceDistance(5.0)
    icp.setInputTarget(tgt)
    icp.setInputSource(src)
    icp.align()
    q = transform_pcl(icp.getFinalTransformation(), src)
    d2 = bf_knn(tgt, q, 1)[1][:, 0]
    assert d2.min() > 0
    # the kernel sums in another order than the reference: equal up to the f64 rounding of the sums
    assert icp.getFitnessScore() == pytest.approx(_fitness_ref(d2, DBL_MAX), rel=1e-12)
    # a max_range equal to one of the distances: the boundary is inclusive (<=, as PCL)
    mr = float(np.sort(d2)[len(d2) // 2])
    assert _fitness_ref(d2, mr) != _fitness_ref(d2, np.nextafter(mr, 0))
    assert icp.getFitnessScore(mr) == pytest.approx(_fitness_ref(d2, mr), rel=1e-12)
    # below every distance: nothing counts and PCL returns DBL_MAX
    assert icp.getFitnessScore(float(d2.min()) / 2) == DBL_MAX
    # max_range 0 with target points exactly where some transformed source points land
    icp.setInputTarget(np.concatenate([tgt, q[::7]]))
    assert icp.getFitnessScore(0.0) == 0.0
    assert icp.getFitnessScore() == pytest.approx(_fitness_ref(bf_knn(np.concatenate([tgt, q[::7]]), q, 1)[1][:, 0], DBL_MAX), rel=1e-12)


def test_fitness_6_level_tree(api, oracle, velodyne_pair):
    tgt = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    src = oracle.voxel_grid(velodyne_pair["source"], 0.4)["points"][:700]
    icp = api.IterativeClosestPoint()
    icp.setMaximumIterations(3)
    icp.setInputTarget(tgt)
    icp.setInputSource(src)
    icp.align()
    rng = np.random.default_rng(9)
    big = lattice(BIG_SHAPE, rng)
    big = np.concatenate([big, big[:1]])
    big[:, :3] -= np.float32([64, 64, 8])  # around the scan
    icp.setInputTarget(big)
    q = transform_pcl(icp.getFinalTransformation(), src)
    d2 = bf_knn(big, q, 1)[1][:, 0]
    assert icp.getFitnessScore() == pytest.approx(_fitness_ref(d2, DBL_MAX), rel=1e-12)
    mr = float(np.sort(d2)[len(d2) // 3])
    assert icp.getFitnessScore(mr) == pytest.approx(_fitness_ref(d2, mr), rel=1e-12)
