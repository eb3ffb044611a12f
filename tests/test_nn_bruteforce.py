"""The brute-force nearest-neighbour reference (nn_bruteforce.py) against the oracle's kd-tree and outlier filter, bit for
bit, on clouds full of ties and at the ends of f32's range.  Needs no GPU: it makes sure that the reference the GPU
tests judge the CUDA index by (test_gpu_nn_exact.py) is itself right, so that it can neither pass nor fail them for the
wrong reason."""
import numpy as np
import pytest

from nn_bruteforce import bf_knn, bf_sor_distances, cloud, lattice, lattice_queries, sor_threshold, transform_pcl


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _edge_clouds():
    rng = np.random.default_rng(20)
    u = rng.uniform(-20, 20, (600, 3)).astype(np.float32)
    uq = rng.uniform(-25, 25, (150, 3)).astype(np.float32)
    plane = u.copy()
    plane[:, 2] = 0
    dupes = np.repeat(u[:3], 70, axis=0)[rng.permutation(210)]
    return {
        "lattice": (lattice((7, 6, 5), rng), lattice_queries((7, 6, 5), rng, 150)),
        "dupes": (cloud(dupes), cloud(np.concatenate([u[:3], uq[:60]]))),
        "subnormal_squares": (cloud(u * np.float32(1e-22)), cloud(uq * np.float32(1e-22))),
        "overflowing_squares": (cloud(u * np.float32(1e20)), cloud(uq * np.float32(1e20))),
        "offset_1e5": (cloud(u + np.float32(1e5)), cloud(uq + np.float32(1e5))),
        "plane": (cloud(plane), cloud(uq)),
    }


EDGE = _edge_clouds()


@pytest.mark.parametrize("name", sorted(EDGE))
@pytest.mark.parametrize("k", [1, 6, 7, 32])
def test_bf_knn_matches_oracle(oracle, name, k):
    pts, q = EDGE[name]
    q = np.concatenate([q, pts[:40]])  # queries on indexed points too (distance 0, duplicates)
    io, do = oracle.knn(pts, q, k)
    ib, db = bf_knn(pts, q, k)
    assert np.array_equal(ib, io)
    assert np.array_equal(_bits(db), _bits(do))


@pytest.mark.parametrize("n", [1, 5, 31])
def test_bf_knn_pads_like_the_kernel(oracle, n):
    pts, q = EDGE["lattice"]
    ib, db = bf_knn(pts[:n], q, 32)
    io, do = oracle.knn(pts[:n], q, 32)
    assert np.array_equal(ib, io) and np.array_equal(_bits(db), _bits(do))
    assert (ib[:, n:] == -1).all() and (_bits(db[:, n:]) == 0).all() and (ib[:, :n] >= 0).all()


def test_bf_knn_collapsed_distances_are_really_tied():
    # the clouds above only test what they claim if f32 really collapses their distances onto few values
    _, d_sub = bf_knn(*EDGE["subnormal_squares"], 32)
    _, d_big = bf_knn(*EDGE["overflowing_squares"], 32)
    sub = d_sub[d_sub > 0]
    assert sub.size and (sub < np.finfo(np.float32).tiny).all()  # subnormal squares, not flushed to zero
    assert np.isinf(d_big).mean() > 0.5


@pytest.mark.parametrize("name", sorted(EDGE))
@pytest.mark.parametrize("mean_k", [1, 5, 30, 31])
def test_bf_sor_matches_oracle(oracle, name, mean_k):
    pts, _ = EDGE[name]
    ref = oracle.statistical_outlier_removal(pts, mean_k=mean_k, stddev_mul=1.0)
    dist = bf_sor_distances(pts, mean_k)
    assert np.array_equal(_bits(dist), _bits(ref["distances"]))
    thr = sor_threshold(dist, 1.0)
    assert np.array_equal(np.float64(thr), np.float64(ref["threshold"]), equal_nan=True)
    assert np.array_equal(~(dist > thr), ref["keep"])


def test_bf_sor_small_cloud_divides_by_mean_k(oracle):
    pts = EDGE["lattice"][0][:5]
    ref = oracle.statistical_outlier_removal(pts, mean_k=30, stddev_mul=1.0)
    assert np.array_equal(_bits(bf_sor_distances(pts, 30)), _bits(ref["distances"]))


def test_transform_pcl_matches_oracle(oracle):
    rng = np.random.default_rng(3)
    pts = cloud(rng.uniform(-80, 80, (2000, 3)))
    pts[:, 3] = rng.uniform(0, 1, 2000)
    c, s = np.cos(0.3), np.sin(0.3)
    T = np.array([[c, -s, 0.1, 1.5], [s, c, -0.2, -2.25], [0.05, 0.2, 0.97, 0.3], [0, 0, 0, 1]], np.float32)
    assert np.array_equal(transform_pcl(T, pts).view(np.uint32), oracle.transform_point_cloud(pts, T).view(np.uint32))
