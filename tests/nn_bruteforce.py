"""Brute-force reference of the exact nearest-neighbour searches (csrc/nn.cuh) and of the statistical outlier filter's
mean neighbour distances (csrc/outlier.cu), in plain numpy.

Every squared distance is formed as the kernels form it, `(dx*dx + dy*dy) + dz*dz` in f32 with each subtraction,
product and sum rounded on its own (numpy's float32 ufuncs do exactly that; no FMA, no flush-to-zero), and every query
is compared with every point.  Rows are ordered by (distance, original index), so the result is the one answer any
exact search with the smaller-index tie rule must return.  Nothing here shares code or pruning logic with the CUDA index
or with the oracle's kd-tree.
"""
import numpy as np

_CHUNK_ELEMS = 1 << 24  # query x point distances per block: 64 MB of f32


def _xyz(a):
    a = np.asarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] >= 3
    return np.ascontiguousarray(a[:, 0]), np.ascontiguousarray(a[:, 1]), np.ascontiguousarray(a[:, 2])


def _d2_blocks(pts, queries):
    """Yields (first query, f32 squared distances of a block of queries to every point)."""
    px, py, pz = _xyz(pts)
    qx, qy, qz = _xyz(queries)
    n, m = px.shape[0], qx.shape[0]
    step = max(1, _CHUNK_ELEMS // max(n, 1))
    with np.errstate(over="ignore"):  # squares of huge coordinates overflow to +inf, as on the GPU
        for s in range(0, m, step):
            e = min(m, s + step)
            dx = np.subtract(qx[s:e, None], px[None, :])
            d2 = np.multiply(dx, dx)
            dy = np.subtract(qy[s:e, None], py[None, :], out=dx)
            d2 += np.multiply(dy, dy)
            dz = np.subtract(qz[s:e, None], pz[None, :], out=dx)
            d2 += np.multiply(dz, dz)
            yield s, d2


def bf_knn(pts, queries, k, farthest=False):
    """The k nearest points of every query: (idx (m, k) int32, d2 (m, k) f32), ascending by (d2, index).  Rows of a
    cloud with fewer than k points end with idx -1 / d2 0.0, as nn_knn_kernel writes them.  farthest=True also returns
    the index of a point at the largest distance from each query."""
    n, m = len(pts), len(queries)
    idx = np.full((m, k), -1, np.int32)
    d2o = np.zeros((m, k), np.float32)
    far = np.zeros(m, np.int64)
    kk = min(k, n)
    if kk > 0:
        for s, d2 in _d2_blocks(pts, queries):
            rows = d2.shape[0]
            if farthest:
                far[s:s + rows] = np.argmax(d2, axis=1)
            # every point at or below the kk-th smallest distance is a candidate (ties at the boundary included) ...
            kth = np.partition(d2, kk - 1, axis=1)[:, kk - 1:kk]
            r, c = np.nonzero(d2 <= kth)
            dc = d2[r, c]
            # ... ordered by (row, distance, index); the first kk of each row are its neighbours
            order = np.lexsort((c, dc, r))
            r, c, dc = r[order], c[order], dc[order]
            start = np.searchsorted(r, np.arange(rows))
            take = (start[:, None] + np.arange(kk)[None, :]).ravel()
            idx[s:s + rows, :kk] = c[take].reshape(rows, kk)
            d2o[s:s + rows, :kk] = dc[take].reshape(rows, kk)
    return (idx, d2o, far) if farthest else (idx, d2o)


def sor_distances_from_knn(idx, d2, mean_k):
    """distances[i] of pcl::StatisticalOutlierRemoval (outlier.cu) from rows of at least mean_k + 1 neighbours of each
    point in its own cloud: entries 1 .. mean_k, f32 square roots summed in f64 in neighbour order, divided by mean_k
    and rounded to f32.  Missing neighbours (a cloud of at most mean_k points) add nothing."""
    r = np.where(idx[:, 1:mean_k + 1] >= 0, np.sqrt(d2[:, 1:mean_k + 1]), np.float32(0.0))
    s = np.zeros(idx.shape[0], np.float64)
    for j in range(mean_k):
        s = s + r[:, j].astype(np.float64)
    return (s / mean_k).astype(np.float32)


def bf_sor_distances(pts, mean_k):
    """distances of pcl::StatisticalOutlierRemoval for every point of the cloud (see sor_distances_from_knn)."""
    idx, d2 = bf_knn(pts, pts, mean_k + 1)
    return sor_distances_from_knn(idx, d2, mean_k)


def sor_threshold(distances, std_mul):
    """mean + std_mul * sample standard deviation of the distances, summed serially in index order in f64 (the squares
    are f32), as outlier.cpp does."""
    d = np.asarray(distances, np.float32)
    n = float(d.size)
    total = float(np.cumsum(d.astype(np.float64))[-1])
    sq = float(np.cumsum((d * d).astype(np.float64))[-1])
    with np.errstate(invalid="ignore", divide="ignore"):
        var = np.float64(sq - total * total / n) / np.float64(n - 1.0)
        return total / n + std_mul * float(np.sqrt(var))


def transform_pcl(T, pts):
    """The f32 point transform of common.cuh (transform_pcl): x' = T00 x + (T01 y + (T02 z + T03)) with every product
    and sum rounded to f32.  T is a 4x4 matrix (row-major numpy, as getFinalTransformation returns it).  Returns (n, 4)
    with the input's fourth column."""
    T = np.asarray(T, np.float32).reshape(4, 4)
    x, y, z = _xyz(pts)
    out = np.zeros((len(x), 4), np.float32)
    for r in range(3):
        out[:, r] = T[r, 0] * x + (T[r, 1] * y + (T[r, 2] * z + T[r, 3]))
    if np.asarray(pts).shape[1] >= 4:
        out[:, 3] = np.asarray(pts, np.float32)[:, 3]
    return out


# ---- clouds full of ties ------------------------------------------------------------------------------------------

def cloud(xyz):
    """(n, 4) f32 cloud with intensity 0 from (n, 3) coordinates."""
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    return np.concatenate([xyz, np.zeros((len(xyz), 1), np.float32)], axis=1)


def lattice(shape, rng, spacing=1.0):
    """Integer lattice of shape (nx, ny, nz) in a random order, so that the original index of a point says nothing about
    where it is (the tie rule then matters at every equidistant neighbour)."""
    g = np.stack(np.meshgrid(*[np.arange(s, dtype=np.float32) for s in shape], indexing="ij"), axis=-1).reshape(-1, 3)
    return cloud(g[rng.permutation(len(g))] * np.float32(spacing))


def lattice_queries(shape, rng, m, spacing=1.0):
    """m queries on an integer lattice: a third on lattice points, a third at cell centres (8 equidistant neighbours) and
    a third at face centres (4 equidistant neighbours)."""
    hi = np.asarray(shape, np.float32) - 1
    a = rng.integers(0, np.asarray(shape), (m, 3)).astype(np.float32)
    c = np.minimum(rng.integers(0, np.asarray(shape), (m, 3)), hi - 1).astype(np.float32) + np.float32(0.5)
    f = c.copy()
    f[np.arange(m), rng.integers(0, 3, m)] -= np.float32(0.5)
    q = np.concatenate([a[: m // 3], c[: m // 3], f[: m - 2 * (m // 3)]])
    return cloud(q * np.float32(spacing))
