"""Deterministic edge corpus for the small dense solvers of csrc/math.cuh and csrc/ndt_opt.cuh (svd_jacobi, eig_sym3,
inv3, svd_solve<6>, schur_solve6, ldlt_solve6).  Every family aims at a place where these routines branch or lose
digits; each function returns (name, array) blocks so that a failing comparison can name its family.

    mats3(seed)        (n, 9) row-major 3x3 inputs for SVD3 / EIG3 / INV3
    mats3_f32(seed)    the same families at float-representable values and scales, for svd_jacobi<3, float>
    systems6(seed)     (n, 42) = H row-major + b for the 6x6 solvers
"""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EPS = np.finfo(np.float64).eps


def _rot(rng):
    q, r = np.linalg.qr(rng.normal(size=(3, 3)))
    return q * np.sign(np.diag(r))


def _neighbourhood_covs(pts, k, offset=0.0):
    """Single-pass covariances of the k nearest neighbours of every point (sum x x^T / k - mean mean^T), as the GICP and
    NDT kernels form them: at a large offset the cancellation leaves slightly negative eigenvalues."""
    from scipy.spatial import cKDTree
    p = pts[:, :3].astype(np.float64) + offset
    _, nb = cKDTree(p).query(p, k=k)
    q = p[nb]
    mean = q.mean(axis=1)
    s = np.einsum("nki,nkj->nij", q, q) / k
    return (s - mean[:, :, None] * mean[:, None, :]).reshape(-1, 9)


def _threshold_block(rng, n, eps, dtype):
    """Off-diagonal entries at svd_jacobi's rotation threshold 2 eps max_diag, and one ulp either side: max |A| = 1 on the
    diagonal, so the scaled matrix is A itself and the threshold is exactly 2 eps."""
    out = []
    for t in range(n):
        d = rng.uniform(0.25, 1.0, size=3).astype(dtype)
        d[t % 3] = 1.0
        d *= rng.choice([-1.0, 1.0], size=3).astype(dtype)
        A = np.diag(d).astype(dtype)
        thr = dtype(2) * dtype(eps)
        v = [np.nextafter(thr, dtype(0)), thr, np.nextafter(thr, dtype(1))][t % 3]
        v = v * dtype(rng.choice([-1.0, 1.0]))
        p, q = [(1, 0), (2, 0), (2, 1)][(t // 3) % 3]
        if (t // 9) % 2:
            p, q = q, p
        A[p, q] = v
        if (t // 18) % 2:  # the other entry of the pair below the threshold, or a second pair at it
            A[q, p] = v / dtype(4) if (t // 36) % 2 == 0 else dtype(0)
        out.append(A.astype(np.float64).ravel())
    return np.array(out)


def _families3(rng, f32=False):
    dt = np.float32 if f32 else np.float64
    n = 3000
    fam = []
    G = rng.normal(size=(n, 3, 3))
    fam.append(("random", G.reshape(-1, 9)))
    # integer-valued with signed zeros: rounding small negatives gives -0.0, plus explicit -0.0 entries
    I = np.round(rng.normal(scale=1.5, size=(n, 3, 3)))
    I[rng.random(size=I.shape) < 0.3] = -0.0
    fam.append(("integer_signed_zero", I.reshape(-1, 9)))
    fam.append(("zero_and_negative_zero", np.array([np.zeros(9), -np.zeros(9), np.where(np.arange(9) % 2, -0.0, 0.0)])))
    # diagonal (signed, with zeros) and signed permutation matrices: no rotation at all
    D = np.zeros((n, 3, 3))
    dv = rng.normal(size=(n, 3)) * (rng.random(size=(n, 3)) > 0.2)
    D[:, [0, 1, 2], [0, 1, 2]] = dv
    D[rng.random(size=D.shape) < 0.2] *= -1.0
    D[:, [0, 0, 1, 1, 2, 2], [1, 2, 0, 2, 0, 1]] = np.where(rng.random(size=(n, 6)) < 0.5, -0.0, 0.0)
    fam.append(("diagonal", D.reshape(-1, 9)))
    perms = [np.eye(3)[list(p)] for p in ((0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0))]
    P = np.array([perms[t % 6] * rng.choice([-1.0, 1.0, 2.0, 0.5], size=3) for t in range(600)])
    fam.append(("permutation", P.reshape(-1, 9)))
    fam.append(("rotation_threshold", _threshold_block(rng, 720, np.finfo(dt).eps, dt)))
    # rank 1 and rank 2 symmetric
    u, v = rng.normal(size=(n, 3)), rng.normal(size=(n, 3))
    fam.append(("rank1_sym", (u[:, :, None] * u[:, None, :]).reshape(-1, 9)))
    fam.append(("rank2_sym", (u[:, :, None] * u[:, None, :] + v[:, :, None] * v[:, None, :]).reshape(-1, 9)))
    fam.append(("rank1_general", (u[:, :, None] * v[:, None, :]).reshape(-1, 9)))
    # repeated eigenvalues: 2+1 and triple, exact (diagonal) and rotated (rounded)
    rep = []
    for t in range(1500):
        a, b = rng.normal(), rng.normal()
        w = [(a, a, b), (b, a, a), (a, a, a), (a, a, 0.0), (0.0, 0.0, a)][t % 5]
        R = _rot(rng) if t % 2 else np.eye(3)
        rep.append((R * np.array(w)) @ R.T)
    fam.append(("repeated_eigenvalues", np.array(rep).reshape(-1, 9)))
    # symmetric positive semi-definite with random spectrum spread (covariance-like)
    S = []
    for t in range(n):
        R = _rot(rng)
        w = np.exp(rng.uniform(-40, 5, size=3)) if t % 2 else rng.uniform(0, 1, size=3)
        S.append((R * w) @ R.T)
    fam.append(("spd_spread", np.array(S).reshape(-1, 9)))
    # real covariance shapes: k = 20 neighbourhoods of the Velodyne scan, planar and collinear ones, 1e4 m away
    z = np.load(os.path.join(GOLDEN, "velodyne_pair.npz"))
    tgt = z["target"][rng.permutation(z["target"].shape[0])[:4000]]
    fam.append(("velodyne_k20", _neighbourhood_covs(tgt, 20)))
    fam.append(("velodyne_k20_offset_1e4", _neighbourhood_covs(tgt, 20, 1e4)))
    plane = np.c_[rng.uniform(-1, 1, size=(1500, 2)), np.zeros(1500)] @ _rot(rng).T
    line = rng.uniform(-1, 1, size=(1500, 1)) * rng.normal(size=3)
    for name, pts in (("planar", plane), ("collinear", line)):
        pts = pts.astype(np.float32)
        fam.append((name + "_k20", _neighbourhood_covs(pts, 20)))
        fam.append((name + "_k20_offset_1e4", _neighbourhood_covs(pts, 20, 1e4)))
    # non-symmetric (EIG3 reads the lower triangle only)
    fam.append(("nonsymmetric", rng.normal(size=(n, 9))))
    base = np.concatenate([b for _, b in fam])
    # scales: subnormal to huge powers of two (exact), and rows 1e150 apart
    if f32:
        exps = np.arange(-140, 120, 7)
    else:
        exps = np.concatenate([[-1070, -1060, -1040, -1022, -1000], np.arange(-900, 901, 60), [960, 990, 1000]])
    pick = base[rng.integers(0, base.shape[0], size=(exps.size, 120))]
    fam.append(("power_of_two_scales", (pick * np.ldexp(1.0, exps)[:, None, None]).reshape(-1, 9)))
    if not f32:
        R = base[rng.integers(0, base.shape[0], size=600)].reshape(-1, 3, 3)
        rs = np.array([[1e-150, 1.0, 1e150], [1e150, 1.0, 1e-150], [1.0, 1e150, 1e150], [1e-150, 1e-150, 1.0]])
        fam.append(("rows_1e150_apart", (R * rs[np.arange(600) % 4][:, :, None]).reshape(-1, 9)))
    # NaN and Inf entries: bounded loops, no fault
    bad = base[rng.integers(0, base.shape[0], size=400)].copy()
    for t in range(400):
        bad[t, rng.integers(0, 9, size=1 + t % 3)] = [np.nan, np.inf, -np.inf][t % 3]
    fam.append(("nan_inf", bad))
    out = []
    for name, a in fam:
        a = np.asarray(a, np.float64)
        if f32:
            with np.errstate(over="ignore"):
                a = a.astype(np.float32).astype(np.float64)
        out.append((name, a))
    return out


def mats3(seed=0):
    return _families3(np.random.default_rng(seed))


def mats3_f32(seed=0):
    return _families3(np.random.default_rng(seed + 1000), f32=True)


def schur_det_edge(rng, n):
    """Translation block [[1, 1, 0], [1, 1 + d, 0], [0, 0, 1]] (det d against products of magnitude 2 + d): d sweeps across
    mat3_adjugate's cancellation rule |det| > 1e-10 mag."""
    out = []
    for t in range(n):
        d = 2e-10 * np.exp(rng.uniform(-0.5, 0.5)) if t % 2 else 10.0 ** rng.uniform(-12, -7)
        A = np.array([[1.0, 1.0, 0.0], [1.0, 1.0 + d, 0.0], [0.0, 0.0, 1.0]])
        Q = np.eye(6)
        Q[:3, :3] = A
        D = rng.normal(size=(3, 3))
        Q[3:, 3:] = D @ D.T + 3 * np.eye(3)
        C = rng.normal(scale=0.01, size=(3, 3))
        Q[3:, :3], Q[:3, 3:] = C, C.T
        if t % 4 >= 2:  # the same edge in the Schur complement
            Q = Q[[3, 4, 5, 0, 1, 2]][:, [3, 4, 5, 0, 1, 2]]
            Q[:3, :3] += 10 * np.eye(3)
        out.append(np.concatenate([Q.ravel(), rng.normal(size=6)]))
    return np.array(out)


def _sym_with_spectrum(rng, s):
    Q, r = np.linalg.qr(rng.normal(size=(6, 6)))
    Q = Q * np.sign(np.diag(r))
    return (Q * s) @ Q.T


def systems6(seed=0):
    rng = np.random.default_rng(seed + 2000)
    fam = []
    n = 2500
    b = lambda m: rng.normal(size=(m, 6))
    fam.append(("random_general", np.c_[rng.normal(size=(n, 36)), b(n)]))
    # J^T J Hessians with translation and rotation columns 1e6 apart (and the other way round)
    H = []
    for t in range(n):
        J = rng.normal(size=(40, 6))
        J[:, 3:] *= 1e-3 if t % 2 else 1e3
        H.append((J.T @ J).ravel())
    fam.append(("jtj_blocks_1e6_apart", np.c_[np.array(H), b(n)]))
    # the NDT Hessian's two triangles differ by ~1e-8 relative
    Hn = np.array(H)[:1000].reshape(-1, 6, 6) * (1 + 1e-8 * rng.normal(size=(1000, 6, 6)))
    fam.append(("jtj_nonsymmetric_1e-8", np.c_[Hn.reshape(-1, 36), b(1000)]))
    I = []
    for t in range(n):
        M = rng.normal(size=(6, 6))
        I.append((M + M.T).ravel())
    fam.append(("indefinite", np.c_[np.array(I), b(n)]))
    # rank 5 and rank 4 (b in the range and b anywhere); an exactly dependent pair of columns
    R = []
    for t in range(n):
        k = 5 if t % 2 else 4
        J = rng.normal(size=(40, k)) @ rng.normal(size=(k, 6))
        R.append((J.T @ J).ravel())
    R = np.array(R)
    rb = b(n)
    rb[::2] = np.einsum("nij,nj->ni", R.reshape(-1, 6, 6), rng.normal(size=(n, 6)))[::2]
    fam.append(("rank5_rank4", np.c_[R, rb]))
    Dp = rng.normal(size=(600, 6, 6))
    Dp[:, :, 5] = Dp[:, :, 4]
    fam.append(("dependent_columns", np.c_[Dp.reshape(-1, 36), b(600)]))
    fam.append(("zero_matrix", np.c_[np.zeros((4, 36)), b(4)]))
    # singular values on Eigen's rank threshold 6 eps sigma_max: block-diagonal, the rotated 2x2 block and the exact diagonal
    # entries below sigma_max = 2^k keep the small singular value exact through the sweeps
    T = []
    for t in range(1200):
        k = int(rng.integers(-20, 20))
        smax = np.ldexp(1.0, k)
        thr = smax * 6 * EPS
        small = [thr * (1 - 2.0 ** -20), thr * (1 + 2.0 ** -20), thr, np.nextafter(thr, 0), np.nextafter(thr, np.inf), 0.0][t % 6]
        M = np.diag([smax, 0.0, 0.0, smax * 0.25, smax * 0.125, small])
        phi = rng.uniform(0, np.pi)
        c, s = np.cos(phi), np.sin(phi)
        Rt = np.array([[c, -s], [s, c]])
        M[1:3, 1:3] = Rt @ np.diag(smax * rng.uniform(0.3, 0.9, size=2)) @ Rt.T
        p = rng.permutation(6) if (t // 6) % 2 else np.arange(6)
        M = M[p][:, p]
        T.append(np.concatenate([M.ravel(), rng.normal(size=6)]))
    fam.append(("rank_threshold", np.array(T)))
    # cond(H) from 1e2 to 1e12 around the Schur refinement rule (n_dx <= 1e-20 n_x) and the determinant rule
    C = []
    for t in range(n):
        cond = 10.0 ** rng.uniform(2, 12)
        s = np.exp(rng.uniform(0, np.log(cond), size=6))
        s[0], s[1] = 1.0, cond
        s *= rng.choice([-1.0, 1.0], size=6) if t % 3 == 0 else 1.0
        C.append(_sym_with_spectrum(rng, s / cond).ravel())
    fam.append(("condition_sweep", np.c_[np.array(C), b(n)]))
    fam.append(("schur_determinant_edge", schur_det_edge(rng, 1200)))
    base = np.concatenate([a for _, a in fam])
    pick = base[rng.integers(0, base.shape[0], size=(12, 100))]
    exps = np.array([-1000, -600, -300, -100, -30, -10, 10, 30, 100, 300, 600, 900])
    sc = pick * np.ldexp(1.0, exps)[:, None, None]
    fam.append(("power_of_two_scales", sc.reshape(-1, 42)))
    bad = base[rng.integers(0, base.shape[0], size=300)].copy()
    for t in range(300):
        bad[t, rng.integers(0, 42 if t % 2 else 36, size=1 + t % 2)] = [np.nan, np.inf, -np.inf][t % 3]
    fam.append(("nan_inf", bad))
    return fam


def stack(families):
    return np.concatenate([a for _, a in families]), np.concatenate([[name] * len(a) for name, a in families])
