"""The small dense solvers of csrc/math.cuh and csrc/ndt_opt.cuh, compiled for the host (tests/linalg_check.cpp), equal the
oracle's Eigen restatement (oracle/linalg.hpp) bit for bit on the edge corpus of tests/linalg_corpus.py; and the oracle
itself is checked against numpy / LAPACK, so that a wrong oracle can neither pass nor fail the GPU comparisons
(tests/test_gpu_linalg.py).  No GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import linalg_corpus as corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = np.finfo(np.float64).eps
SVD3, EIG3, INV3, SVD_SOLVE6, SCHUR6, NEWTON6, SVD3_F32, LDLT6 = 0, 1, 2, 3, 4, 5, 16, 17
SHAPES = {0: (9, 21), 1: (9, 13), 2: (9, 9), 3: (42, 6), 4: (42, 7), 5: (42, 12), 16: (9, 21), 17: (42, 6)}


def build_host_linalg(tmp_dir):
    """tests/linalg_check.cpp as a ctypes library in tmp_dir: the header's solvers as the host compiles them."""
    so = os.path.join(str(tmp_dir), "liblinalg_check.so")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared",
                           "-I" + os.path.join(ROOT, "lidar_graph_slam_b200", "csrc"), os.path.join(ROOT, "tests", "linalg_check.cpp"),
                           "-o", so])
    L = C.CDLL(so)
    L.linalg_check_batch.restype = C.c_int
    L.linalg_check_batch.argtypes = [C.c_int, C.c_long, C.c_void_p, C.c_void_p]

    def run(op, inputs):
        nin, nout = SHAPES[op]
        a = np.ascontiguousarray(inputs, dtype=np.float64).reshape(-1, nin)
        out = np.empty((a.shape[0], nout))
        assert L.linalg_check_batch(op, a.shape[0], a.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)) == 0
        return out
    return run


def bits(a):
    """f64 bit patterns with every NaN made the same NaN: equal bits means equal values, equal signs of zero and NaN in the
    same places (not the same payloads)."""
    a = np.array(a, dtype=np.float64, copy=True)
    a[np.isnan(a)] = np.nan
    return a.view(np.uint64)


def assert_same_bits(got, want, names, what):
    diff = np.any(bits(got) != bits(want), axis=1)
    if diff.any():
        i = np.flatnonzero(diff)
        fams = sorted(set(names[i]))
        k = i[0]
        raise AssertionError("%s: %d of %d problems differ (families %s); first #%d:\n got  %s\n want %s" %
                             (what, i.size, len(diff), fams, k, got[k].tolist(), want[k].tolist()))


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return build_host_linalg(tmp_path_factory.mktemp("linalg"))


@pytest.fixture(scope="module")
def m3():
    return corpus.stack(corpus.mats3())


@pytest.fixture(scope="module")
def m3f():
    return corpus.stack(corpus.mats3_f32())


@pytest.fixture(scope="module")
def s6():
    return corpus.stack(corpus.systems6())


# ---- host-compiled header == oracle, bit for bit ----------------------------------------------------------------------
@pytest.mark.parametrize("op", [SVD3, EIG3, INV3])
def test_header_3x3_equals_oracle_bitwise(oracle, host, m3, op):
    A, names = m3
    with np.errstate(all="ignore"):
        assert_same_bits(host(op, A), oracle.linalg_batch(op, A), names, "op %d" % op)


def test_header_svd3_f32_equals_oracle_bitwise(oracle, host, m3f):
    A, names = m3f
    assert_same_bits(host(SVD3_F32, A), oracle.linalg_batch(oracle.LINALG_SVD3_F32, A), names, "svd_jacobi<3, float>")


@pytest.mark.parametrize("op", [SVD_SOLVE6, LDLT6])
def test_header_6x6_equals_oracle_bitwise(oracle, host, s6, op):
    X, names = s6
    with np.errstate(all="ignore"):
        assert_same_bits(host(op, X), oracle.linalg_batch(op, X), names, "op %d" % op)


def test_newton_step_rule(oracle, host, s6):
    """Machine::solve: the Schur step when schur_solve6 accepts, otherwise the JacobiSVD solve - the oracle's bits; with the
    exact Newton step always the JacobiSVD solve."""
    X, names = s6
    sch, nw, svd = host(SCHUR6, X), host(NEWTON6, X), oracle.linalg_batch(SVD_SOLVE6, X)
    acc = sch[:, 6] == 1.0
    assert set(np.unique(sch[:, 6])) <= {0.0, 1.0}
    assert_same_bits(nw[acc, :6], sch[acc, :6], names[acc], "Newton step = Schur step where accepted")
    assert_same_bits(nw[~acc, :6], svd[~acc], names[~acc], "Newton step = JacobiSVD where declined")
    assert_same_bits(nw[:, 6:], svd, names, "exact Newton step = JacobiSVD")


def test_sign_of_zero_singular_values(oracle, host):
    """svd_jacobi's |.| clears the sign bit like std::fabs: exact zeros come back as +0.0 (a compare-and-negate returns -0.0
    for -0.0 and differs from Eigen)."""
    A = np.array([[0.0, -0.0, 0.0, -0.0, 0.0, 0.0, 0.0, 0.0, -0.0],
                  [1.0, 0.0, 0.0, 0.0, -0.0, 0.0, 0.0, 0.0, 0.0],
                  [-0.0, 0.0, 0.0, 0.0, 2.0, -0.0, 0.0, -0.0, -0.0],
                  [-2.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, -0.0, 0.0]])
    for op in (SVD3, SVD3_F32):
        S = host(op, A)[:, 9:12]
        assert not np.signbit(S).any(), S
        assert_same_bits(host(op, A), oracle.linalg_batch(op, A), np.array(["signed_zero"] * 4), "op %d" % op)


# ---- the oracle against numpy / LAPACK ----------------------------------------------------------------------------------
def _finite_moderate(X, k=9):
    nrm = np.abs(X[:, :k]).max(axis=1)
    return np.isfinite(X).all(axis=1) & (nrm > 2.0 ** -900) & (nrm < 2.0 ** 900)


def test_oracle_svd3_against_lapack(oracle, m3):
    A, names = m3
    out = oracle.linalg_batch(SVD3, A)
    U, S, V = out[:, :9].reshape(-1, 3, 3), out[:, 9:12], out[:, 12:].reshape(-1, 3, 3)
    fin = np.isfinite(A).all(axis=1)
    # sorted descending, never -0.0, on every finite input (subnormal and huge included)
    assert (np.diff(S[fin], axis=1) <= 0).all()
    assert not np.signbit(S[fin]).any()
    sel = _finite_moderate(A)
    A3 = A[sel].reshape(-1, 3, 3)
    nrm = np.abs(A3).max(axis=(1, 2))
    s_ref = np.linalg.svd(A3, compute_uv=False)
    assert (np.abs(S[sel] - s_ref).max(axis=1) <= 16 * EPS * nrm).all()
    ld = np.longdouble
    I = np.eye(3, dtype=ld)
    for M in (U[sel], V[sel]):
        Ml = M.astype(ld)
        assert (np.abs(np.einsum("nki,nkj->nij", Ml, Ml) - I).max(axis=(1, 2)) <= 16 * EPS).all()
    R = np.einsum("nik,nk,njk->nij", U[sel].astype(ld), S[sel].astype(ld), V[sel].astype(ld)) - A3.astype(ld)
    assert (np.abs(R).max(axis=(1, 2)) <= 32 * EPS * nrm).all()


def test_oracle_eig3_against_lapack(oracle, m3):
    A, names = m3
    out = oracle.linalg_batch(EIG3, A)
    w, Q, ok = out[:, :3], out[:, 3:12].reshape(-1, 3, 3), out[:, 12]
    sel = _finite_moderate(A) & (ok == 1.0)
    assert ok[_finite_moderate(A)].all()  # the QR iteration converges on every finite input
    L = np.tril(A[sel].reshape(-1, 3, 3))
    Asym = L + np.transpose(np.tril(L, -1), (0, 2, 1))  # the lower triangle is what is read
    nrm = np.abs(Asym).max(axis=(1, 2))
    assert (np.diff(w[sel], axis=1) >= 0).all()
    w_ref = np.linalg.eigvalsh(Asym, UPLO="L")
    assert (np.abs(w[sel] - w_ref).max(axis=1) <= 32 * EPS * nrm).all()
    ld = np.longdouble
    Ql = Q[sel].astype(ld)
    assert (np.abs(np.einsum("nki,nkj->nij", Ql, Ql) - np.eye(3, dtype=ld)).max(axis=(1, 2)) <= 16 * EPS).all()
    R = np.einsum("nij,njk->nik", Asym.astype(ld), Ql) - Ql * w[sel].astype(ld)[:, None, :]
    assert (np.abs(R).max(axis=(1, 2)) <= 32 * EPS * nrm).all()


def _pinv_solve(H, b, rank_thr_rel):
    U, s, Vt = np.linalg.svd(H)
    keep = s >= rank_thr_rel * s[0]
    t = (U.T @ b)[keep] / s[keep]
    return Vt[keep].T @ t, s


def test_oracle_svd_solve6_is_the_min_norm_pinv_solution(oracle, s6):
    """jacobi_svd_solve<6> = V diag(1/S) U^T b over the singular values >= 6 eps sigma_max (Eigen's default threshold)."""
    X, names = s6
    x = oracle.linalg_batch(SVD_SOLVE6, X)
    sel = _finite_moderate(X, 42) & (names != "rank_threshold")
    checked = 0
    for i in np.flatnonzero(sel):
        H, b = X[i, :36].reshape(6, 6), X[i, 36:]
        ref, s = _pinv_solve(H, b, 6 * EPS)
        thr = 6 * EPS * s[0]
        if s[0] == 0 or np.any(np.abs(s - thr) <= 8 * EPS * s[0]):
            continue  # LAPACK and Jacobi may round across the threshold
        r = np.count_nonzero(s >= thr)
        cond_r = s[0] / s[r - 1]
        assert np.abs(x[i] - ref).max() <= 1e3 * EPS * cond_r * max(np.abs(ref).max(), 1e-300), (names[i], x[i], ref)
        checked += 1
    assert checked > 8000


def test_oracle_svd_solve6_rank_threshold_exact(oracle, s6):
    """Block-diagonal systems whose smallest singular value sits at 6 eps sigma_max (1 +- 2^-20), on it and one ulp either
    side: exactly representable, so the rank decision is known - kept when >= the threshold, dropped (x = 0 there) below."""
    X, names = s6
    T = X[names == "rank_threshold"]
    x = oracle.linalg_batch(SVD_SOLVE6, T)
    seen = set()
    for i in range(T.shape[0]):
        H, b = T[i, :36].reshape(6, 6), T[i, 36:]
        d = np.abs(np.diag(H))
        smax = d.max()
        iso = [j for j in range(6) if np.count_nonzero(H[j]) <= 1 and d[j] < smax * 1e-3]
        assert len(iso) == 1
        p = iso[0]
        small, thr = d[p], 6 * EPS * smax
        if small >= thr:
            assert x[i, p] == pytest.approx(b[p] / H[p, p], rel=1e-12)
            seen.add("kept")
        else:
            assert x[i, p] == 0.0
            seen.add("dropped")
        others = [j for j in range(6) if j != p]
        ref = np.linalg.solve(H[np.ix_(others, others)], b[others])
        np.testing.assert_allclose(x[i, others], ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())
    assert seen == {"kept", "dropped"}


def test_schur_step_against_svd_and_its_refusals(host, oracle, s6):
    """schur_solve6: whenever it accepts a system of full rank at Eigen's threshold, its step is finite and within
    cond * 1e-15 of the JacobiSVD solution.  It declines every singular system, and every system its refinement finds
    too ill-conditioned: all of the condition sweep (H = Q diag(s) Q^T, dense Q) beyond cond(H) = 1e9.  (Its rules measure
    cancellation: a block-diagonal H whose smallest singular value lies below 6 eps sigma_max loses no digits in the
    elimination and is accepted, where the reference's JacobiSVD drops that direction.)"""
    X, names = s6
    with np.errstate(all="ignore"):
        sch = host(SCHUR6, X)
    acc = sch[:, 6] == 1.0
    assert np.isfinite(sch[acc, :6]).all()
    svd = oracle.linalg_batch(SVD_SOLVE6, X)
    fin = np.isfinite(X).all(axis=1)
    n_acc = 0
    for i in np.flatnonzero(fin):
        H = X[i, :36].reshape(6, 6)
        s = np.linalg.svd(H, compute_uv=False)
        cond = s[0] / s[5] if s[5] > 0 else np.inf
        if names[i] in ("rank5_rank4", "dependent_columns", "zero_matrix") or s[5] == 0:
            assert not acc[i], (names[i], cond)
        if names[i] == "condition_sweep" and cond > 1e9:
            assert not acc[i], (names[i], cond)
        if acc[i] and s[5] >= 8 * EPS * s[0]:
            n_acc += 1
            scale = np.abs(svd[i]).max()
            assert np.abs(sch[i, :6] - svd[i]).max() <= max(cond, 1.0) * 1e-15 * scale, (names[i], cond)
    assert n_acc > 5000 and (~acc[fin]).sum() > 2000
    assert not acc[~fin].any()
