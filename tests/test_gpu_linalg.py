"""The device's small dense solvers (csrc/math.cuh, csrc/ndt_opt.cuh) equal the oracle's Eigen restatement bit for bit.

* lgs_linalg_batch runs SVD3 / EIG3 / INV3 / SVD_SOLVE6 one problem per thread over the edge corpus of
  tests/linalg_corpus.py (>= 10^5 problems); SCHUR6 / NEWTON6 equal the host-compiled header (tests/linalg_check.cpp).
* The covariance builds that call them - FastGICP under every regularisation, pclomp GICP, the NDT voxel statistics - are
  compared bitwise with the oracle on the Velodyne pair and on degenerate clouds: duplicates, collinear, planar, a lattice,
  a 1e4 m offset, subnormal coordinates, and voxels holding 1 to 300 members (the 32-member chunks of voxel_sums_kernel).
  The looser end-to-end tests in test_gpu_parity.py keep their own bars."""
import ctypes as C

import numpy as np
import pytest

import linalg_corpus as corpus
from test_linalg_reference import assert_same_bits, bits, build_host_linalg

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return build_host_linalg(tmp_path_factory.mktemp("linalg_gpu"))


@pytest.fixture(scope="module")
def m3():
    return corpus.stack(corpus.mats3())


@pytest.fixture(scope="module")
def s6():
    return corpus.stack(corpus.systems6())


# ---- the solvers themselves ----------------------------------------------------------------------------------------
def test_device_solvers_equal_oracle_bitwise(api, oracle, m3, s6):
    A, n3 = m3
    X, n6 = s6
    total = 0
    for op in (api.LINALG_SVD3, api.LINALG_EIG3, api.LINALG_INV3):
        with np.errstate(all="ignore"):
            assert_same_bits(api.linalg_batch(op, A), oracle.linalg_batch(op, A), n3, "device op %d" % op)
        total += A.shape[0]
    assert_same_bits(api.linalg_batch(api.LINALG_SVD_SOLVE6, X), oracle.linalg_batch(oracle.LINALG_SVD_SOLVE6, X), n6, "device svd_solve<6>")
    total += X.shape[0]
    assert total >= 100000
    # the zero-sign fix: no -0.0 singular value anywhere on finite inputs
    S = api.linalg_batch(api.LINALG_SVD3, A)[:, 9:12]
    assert not np.signbit(S[np.isfinite(A).all(axis=1)]).any()


def test_device_eig3_reads_the_lower_triangle(api, m3):
    A, _ = m3
    A = A[np.isfinite(A).all(axis=1)][:20000].reshape(-1, 3, 3)
    iu = np.triu_indices(3, 1)
    garbage, sym = A.copy(), A.copy()  # written entry by entry: the lower triangle keeps its signed zeros
    garbage[:, iu[0], iu[1]] = np.random.default_rng(5).normal(size=(len(A), 3))
    sym[:, iu[0], iu[1]] = A[:, iu[1], iu[0]]
    outs = [api.linalg_batch(api.LINALG_EIG3, M.reshape(-1, 9)) for M in (A, garbage, sym)]
    assert np.array_equal(bits(outs[0]), bits(outs[1])) and np.array_equal(bits(outs[0]), bits(outs[2]))


def test_device_schur_and_newton_steps_equal_host(api, host, s6):
    X, names = s6
    with np.errstate(all="ignore"):
        for op in (api.LINALG_SCHUR6, api.LINALG_NEWTON6):
            assert_same_bits(api.linalg_batch(op, X), host(op, X), names, "device op %d" % op)
    acc = api.linalg_batch(api.LINALG_SCHUR6, X)[:, 6]
    assert 0 < acc.sum() < acc.size  # both branches of the Newton step are taken


def test_linalg_batch_refuses_bad_arguments(api):
    ctx = api.default_context()
    L = ctx._L
    a, o = np.zeros(42), np.zeros(21)
    pa, po = a.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p)
    before = ctx.launch_count
    for op, n, x, y in ((-1, 1, pa, po), (6, 1, pa, po), (0, -1, pa, po), (0, 1, None, po), (0, 1, pa, None)):
        assert L.lgs_linalg_batch(ctx._h, op, n, x, y) == -1  # LGS_ERR_INVALID
    assert L.lgs_linalg_batch(ctx._h, 0, 0, None, None) == 0
    assert ctx.launch_count == before
    with pytest.raises(ValueError):
        api.linalg_batch(7, a)


# ---- the covariance builds, bitwise ---------------------------------------------------------------------------------
def _clouds(velodyne_pair, oracle):
    rng = np.random.default_rng(11)
    v = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    out = {"velodyne": v}

    def pts(xyz):
        xyz = np.asarray(xyz, np.float32)
        return np.c_[xyz, np.zeros(len(xyz), np.float32)].astype(np.float32)
    base = rng.uniform(-5, 5, size=(400, 3))
    out["duplicates"] = pts(np.repeat(base[:60], 7, axis=0)[rng.permutation(420)])
    out["collinear"] = pts(rng.uniform(-8, 8, size=(500, 1)) * np.array([0.6, -0.3, 0.74]) + [1.0, 2.0, -0.5])
    out["planar"] = pts(np.c_[rng.uniform(-6, 6, size=(600, 2)), np.full(600, 0.75)])
    g = np.arange(-4, 4, 0.5)
    out["lattice"] = pts(np.stack(np.meshgrid(g, g, g[:6]), -1).reshape(-1, 3)[rng.permutation(16 * 16 * 6)])
    out["offset_1e4"] = pts(v[:3000, :3].astype(np.float64) + [1e4, -1e4, 12.0])
    out["subnormal"] = pts(rng.uniform(-1, 1, size=(300, 3)) * 1e-42)
    return out


def _voxel_cloud(rng, offset=0.0):
    """Voxels of resolution 1 holding 1..300 members (every count up to 40, the 32-member chunk edges 63-65 and 95-97, and
    a few large ones), points well inside their cells; some voxels are planar, collinear or a repeated point."""
    counts = list(range(1, 41)) + [63, 64, 65, 95, 96, 97, 128, 200, 300]
    pts = []
    for i, c in enumerate(counts):
        for kind in range(4):
            cell = np.array([i, kind * 2, (i * 7) % 5], np.float64)
            q = rng.uniform(0.05, 0.95, size=(c, 3))
            if kind == 1:
                q[:, 2] = 0.5
            elif kind == 2:
                q = 0.1 + rng.uniform(0, 0.8, size=(c, 1)) * np.array([[1.0, 0.5, 0.25]])
            elif kind == 3:
                q = np.repeat(q[:1], c, axis=0)
            pts.append(cell + q + offset)
    p = np.concatenate(pts)
    p = p[rng.permutation(len(p))].astype(np.float32)
    return np.c_[p, np.zeros(len(p), np.float32)].astype(np.float32), counts


def _cov_bits_equal(got, want, what):
    assert len(got) == len(want), what
    if len(got) == 0:
        return
    got, want = np.asarray(got).reshape(len(got), -1), np.asarray(want).reshape(len(want), -1)
    assert got.shape == want.shape, what
    assert_same_bits(got, want, np.array([what] * len(got)), what)


@pytest.mark.parametrize("reg", [0, 1, 2, 3, 4])
def test_fast_gicp_covariances_bitwise(api, oracle, velodyne_pair, reg):
    clouds = _clouds(velodyne_pair, oracle)
    for name, c in clouds.items():
        for k in (20,) if name != "duplicates" else (5, 20):
            g, o = api.FastGICP(), oracle.FastGICP()
            for x in (g, o):
                x.setRegularizationMethod(reg)
                x.setCorrespondenceRandomness(k)
                x.setInputSource(c)
                x.setInputTarget(c[: max(len(c) // 2, 1)])
            for which in (0, 1):
                _cov_bits_equal(g.covariances(which), o.covariances(which), "%s k=%d reg=%d which=%d" % (name, k, reg, which))


def test_fast_gicp_covariances_k_above_n_bitwise(api, oracle):
    rng = np.random.default_rng(3)
    for n in (1, 2, 5, 12, 19):
        c = np.c_[rng.uniform(-1, 1, size=(n, 3)), np.zeros(n)].astype(np.float32)
        for reg in (1, 3):
            g, o = api.FastGICP(), oracle.FastGICP()
            for x in (g, o):
                x.setRegularizationMethod(reg)
                x.setCorrespondenceRandomness(20)
                x.setInputSource(c)
                x.setInputTarget(c)
            _cov_bits_equal(g.covariances(0), o.covariances(0), "n=%d k=20 reg=%d" % (n, reg))


def test_pclomp_gicp_covariances_bitwise(api, oracle, velodyne_pair):
    for name, c in _clouds(velodyne_pair, oracle).items():
        g, o = api.GeneralizedIterativeClosestPoint(), oracle.GeneralizedIterativeClosestPoint()
        for x in (g, o):
            x.setInputSource(c)
            x.setInputTarget(c[: max(len(c) // 2, 1)])
        for which in (0, 1):
            _cov_bits_equal(g.covariances(which), o.covariances(which), "%s which=%d" % (name, which))


def _ndt_voxels_bitwise(api, oracle, tgt, res, what):
    g, o = api.NormalDistributionsTransform(), oracle.NDT()
    for x in (g, o):
        x.setResolution(res)
        x.setInputTarget(tgt)
        x.setInputSource(tgt[:10])
    vg, vo = g.export_voxels(), o.export_voxels()
    assert np.array_equal(vg["idx"], vo["idx"]), what
    assert np.array_equal(vg["n"], vo["n"]), what
    _cov_bits_equal(vg["mean"], vo["mean"], what + " mean")
    valid = vo["n"] >= 6
    for key in ("cov", "icov"):
        _cov_bits_equal(vg[key][valid], vo[key][valid], "%s %s" % (what, key))
    return vo


def test_ndt_voxel_statistics_bitwise(api, oracle, velodyne_pair):
    td = oracle.voxel_grid(velodyne_pair["target"], 0.1)["points"]
    for res in (1.0, 0.5, 2.0):
        _ndt_voxels_bitwise(api, oracle, td, res, "velodyne res=%g" % res)
    for name, c in _clouds(velodyne_pair, oracle).items():
        _ndt_voxels_bitwise(api, oracle, c, 1.0, name)
    rng = np.random.default_rng(17)
    for off in (0.0, 1e4):
        cloud, counts = _voxel_cloud(rng, off)
        vo = _ndt_voxels_bitwise(api, oracle, cloud, 1.0, "member counts offset=%g" % off)
        n = vo["n"]
        assert {1, 2, 3, 4, 5} <= set(n.tolist()) and (n == -1).any() and (n >= 6).any()
