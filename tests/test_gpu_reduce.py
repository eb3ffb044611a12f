"""The last-CTA reduction behind every sum an evaluation returns (csrc/reduce.cuh) folds the per-CTA rows in the order it
states, bit for bit: group g of NG adds rows g, g + NG, g + 2 NG, ... in turn from 0.0, then the NG group sums are added in
group order from 0.0.  lgs_grid_fold_check runs the kernels' own grid finish, with each (K, NG) a kernel uses, over rows
whose sum depends on the order: magnitudes 1e16 with +-1, signed zeros, subnormals."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# (K sums, NG groups): NDT calculateScore, FastGICP compute_error and linearize, ICP, NDT derivatives modes 1, 2 and 0
CASES = [(1, 1), (1, 2), (43, 2), (17, 8), (8, 12), (22, 12), (44, 12)]
KINDS = ("cancel", "signed_zero", "subnormal", "mixed")


def fold(rows, ng):
    """The stated order, one Python float operation at a time."""
    G, K = rows.shape
    out = np.empty(K)
    for k in range(K):
        total = 0.0
        for g in range(ng):
            s = 0.0
            for b in range(g, G, ng):
                s += float(rows[b, k])
            total += s
        out[k] = total
    return out


def make_rows(kind, G, K, seed):
    rng = np.random.default_rng(seed)
    if kind == "cancel":  # 1e16 + 1 rounds: each order of the +-1 terms around the large ones keeps a different share of them
        return rng.choice([1e16, -1e16, 1.0, -1.0, 3.0, 0.5], size=(G, K))
    if kind == "signed_zero":  # column 0 all -0.0: every sum starts from +0.0, so it comes out +0.0
        r = rng.choice([0.0, -0.0, -0.0, 5e-324, -5e-324], size=(G, K))
        r[:, 0] = -0.0
        return r
    if kind == "subnormal":  # subnormals next to the smallest normals and to 1: no flush to zero, rounding at 1
        tiny = rng.integers(-2**40, 2**40, size=(G, K)) * 5e-324
        big = rng.choice([0.0, 2.2250738585072014e-308, -2.2250738585072014e-308, 1.0, -1.0], size=(G, K))
        return np.where(rng.random((G, K)) < 0.5, tiny, big)
    mag = 10.0 ** rng.uniform(-20, 20, size=(G, K))
    return rng.standard_normal((G, K)) * mag


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def grids(ng):
    return sorted({g for g in (1, ng - 1, ng, 148, 592) if g >= 1})


@pytest.mark.parametrize("K,ng", CASES)
def test_grid_fold_order_bitwise(api, K, ng):
    for G in grids(ng):
        for i, kind in enumerate(KINDS):
            rows = make_rows(kind, G, K, seed=1000 * G + 10 * K + i)
            got, want = api.grid_fold_check(rows, ng), fold(rows, ng)
            assert np.array_equal(bits(got), bits(want)), "K=%d NG=%d G=%d %s: %r != %r" % (K, ng, G, kind, got, want)


def test_grid_fold_rows_tell_the_orders_apart():
    """The rows above would catch a change of NG: at G = 592 every group count the kernels use gives other bits."""
    rows = make_rows("cancel", 592, 44, seed=7)
    sums = {ng: bits(fold(rows, ng)) for ng in (1, 2, 8, 12)}
    for a in sums:
        for b in sums:
            if a < b:
                assert not np.array_equal(sums[a], sums[b]), (a, b)


def test_grid_fold_check_refuses_bad_arguments(api):
    ctx = api.default_context()
    L = ctx._L
    rows, out = np.zeros(44 * 4), np.zeros(44)
    pr, po = rows.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)
    before = ctx.launch_count
    for G, K, ng, r, o in ((4, 43, 1, pr, po), (4, 17, 12, pr, po), (4, 2, 2, pr, po), (0, 1, 1, pr, po), (-1, 1, 1, pr, po),
                           (4, 1, 1, None, po), (4, 1, 1, pr, None)):
        assert L.lgs_grid_fold_check(ctx._h, r, G, K, ng, o) == -1  # LGS_ERR_INVALID
    assert ctx.launch_count == before
