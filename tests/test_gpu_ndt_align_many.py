"""lgs_ndt_align_many (-m gpu): N NDT aligns in one call.  Every record must be bit for bit what lgs_ndt_align returns for
that problem alone, and every handle must end in the state the same sequence of single aligns leaves."""
import ctypes as C

import numpy as np
import pytest

from conftest import pose_error

pytestmark = pytest.mark.gpu

LGS_ERR_INVALID, LGS_ERR_STATE = -1, -3


def _guesses(rel, seed, count, yaw_deg=4.0, xy=0.6):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        d = np.eye(4)
        yaw = rng.uniform(-1, 1) * np.radians(yaw_deg)
        d[:2, :2] = [[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]
        d[:3, 3] = rng.uniform(-1, 1, 3) * np.array([xy, xy, 0.1])
        out.append((d @ np.asarray(rel, np.float64)).astype(np.float32))
    return out


def _ndt(api, tgt, src, res=1.0, method=None, exact=False, it=64, ctx=None):
    g = api.NormalDistributionsTransform(ctx)
    g.setResolution(res)
    g.setTransformationEpsilon(0.01)
    g.setMaximumIterations(it)
    g.setStepSize(0.1)
    if method is not None:
        g.setNeighborhoodSearchMethod(method)
    if exact:
        g.setExactNewtonStep(True)
    g.setInputTarget(tgt)
    g.setInputSource(src)
    return g


def _key(r):
    """Everything a record reports, as exact values (T as its 64 bytes)."""
    return (np.array(r.T, np.float32).tobytes(), np.float64(r.trans_probability).tobytes(), r.iterations, r.converged, r.evaluations, r.line_search_trials,
            r.hessian_recomputes)


@pytest.fixture(scope="module")
def pair(oracle, velodyne_pair):
    return dict(target=oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"], source=oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"],
                relative=velodyne_pair["relative"])


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("method", [2, 3, 1])  # DIRECT7, DIRECT1, DIRECT26
def test_align_guesses_is_bitwise_the_single_aligns(api, pair, method, exact):
    guesses = _guesses(pair["relative"], 1000 + 10 * method + exact, 16)
    many = _ndt(api, pair["target"], pair["source"], method=method, exact=exact)
    one = _ndt(api, pair["target"], pair["source"], method=method, exact=exact)
    ctx = api.default_context()
    before = ctx.launch_count
    recs = many.align_guesses(guesses)
    assert ctx.launch_count - before == 16  # one ndt_align_kernel launch per align
    assert len(recs) == 16
    for k, (r, guess) in enumerate(zip(recs, guesses)):
        one.align(guess)
        assert _key(r) == _key(one.result), (method, exact, k)
        assert r.pair_id == k
    # the object holds the last guess's result, on the Python and on the library side
    assert _key(many.result) == _key(one.result)
    assert np.array_equal(many.getFinalTransformation(), one.getFinalTransformation())
    assert many.getFitnessScore() == one.getFitnessScore()
    assert len({r.iterations for r in recs}) > 3  # the seeds take different paths


def test_align_guesses_cfg0_multi_tile(api):
    """BASELINE configs[0]: 120 000 source points (several tiles per CTA) against a 1 000 000-point map."""
    from lidar_graph_slam_b200 import synth
    d = synth.ndt_scan_to_map()
    guesses = _guesses(d["guess"], 7, 8, yaw_deg=2.0, xy=0.5)
    many = _ndt(api, d["target"], d["source"])
    one = _ndt(api, d["target"], d["source"])
    ctx = api.default_context()
    before = ctx.launch_count
    recs = many.align_guesses(guesses)
    assert ctx.launch_count - before == 8
    for k, (r, guess) in enumerate(zip(recs, guesses)):
        one.align(guess)
        assert _key(r) == _key(one.result), k


def _mixed_problems(api, pair, velodyne_pair, ctx=None):
    """Handles of different targets, resolutions and search methods, an empty source, a tiny source and a target too small for any
    voxel to be valid (the host steps that align)."""
    td, sd = pair["target"], pair["source"]
    tiny = sd[::200].copy()
    assert 0 < len(tiny) < 32 * 8
    mk = [
        lambda: _ndt(api, td, sd, res=1.0, ctx=ctx),
        lambda: _ndt(api, td, sd, res=2.0, method=1, ctx=ctx),
        lambda: _ndt(api, velodyne_pair["target"], sd, res=1.5, method=3, ctx=ctx),
        lambda: _ndt(api, td, np.zeros((0, 4), np.float32), ctx=ctx),
        lambda: _ndt(api, td, tiny, res=1.0, ctx=ctx),
        lambda: _ndt(api, td[:5].copy(), sd, ctx=ctx),
    ]
    return mk


def test_mixed_handles_equal_the_sequential_calls(api, pair, velodyne_pair):
    mk = _mixed_problems(api, pair, velodyne_pair)
    many = [f() for f in mk]
    seq = [f() for f in mk]
    g = _guesses(pair["relative"], 99, 8)
    order = [0, 1, 2, 3, 4, 5, 0, 2]  # handles 0 and 2 twice
    max_range = 1.0
    recs, clouds = api.ndt_align_many([many[h] for h in order], g, fitness_max_range=max_range, want_output=True)
    for i, h in enumerate(order):
        ref_cloud = seq[h].align(g[i], want_output=True)
        ref_fit = seq[h].getFitnessScore(max_range)
        assert _key(recs[i]) == _key(seq[h].result), i
        assert recs[i].pair_id == i
        assert np.array_equal(clouds[i], ref_cloud), i
        assert np.float64(recs[i].fitness).tobytes() == np.float64(ref_fit).tobytes(), i
    for h in range(len(mk)):  # post-call state: the last occurrence's
        assert _key(many[h].result) == _key(seq[h].result), h
        assert many[h].getFitnessScore(2.0) == seq[h].getFitnessScore(2.0), h


def test_errors_leave_everything_untouched(api, pair):
    td, sd = pair["target"], pair["source"]
    L = api._lib.load()
    a = _ndt(api, td, sd)
    b = _ndt(api, td, sd)
    a.align()
    b.align()
    other_ctx = api.Context(0)
    c = _ndt(api, td, sd, ctx=other_ctx)
    no_target = api.NormalDistributionsTransform()
    no_target.setInputSource(sd)
    g = np.ascontiguousarray(np.stack([np.eye(4, dtype=np.float32).ravel(order="F")] * 3))
    recs = (api.AlignResult * 3)()
    ctx = api.default_context()

    def call(handles, n=None, records=recs):
        hs = (C.c_void_p * max(len(handles), 1))(*[h._h.value if h is not None else None for h in handles])
        return L.lgs_ndt_align_many(hs, len(handles) if n is None else n, g.ctypes.data_as(C.c_void_p), None, records, None)

    fit_a, fit_b = a.getFitnessScore(), b.getFitnessScore()
    before = ctx.launch_count, other_ctx.launch_count
    assert call([a, c, b]) == LGS_ERR_INVALID  # two contexts
    assert call([a, no_target, b]) == LGS_ERR_STATE  # no target
    assert call([a, None, b]) == LGS_ERR_INVALID  # null handle
    assert L.lgs_ndt_align_many(None, 2, None, None, recs, None) == LGS_ERR_INVALID
    assert call([a, b], records=None) == LGS_ERR_INVALID
    assert call([a], n=-1) == LGS_ERR_INVALID
    assert call([], n=0) == 0  # nothing to do
    assert (ctx.launch_count, other_ctx.launch_count) == before
    assert a.getFitnessScore() == fit_a and b.getFitnessScore() == fit_b


def test_align_many_against_the_oracle(api, oracle, pair):
    """Four seeds on the bundled Velodyne pair against oracle.NDT at the parity suite's tolerances."""
    g = _ndt(api, pair["target"], pair["source"])
    guesses = _guesses(pair["relative"], 4242, 4)
    recs = g.align_guesses(guesses)
    o = oracle.NDT()
    o.setResolution(1.0)
    o.setTransformationEpsilon(0.01)
    o.setMaximumIterations(64)
    o.setStepSize(0.1)
    o.setInputTarget(pair["target"])
    o.setInputSource(pair["source"])
    for r, guess in zip(recs, guesses):
        o.align(guess)
        assert (r.iterations, bool(r.converged)) == (o.nr_iterations, o.converged)
        assert (r.evaluations, r.line_search_trials, r.hessian_recomputes) == (o.stats["derivative_evals"], o.stats["line_search_trials"],
                                                                             o.stats["hessian_recomputes"])
        t_err, r_err = pose_error(o.final_transformation, np.array(r.T, np.float32).reshape(4, 4, order="F"))
        assert t_err < 1e-4 and r_err < 1e-4
        assert r.trans_probability == pytest.approx(o.trans_probability, rel=1e-5)


def test_cpp_shim_align_guesses_and_align_many(api, tmp_path):
    """The C++ entry points (NormalDistributionsTransform::alignGuesses, lgs::alignMany) on the GPU: their records equal the
    single aligns bitwise."""
    import subprocess
    from test_shim_align_many import build_shim_align_many
    exe = build_shim_align_many(tmp_path)
    out = subprocess.check_output([exe, "--run"]).decode()
    assert "align_many ok" in out, out
