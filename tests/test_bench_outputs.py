"""bench.py --dump-outputs: what the benchmark writes is what its last timed step returned, so that two builds can be
compared output for output on the benchmark's own (seeded) workload."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, pose_error

pytestmark = pytest.mark.gpu

STEPS = 4
T_TOL_M, R_TOL_RAD, FIT_RTOL = 1e-4, 1e-4, 1e-5


def test_bench_dumps_its_last_timed_step(api, oracle, tmp_path):
    """--steps sets the number of timed steps, and --dump-outputs writes what step STEPS - 1 returned: the headline align (sweep
    resident in HBM) and the e2e one (host buffers, aligned cloud back on the host) equal, bit for bit, the same calls made here on
    the same seeded sweep and guess; against the oracle the align keeps the counts and lands within 1e-4 m / 1e-4 rad."""
    out = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(STEPS), "--warmup", "1", "--loop-pairs", "0",
           "--odometry-sweeps", "0", "--no-big-map", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == STEPS
    got = {f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    names = ("final_transformation", "fitness_score", "transformation_probability", "align_counts")
    assert set(got) == set(names) | {"e2e_" + n for n in names} | {"e2e_aligned_cloud"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    import bench
    target, sweeps, guesses, _ = bench.make_workload(0)
    k = (STEPS - 1) % len(sweeps)
    p = bench.NDT_PARAMS
    g, o = api.NormalDistributionsTransform(), oracle.NDT()
    for n in (g, o):
        n.setResolution(p["resolution"])
        n.setStepSize(p["step"])
        n.setTransformationEpsilon(p["eps"])
        n.setMaximumIterations(p["max_iter"])
        n.setNeighborhoodSearchMethod(api.NDT_DIRECT7)
        n.setInputTarget(target)
        n.setInputSource(sweeps[k])
    aligned = g.align(guesses[k], want_output=True)
    res = g.result
    counts = [res.iterations, res.converged, res.evaluations, res.line_search_trials, res.hessian_recomputes]
    for prefix in ("", "e2e_"):
        assert np.array_equal(got[prefix + "final_transformation"], g.getFinalTransformation())
        assert got[prefix + "align_counts"].tolist() == counts
        assert got[prefix + "transformation_probability"][0] == g.getTransformationProbability()
        assert got[prefix + "fitness_score"][0] == g.getFitnessScore()
    assert np.array_equal(got["e2e_aligned_cloud"], aligned)

    o.align(guesses[k])
    assert counts == [o.nr_iterations, o.converged, o.stats["derivative_evals"], o.stats["line_search_trials"], o.stats["hessian_recomputes"]]
    t_err, r_err = pose_error(o.final_transformation, got["final_transformation"])
    assert t_err < T_TOL_M and r_err < R_TOL_RAD
    assert got["transformation_probability"][0] == pytest.approx(o.trans_probability, rel=FIT_RTOL)
    assert got["fitness_score"][0] == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)
