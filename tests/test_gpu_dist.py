"""cfg 4 (BASELINE configs[4]) at its full size through the distributed C-ABI: lgs_batch_align_keyframes_dist /
lgs_batch_align_dist with the NCCL gather issued by the C++ host (csrc/dist.cu), SURVEY.md section 8e.

  * world 1 (always): the collective path returns, bit for bit, what the plain batch returns; a seeded sample of 96 of the
    4096 pairs is compared with the oracle at the full tolerances (1e-4 m / 1e-4 rad, fitness 1e-5 rel, same iteration count);
  * world 2 / 4 / 8 (when the box has the GPUs): real ranks under torch.distributed.run produce the same 4096 records, bit
    for bit, as the one-rank run (each pair runs on exactly one GPU with deterministic reductions).
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, pose_error

pytestmark = pytest.mark.gpu
N_PAIRS = 4096
T_TOL_M, R_TOL_RAD, FIT_RTOL = 1e-4, 1e-4, 1e-5


def _bytes(recs):
    return b"".join(ctypes.string_at(ctypes.addressof(r), ctypes.sizeof(r)) for r in recs)


def _run_ranks(world, out, pairs=N_PAIRS, host_arrays=0):
    script = os.path.join(ROOT, "tests", "dist_loop_closure.py")
    args = [script, "--pairs", str(pairs), "--out", out, "--host-arrays", str(host_arrays)]
    if world == 1:
        cmd = [sys.executable] + args
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", str(29530 + world)] + args
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:]
    return np.load(out), r.stdout


@pytest.fixture(scope="module")
def cfg4(api):
    from lidar_graph_slam_b200 import synth
    d = synth.loop_keyframes(n_pairs=N_PAIRS, n_keyframes=41, n_azimuth=900, n_unique=2)
    kf = api.KeyFrameArray()
    for c, P in zip(d["clouds"], d["poses"]):
        kf.push(c, P)
    comm = api.Comm(api.Comm.unique_id(), 0, 1, 0)
    recs, info = kf.batch_align_dist(comm, d["scan_ids"], d["center_ids"], search_key_frame_num=20)
    assert info["n_local"] == N_PAIRS and info["n_received"] == N_PAIRS and info["world"] == 1
    yield dict(d=d, kf=kf, comm=comm, recs=recs)
    comm.close()


def test_cfg4_collective_path_equals_plain_batch(api, cfg4):
    """The records that travelled device send buffer -> ncclAllGather -> host are the records the plain batch returns."""
    d, kf, recs = cfg4["d"], cfg4["kf"], cfg4["recs"]
    assert [r.pair_id for r in recs] == list(range(N_PAIRS))
    rng = np.random.default_rng(7)
    pick = sorted(rng.choice(N_PAIRS, 128, replace=False).tolist())
    plain = kf.batch_align([d["scan_ids"][i] for i in pick], [d["center_ids"][i] for i in pick], search_key_frame_num=20, n_workers=2)
    for r, i in zip(plain, pick):
        q = recs[i]
        assert list(r.T) == list(q.T) and r.fitness == q.fitness and (r.iterations, r.converged, r.evaluations, r.line_search_trials) == \
            (q.iterations, q.converged, q.evaluations, q.line_search_trials)


def test_cfg4_sample_of_96_pairs_matches_oracle(api, oracle, cfg4):
    """96 seeded pairs of the 4096 against fast_gicp's restatement: same pose (1e-4 m / 1e-4 rad), same iteration count and
    convergence flag, fitness within 1e-5 relative.  The oracle keeps one target per place (FG:84-86 caches it as well)."""
    d, recs = cfg4["d"], cfg4["recs"]
    K, n_kf = 20, 2 * 41
    rng = np.random.default_rng(11)
    pick = sorted(rng.choice(N_PAIRS, 96, replace=False).tolist())
    oracles = {}
    for i in pick:
        cid, sid = d["center_ids"][i], d["scan_ids"][i]
        if cid not in oracles:
            ids = [j for j in range(cid - K, cid + K + 1) if 0 <= j < n_kf]
            o = oracle.FastGICP()
            o.setMaxCorrespondenceDistance(2.0)
            o.setMaximumIterations(100)
            o.setTransformationEpsilon(0.01)
            o.setInputTarget(oracle.voxel_grid(oracle.assemble_submap(d["clouds"], d["poses"], ids), 0.5)["points"])
            oracles[cid] = o
        o = oracles[cid]
        o.setInputSource(oracle.transform_point_cloud(d["clouds"][sid], d["poses"][sid]))
        o.align()
        r = recs[i]
        t_err, r_err = pose_error(o.final_transformation, np.array(r.T, np.float32).reshape(4, 4, order="F"))
        assert t_err < T_TOL_M and r_err < R_TOL_RAD, (i, t_err, r_err)
        assert (r.iterations, bool(r.converged)) == (o.nr_iterations, o.converged), i
        assert r.fitness == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL), i


def test_cfg4_host_array_collective(api):
    """lgs_batch_align_dist (clouds from host arrays, a rank uploads only the pairs it owns) against the plain host-array batch."""
    from lidar_graph_slam_b200 import synth
    scans, submaps, _ = synth.loop_pairs(n_pairs=6, n_keyframes=41, n_azimuth=900, n_unique=2)
    comm = api.Comm(api.Comm.unique_id(), 0, 1, 0)
    a, info = api.batch_align_dist(comm, scans, submaps, n_workers=2)
    b = api.batch_align(scans, submaps, n_workers=2)
    comm.close()
    assert info["n_received"] == 6
    assert _bytes(a) == _bytes(b)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_cfg4_real_ranks_bitwise_equal_to_one_rank(api, cfg4, tmp_path, world):
    """4096 pairs on `world` real ranks (one process per GPU, NCCL gather in the C++ host): every rank receives all
    records, and they equal the one-rank records bit for bit."""
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs on one machine" % world)
    z, log = _run_ranks(world, str(tmp_path / ("w%d.npz" % world)), host_arrays=16)
    assert int(z["world"]) == world
    assert z["records"].tobytes() == _bytes(cfg4["recs"]), log[-2000:]
    z1, _ = _run_ranks(1, str(tmp_path / "w1h.npz"), pairs=64, host_arrays=16)
    assert z["host_records"].tobytes() == z1["host_records"].tobytes()
