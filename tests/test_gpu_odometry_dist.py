"""Offline odometry over the GPUs of a box (lgs_odometry_run_dist / _dev, DESIGN section 8): sequences dealt to the ranks by
lgs_batch_partition over their point counts, one ncclAllGather of the 112-byte records.

  * world 1: the collective path equals lgs_odometry_run bit for bit (host and device forms);
  * world 2 / 4 / 8 under torch.distributed.run (skipped on a box with fewer GPUs): every rank receives the same records,
    bitwise equal to the one-rank run, and each rank's share is lgs_batch_partition over the sequence sizes.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _run_ranks(world, out, solo=0):
    script = os.path.join(ROOT, "tests", "dist_odometry.py")
    args = [script, "--out", out, "--solo", str(solo)]
    if world == 1:
        cmd = [sys.executable] + args
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
               "--master-port", str(29540 + world)] + args
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)
    r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:]
    return np.load(out), r.stdout


@pytest.fixture(scope="module")
def world1(tmp_path_factory):
    return _run_ranks(1, str(tmp_path_factory.mktemp("odo") / "w1.npz"), solo=1)[0]


def test_world1_equals_plain_run(world1):
    assert len(world1["records"]) > 0 and world1["records"].tobytes() == world1["solo"].tobytes()
    assert list(world1["share0"]) == list(range(len(world1["sizes"])))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_ranks_receive_the_one_rank_records(world, world1, tmp_path):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs in one machine, this one has %d" % (world, torch.cuda.device_count()))
    from lidar_graph_slam_b200 import api
    got, log = _run_ranks(world, str(tmp_path / ("w%d.npz" % world)))
    assert got["records"].tobytes() == world1["records"].tobytes(), log[-2000:]
    sizes = got["sizes"]
    for r in range(world):
        assert list(got["share%d" % r]) == api.partition_pairs(sizes, r, world)
