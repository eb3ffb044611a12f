"""The pcl::Registration shell the four registration objects share: the aligned output cloud, host and device cloud
inputs, the resident evaluators of ICP and pclomp GICP, and the validation of cloud arguments."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TYPES = ("ndt", "gicp", "gicp_omp", "icp")


def _guess(x, y, z, yaw):
    c, s = np.cos(yaw), np.sin(yaw)
    T = np.eye(4, dtype=np.float32)
    T[:2, :2] = [[c, -s], [s, c]]
    T[:3, 3] = [x, y, z]
    return T


GUESS = _guess(0.2, -0.1, 0.02, 0.01)


def _make(api, kind):
    """A registration object with the parameters its node uses."""
    if kind == "ndt":
        x = api.NormalDistributionsTransform()
        x.setResolution(1.0)
        x.setTransformationEpsilon(0.01)
        x.setMaximumIterations(64)
    elif kind == "gicp":
        x = api.FastGICP()
        x.setMaxCorrespondenceDistance(2.0)
    elif kind == "gicp_omp":
        x = api.GeneralizedIterativeClosestPoint()
        x.setMaxCorrespondenceDistance(2.0)
        x.setTransformationEpsilon(0.01)
        x.setMaximumIterations(30)
        x.setMaximumOptimizerIterations(10)
    else:
        x = api.IterativeClosestPoint()
        x.setMaxCorrespondenceDistance(30)
        x.setMaximumIterations(100)
        x.setTransformationEpsilon(1e-8)
        x.setEuclideanFitnessEpsilon(1e-6)
    assert x._prefix == kind
    return x


@pytest.fixture(scope="module")
def clouds(oracle, velodyne_pair):
    return (oracle.voxel_grid(velodyne_pair["target"], 0.25)["points"], oracle.voxel_grid(velodyne_pair["source"], 0.25)["points"])


@pytest.mark.parametrize("kind", TYPES)
def test_output_cloud_is_source_transformed_bit_exact(api, oracle, clouds, kind):
    """align(output, guess): the source transformed by the final transformation with pcl::transformPointCloud's f32
    arithmetic, bit for bit, intensities carried over."""
    target, source = clouds
    x = _make(api, kind)
    x.setInputTarget(target)
    x.setInputSource(source)
    out = x.align(GUESS, want_output=True)
    assert out.shape == source.shape
    assert np.array_equal(out, oracle.transform_point_cloud(source, x.getFinalTransformation()))
    if kind in ("ndt", "gicp"):  # the two types that align an empty source
        x.setInputSource(np.zeros((0, 4), np.float32))
        out = x.align(GUESS, want_output=True)
        assert out.shape == (0, 4)


@pytest.mark.parametrize("kind", TYPES)
def test_device_inputs_match_host_inputs(api, clouds, kind):
    """set_{source,target}_dev (CUDA tensors) and the host uploads give bitwise equal records and fitness."""
    import torch
    target, source = clouds
    runs = []
    for dev in (False, True):
        x = _make(api, kind)
        x.setInputTarget(torch.from_numpy(target).cuda() if dev else target)
        x.setInputSource(torch.from_numpy(source).cuda() if dev else source)
        x.align(GUESS)
        runs.append((bytes(x.result), float(x.getFitnessScore()).hex()))
    assert runs[0] == runs[1]


_RESIDENT_RUN = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from lidar_graph_slam_b200 import api
target, source = np.load(sys.argv[2]), np.load(sys.argv[3])
guesses = np.load(sys.argv[4])
ctx = api.default_context()
out = {}
for kind, cls in (("icp", api.IterativeClosestPoint), ("gicp_omp", api.GeneralizedIterativeClosestPoint)):
    x = cls()
    x.setMaxCorrespondenceDistance(2.0)
    x.setMaximumIterations(30)
    x.setInputTarget(target)
    x.setInputSource(source)
    rows = []
    for G in guesses:
        before = ctx.launch_count
        x.align(G)
        launches = ctx.launch_count - before
        rows.append([bytes(x.result).hex(), float(x.getFitnessScore()).hex(), launches])
    out[kind] = rows
print("RESULT " + json.dumps(out))
"""


def test_resident_and_plain_launches_agree(clouds, tmp_path):
    """ICP and pclomp GICP with their resident evaluators on (LGS_NDT_PERSISTENT=1) and off (=0), each in a process of
    its own (the setting is read once per process): bitwise equal records and fitness, and fewer launches per align
    with the resident grid, which shows that it ran."""
    target, source = clouds
    rs = np.random.RandomState(7)
    guesses = np.stack([_guess(*rs.uniform(-0.3, 0.3, 3), rs.uniform(-0.03, 0.03)) for _ in range(4)])
    paths = []
    for name, a in (("target", target), ("source", source), ("guesses", guesses)):
        paths.append(str(tmp_path / (name + ".npy")))
        np.save(paths[-1], a)
    results = {}
    for knob in ("1", "0"):
        env = dict(os.environ, LGS_NDT_PERSISTENT=knob)
        p = subprocess.run([sys.executable, "-c", _RESIDENT_RUN, ROOT] + paths, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-4000:]
        line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")][-1]
        results[knob] = json.loads(line[len("RESULT "):])
    for kind in ("icp", "gicp_omp"):
        for resident, plain in zip(results["1"][kind], results["0"][kind]):
            assert resident[:2] == plain[:2]
            assert resident[2] < plain[2]


def _align_rc(api, x):
    res = api.AlignResult()
    rc = x._fn("align")(x._h, None, C.byref(res), None)
    return rc, bytes(res)


@pytest.mark.parametrize("kind", TYPES)
def test_dev_setters_validate_their_arguments(api, clouds, kind):
    """set_{source,target}_dev(h, NULL, n > 0) is refused on the host (LGS_ERR_INVALID, no copy, no launch);
    (NULL, 0) sets an empty cloud, after which the object behaves as with an empty host cloud."""
    cloud, _ = clouds
    ctx = api.default_context()
    for which, other in (("source", "Target"), ("target", "Source")):
        x, ref = _make(api, kind), _make(api, kind)
        set_dev = x._fn("set_%s_dev" % which)
        before = ctx.launch_count
        assert set_dev(x._h, None, 5) == -1
        assert ctx.launch_count == before
        assert set_dev(x._h, None, 0) == 0
        getattr(ref, "setInput" + which.capitalize())(np.zeros((0, 4), np.float32))
        for y in (x, ref):
            getattr(y, "setInput" + other)(cloud)
        assert _align_rc(api, x) == _align_rc(api, ref)
