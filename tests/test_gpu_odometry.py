"""Offline odometry (lgs_odometry_run / _dev, DESIGN section 8) on the GPU.

  * the composition is exact: records are bit for bit those of a Python loop over today's public calls (VoxelGrid,
    StatisticalOutlierRemoval, a scratch KeyFrameArray posed at the extrinsic for the base-frame cloud, setInputSource,
    align, KeyFrameArray.push, setInputTargetKeyFrames / assemble), for the three methods, prefilter and SOR on and off,
    identity and non-identity extrinsics; the filled key-frame array holds the loop's poses and assembles the same windows;
  * host form = device form; several sequences in one call, in either order, give each its solo records;
  * oracle parity on a short sequence per method; accuracy against the synthetic truth over 200 frames;
  * dropped frames (hasConverged() false) and refusals before any launch.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import pose_error
from odometry_reference import OracleBackend, make_drive, run_sequence

pytestmark = pytest.mark.gpu
N_FRAMES = 10
METHODS = {"ndt": 0, "gicp": 1, "gicp_omp": 3}
PREFILTERS = {"vg": dict(leaf=0.2, range_min=1.0, sor_mean_k=0), "vg_sor": dict(leaf=0.2, range_min=1.0, sor_mean_k=10, sor_stddev_mul=1.0),
              "off": dict(leaf=None, range_min=None, sor_mean_k=0)}


def _extrinsic(kind):
    if kind == "identity":
        return None
    c, s = np.cos(0.02), np.sin(0.02)
    return np.array([[c, -s, 0, 0.1], [s, c, 0, -0.05], [0, 0, 1, 0.3], [0, 0, 0, 1]], np.float32)


@pytest.fixture(scope="module")
def drives():
    import torch
    a, pa = make_drive(N_FRAMES, n_azimuth=900, spacing=0.4)
    b, pb = make_drive(N_FRAMES - 3, n_azimuth=900, spacing=0.5, seed=7)
    torch.cuda.synchronize()
    return dict(a=(a, pa), b=(b, pb))


class ApiBackend:
    """The loop over the public per-call API, configured as lgs_odometry_run resolves its defaults."""

    def __init__(self, method, leaf, range_min, sor_mean_k=0, sor_stddev_mul=1.0, base_from_sensor=None, max_iterations=64):
        from lidar_graph_slam_b200 import api
        self.api, self.method = api, method
        self.leaf, self.range_min, self.sor_mean_k, self.sor_stddev_mul = leaf, range_min, sor_mean_k, sor_stddev_mul
        self.E = np.eye(4, dtype=np.float32) if base_from_sensor is None else base_from_sensor
        if method == "ndt":
            r = api.NormalDistributionsTransform()
            r.setResolution(2.0)
            r.setStepSize(0.1)
        else:
            r = api.FastGICP() if method == "gicp" else api.GeneralizedIterativeClosestPoint()
            r.setCorrespondenceRandomness(20)
            r.setMaxCorrespondenceDistance(2.0)
            if method == "gicp_omp":
                r.setMaximumOptimizerIterations(20)
        r.setTransformationEpsilon(0.01)
        r.setMaximumIterations(max_iterations)
        self.reg, self.kf, self.scratch = r, api.KeyFrameArray(), api.KeyFrameArray()

    def prefilter(self, cloud):
        x = cloud
        if self.leaf:
            vg = self.api.VoxelGrid()
            vg.setLeafSize(self.leaf)
            vg.setRangeCrop(self.range_min)
            vg.setInputCloud(x)
            x = vg.filter()
        if self.sor_mean_k > 0 and len(x):
            s = self.api.StatisticalOutlierRemoval()
            s.setMeanK(self.sor_mean_k)
            s.setStddevMulThresh(self.sor_stddev_mul)
            s.setInputCloud(x)
            x = s.filter()
        return self.scratch.assemble([self.scratch.push(x, self.E)])  # the base frame, by transform_pcl

    def set_source(self, cloud):
        self.reg.setInputSource(cloud)

    def align(self, T):
        self.reg.align(T)
        r = self.reg.result
        return dict(T=self.reg.getFinalTransformation(), converged=r.converged, iterations=r.iterations, evaluations=r.evaluations,
                    trans_probability=r.trans_probability)

    def push_keyframe(self, cloud, T, accum):
        kid = self.kf.push(cloud, T)
        self.kf.set_accum_distance(kid, accum)
        self.kf.set_position(kid, np.asarray(T, np.float64)[:3, 3])
        return kid

    def set_target(self, ids):
        if self.method == "ndt":
            self.reg.setInputTargetKeyFrames(self.kf, ids)
        else:
            self.reg.setInputTarget(self.kf.assemble(ids))


def _check_records(recs, loop, seq=0):
    from lidar_graph_slam_b200 import api
    assert len(recs) == len(loop)
    T = api.odometry_poses(recs)
    for k, (r, l) in enumerate(zip(recs, loop)):
        assert r["sequence"] == seq and r["frame"] == k
        assert np.array_equal(T[k].view(np.uint32), l["T"].view(np.uint32)), k
        for f in ("n_source", "keyframe_id", "converged", "iterations", "evaluations"):
            assert int(r[f]) == int(l[f]), (k, f, r[f], l[f])
        assert r["accum_distance"] == l["accum_distance"] and r["trans_probability"] == l["trans_probability"], k


def _run(sequences, method, pre, ext=None, **kw):
    from lidar_graph_slam_b200 import api
    return api.odometry(sequences, method=METHODS[method], base_from_sensor=ext, **PREFILTERS[pre], **kw)


@pytest.mark.parametrize("ext", ["identity", "moved"])
@pytest.mark.parametrize("pre", list(PREFILTERS))
@pytest.mark.parametrize("method", list(METHODS))
def test_composition_is_exact(drives, method, pre, ext):
    from lidar_graph_slam_b200 import api, synth
    sweeps, poses = drives["a"]
    frames = [sweeps[k] for k in range(N_FRAMES)]
    if pre == "off":  # without the range crop the invalid rays (zeros) would stay in the cloud
        frames = [f[(f[:, :3] != 0).any(dim=1)].contiguous() for f in frames]
    E = _extrinsic(ext)
    # NDT with the scan-matcher settings stops within about a centimetre of the previous pose on these drives (the oracle
    # does the same): a small displacement gives it key frames; a 3-frame window makes the target window slide
    kd = 0.005 if method == "ndt" else 1.0
    be = ApiBackend(method, base_from_sensor=E, **PREFILTERS[pre])
    loop = run_sequence(frames, be, keyframe_displacement=kd, max_scan_accumulate_num=3, initial_pose=poses[0])
    kf = api.KeyFrameArray()
    recs = _run([frames], method, pre, E, initial_poses=[poses[0]], keyframes=[kf], keyframe_displacement=kd, max_scan_accumulate_num=3)
    _check_records(recs, loop)
    kids = [l["keyframe_id"] for l in loop if l["keyframe_id"] >= 0]
    assert len(kf) == len(kids) == len(be.kf) and 3 < len(kids) <= N_FRAMES
    for w in ([kids[-1]], kids[::-1], kids[:2]):
        assert np.array_equal(kf.assemble(w).cpu().numpy().view(np.uint32), be.kf.assemble(w).cpu().numpy().view(np.uint32))
    # the array's loop-detection inputs are the loop's: accum_distance and f64 positions
    a, b = kf.detect_loop(kids[-1], 0.0, 1e9), be.kf.detect_loop(kids[-1], 0.0, 1e9)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]


@pytest.mark.parametrize("method", list(METHODS))
def test_host_form_equals_device_form(drives, method):
    sweeps, poses = drives["a"]
    dev = _run([[sweeps[k] for k in range(N_FRAMES)]], method, "vg", initial_poses=[poses[0]])
    host = [sweeps[k].cpu().numpy() for k in range(N_FRAMES)]
    h16 = _run([host], method, "vg", initial_poses=[poses[0]])
    z = lambda h, k: np.zeros((len(h), k), np.float32)
    wide = [np.concatenate([h[:, :3], z(h, 1), h[:, 3:4], z(h, 3)], axis=1) for h in host]  # 32-byte pcl::PointXYZI records
    h32 = _run([wide], method, "vg", initial_poses=[poses[0]])
    assert dev.tobytes() == h16.tobytes() == h32.tobytes()


def test_sequences_in_one_call_equal_solo_runs(drives):
    (a, pa), (b, pb) = drives["a"], drives["b"]
    A = [a[k] for k in range(a.shape[0])]
    B = [b[k] for k in range(b.shape[0])]
    solo_a = _run([A], "ndt", "vg", initial_poses=[pa[0]])
    solo_b = _run([B], "ndt", "vg", initial_poses=[pb[0]])
    ab = _run([A, B], "ndt", "vg", initial_poses=[pa[0], pb[0]])
    ba = _run([B, A], "ndt", "vg", initial_poses=[pb[0], pa[0]])
    na = len(A)
    for solo, got, seq in ((solo_a, ab[:na], 0), (solo_b, ab[na:], 1), (solo_b, ba[: len(B)], 0), (solo_a, ba[len(B):], 1)):
        g = got.copy()
        assert (g["sequence"] == seq).all()
        g["sequence"] = 0
        assert g.tobytes() == solo.tobytes()
    # the host form, with an empty sequence in the middle
    hA, hB = [x.cpu().numpy() for x in A], [x.cpu().numpy() for x in B]
    h = _run([hA, [], hB], "ndt", "vg", initial_poses=[pa[0], np.eye(4), pb[0]])
    assert h[:na]["T"].tobytes() == solo_a["T"].tobytes() and h[na:]["T"].tobytes() == solo_b["T"].tobytes()
    assert (h[na:]["sequence"] == 2).all()


def test_dropped_frames_follow_the_loop(drives):
    """FastGICP stopped after one iteration reports hasConverged() false: the pose and the key frames stay (LSM:167-170)."""
    from lidar_graph_slam_b200 import api
    sweeps, poses = drives["a"]
    frames = [sweeps[k] for k in range(N_FRAMES)]
    be = ApiBackend("gicp", max_iterations=1, **PREFILTERS["vg"])
    loop = run_sequence(frames, be, initial_pose=poses[0])
    recs = _run([frames], "gicp", "vg", initial_poses=[poses[0]], max_iterations=1)
    _check_records(recs, loop)
    dropped = [k for k in range(1, N_FRAMES) if not recs[k]["converged"]]
    assert dropped, "no frame was dropped"
    for k in dropped:
        assert recs[k]["keyframe_id"] == -1 and recs[k]["T"].tobytes() == recs[k - 1]["T"].tobytes()


@pytest.mark.parametrize("method", list(METHODS))
def test_oracle_parity(method):
    """12 frames at n_azimuth=900 against the oracle's restatement of the loop: the same key-frame decisions, every pose
    within 1e-4 m / 1e-4 rad, the same iteration counts."""
    sweeps, poses = make_drive(12, n_azimuth=900, spacing=0.4)
    frames = [sweeps[k].cpu().numpy() for k in range(12)]
    ref = run_sequence(frames, OracleBackend(method, leaf=0.2, range_min=1.0), initial_pose=poses[0])
    deltas = [r["delta"] for r in ref if r["delta"] is not None]
    assert all(abs(d - 1.0) > 1e-3 for d in deltas), deltas  # no decision within tolerance of the threshold
    recs = _run([frames], method, "vg", initial_poses=[poses[0]])
    from lidar_graph_slam_b200 import api
    T = api.odometry_poses(recs)
    for k, r in enumerate(ref):
        assert recs[k]["keyframe_id"] == r["keyframe_id"] and recs[k]["converged"] == r["converged"], k
        assert recs[k]["iterations"] == r["iterations"], (k, recs[k]["iterations"], r["iterations"])
        dt, dr = pose_error(r["T"], T[k])
        assert dt < 1e-4 and dr < 1e-4, (k, dt, dr)


def test_accuracy_against_synthetic_truth():
    """200 frames of FastGICP odometry: every frame-to-frame relative pose within 0.05 m / 0.5 deg of the truth (cfg 0
    bounds).  FastGICP, because NDT with the scan-matcher settings stops near the previous pose on these drives."""
    from lidar_graph_slam_b200 import api
    n = 200
    sweeps, poses = make_drive(n, n_azimuth=1875, spacing=0.5)
    recs = api.odometry([sweeps], method=api.METHOD_GICP, leaf=0.2, initial_poses=[poses[0]])
    assert recs["converged"].all()
    T = api.odometry_poses(recs).astype(np.float64)
    worst_t = worst_r = 0.0
    for k in range(1, n):
        rel = np.linalg.inv(T[k - 1]) @ T[k]
        dt, dr = pose_error(np.linalg.inv(poses[k - 1]) @ poses[k], rel)
        worst_t, worst_r = max(worst_t, dt), max(worst_r, dr)
    assert worst_t < 0.05 and np.degrees(worst_r) < 0.5, (worst_t, np.degrees(worst_r))
    assert (recs["keyframe_id"] >= 0).sum() > n // 3


def test_refusals_launch_nothing(drives):
    from lidar_graph_slam_b200 import _lib, api
    ctx = api.default_context()
    L = ctx._L
    sweeps, _ = drives["a"]
    host = [sweeps[k].cpu().numpy() for k in range(3)]

    def call(method=api.METHOD_NDT, n_frames=(3,), sizes=None, ptrs=None, msan=20, kfs=None):
        p = api._odometry_params(method, 1.0, msan, 1.0, 0.2, 0, 1.0, None, 0, 0.0, 0.0, 0, 0.0, 0.0, 0)
        nf = (C.c_int32 * len(n_frames))(*n_frames)
        sz = sizes if sizes is not None else [len(h) for h in host]
        npts = (C.c_int64 * len(sz))(*sz)
        pp = (C.c_void_p * len(sz))(*(ptrs if ptrs is not None else [h.ctypes.data for h in host]))
        recs = np.zeros(8, api.ODOMETRY_FRAME)
        k = (C.c_void_p * 1)(*[x._h.value for x in kfs]) if kfs else None
        before = ctx.launch_count
        rc = L.lgs_odometry_run(ctx._h, C.byref(p), len(n_frames), nf, pp, npts, 16, None, k, recs.ctypes.data_as(C.c_void_p))
        assert ctx.launch_count == before
        return rc

    full = api.KeyFrameArray(ctx)
    full.push(host[0], np.eye(4))
    assert call(method=api.METHOD_ICP) == -1
    assert call(n_frames=(-1,)) == -1
    assert call(sizes=[len(host[0]), -5, len(host[2])]) == -1
    assert call(ptrs=[host[0].ctypes.data, None, host[2].ctypes.data]) == -1
    assert call(kfs=[full]) == -1
    assert call(msan=0) == -1
    assert len(full) == 1
    with pytest.raises(_lib.LgsError, match="ICP|method"):
        api.odometry([host], method=api.METHOD_ICP)
