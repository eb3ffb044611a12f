"""CPU checks of the offline odometry bookkeeping (tests/odometry_reference.py, the statement lgs_odometry_run is compared
with) driven by a scripted fake registration, and of the ctypes mirror of lgs_odometry_frame against the C header."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from odometry_reference import keyframe_delta, run_sequence, window


def _pose(x, y=0.0, z=0.0):
    T = np.eye(4, dtype=np.float32)
    T[:3, 3] = (x, y, z)
    return T


class ScriptedBackend:
    """align returns the scripted pose of each frame; converged is False where the script says None."""

    def __init__(self, script):
        self.script, self.k, self.targets, self.pushed = script, 0, [], []

    def prefilter(self, cloud):
        return cloud

    def set_source(self, cloud):
        self.k += 1

    def align(self, T):
        p = self.script[self.k]
        if p is None:
            return dict(T=_pose(123.0), converged=False, iterations=7, evaluations=8, trans_probability=0.5)
        return dict(T=p, converged=True, iterations=3, evaluations=4, trans_probability=1.5)

    def push_keyframe(self, cloud, T, accum):
        self.pushed.append((T.copy(), accum))
        return len(self.pushed) - 1

    def set_target(self, ids):
        self.targets.append(list(ids))


def _run(xs, **kw):
    script = [None if x is None else _pose(x) for x in xs]
    be = ScriptedBackend(script)
    return run_sequence([np.zeros((5, 4), np.float32)] * len(xs), be, **kw), be


def test_keyframe_ids_windows_and_accum_distance():
    xs = [0.0] + [0.4 * k for k in range(1, 60)]
    recs, be = _run(xs, keyframe_displacement=1.0, max_scan_accumulate_num=20)
    kids = [r["keyframe_id"] for r in recs]
    # key frames at 0, 1.2, 2.4, ... (every third frame: 0.4 and 0.8 stay below 1 m)
    assert [k for k, v in enumerate(kids) if v >= 0] == list(range(0, 60, 3))
    assert [v for v in kids if v >= 0] == list(range(20))
    # newest first; fewer than 20 key frames at the start, then the window slides
    assert be.targets[0] == [0] and be.targets[1] == [1, 0] and be.targets[19] == list(range(19, -1, -1))
    assert len(be.targets) == 20 and all(len(t) == min(i + 1, 20) for i, t in enumerate(be.targets))
    recs2, be2 = _run([0.4 * k for k in range(70)], max_scan_accumulate_num=20)
    assert be2.targets[21] == list(range(21, 1, -1))
    # accum_distance: the sum of the f32 deltas, promoted to f64, carried by every later frame
    acc, expect = 0.0, []
    for k in range(60):
        if k and k % 3 == 0:
            acc += float(keyframe_delta(_pose(xs[k]), _pose(xs[k - 3])))
        expect.append(acc)
    assert [r["accum_distance"] for r in recs] == expect
    assert [a for _, a in be.pushed] == [expect[k] for k in range(0, 60, 3)]


def test_delta_equal_to_threshold_makes_a_keyframe():
    d = float(keyframe_delta(_pose(0.75), _pose(0.0)))
    assert d == 0.75
    recs, _ = _run([0.0, 0.75, 1.5], keyframe_displacement=0.75)
    assert [r["keyframe_id"] for r in recs] == [0, 1, 2]
    recs, _ = _run([0.0, 0.75], keyframe_displacement=float(np.nextafter(0.75, 1.0)))
    assert [r["keyframe_id"] for r in recs] == [0, -1]


def test_delta_is_the_f32_norm_of_the_f32_difference():
    a, b = _pose(1e4 + 0.3, 2.0, 0.1), _pose(1e4, 1.0, 0.0)
    d = [np.float32(a[i, 3] - b[i, 3]) for i in range(3)]
    want = np.float32(np.sqrt(np.float32(np.float32(d[0] * d[0] + d[1] * d[1]) + d[2] * d[2])))
    assert keyframe_delta(a, b) == want and keyframe_delta(a, b).dtype == np.float32


def test_dropped_frames_keep_pose_and_keyframes():
    recs, be = _run([0.0, 0.6, None, 1.1, None, 2.3])
    assert [r["converged"] for r in recs] == [1, 1, 0, 1, 0, 1]
    assert [r["keyframe_id"] for r in recs] == [0, -1, -1, 0 + 1, -1, 2]
    assert np.array_equal(recs[2]["T"], recs[1]["T"]) and np.array_equal(recs[4]["T"], recs[3]["T"])
    assert recs[2]["iterations"] == 7 and recs[2]["trans_probability"] == 0.5  # the record still reports the align
    assert recs[2]["accum_distance"] == recs[1]["accum_distance"]


def test_window_helper():
    assert window(0, 20) == [0] and window(3, 2) == [3, 2] and window(25, 20) == list(range(25, 5, -1))


def test_initial_pose_is_keyframe_zero():
    T0 = _pose(5.0, 1.0)
    recs, be = _run([0.0, 5.0 + 0.2], initial_pose=T0)
    assert np.array_equal(recs[0]["T"], T0) and np.array_equal(be.pushed[0][0], T0) and be.pushed[0][1] == 0.0
    assert recs[0]["converged"] == 1 and recs[0]["iterations"] == 0 and recs[0]["keyframe_id"] == 0


def test_ctypes_odometry_frame_matches_the_c_header(tmp_path):
    """lgs_odometry_frame crosses NCCL as bytes: the ctypes mirror and the numpy record have the C size and offsets."""
    from lidar_graph_slam_b200 import _lib, api
    fields = [f for f, _ in _lib.OdometryFrame._fields_]
    src = tmp_path / "sz.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "lgs_c.h"\nint main(void) {\n  printf("%zu", sizeof(lgs_odometry_frame));\n' +
                   "".join('  printf(" %%zu", offsetof(lgs_odometry_frame, %s));\n' % f for f in fields) +
                   '  printf(" %zu\\n", sizeof(lgs_odometry_params));\n  return 0;\n}\n')
    exe = tmp_path / "sz"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.check_call([cc, "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert out[0] == 112 == ctypes.sizeof(_lib.OdometryFrame) == api.ODOMETRY_FRAME.itemsize
    assert out[1:-1] == [getattr(_lib.OdometryFrame, f).offset for f in fields] == [api.ODOMETRY_FRAME.fields[f][1] for f in fields]
    assert out[-1] == ctypes.sizeof(_lib.OdometryParams)
