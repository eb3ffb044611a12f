"""The wide VoxelGrid and the map export on the GPU: bit-identical to the 32-bit grid wherever that one does not refuse,
bit-identical to the wide grid's reference (tests/voxel_grid_wide_ref.cpp) beyond it (points, int64 index, membership, info), refused at the same limits,
and lgs_keyframes_export_map / save_map on a key-frame array filled from a synthetic drive."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import map_export_clouds as mc
import voxel_grid_wide_ref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def wide(tmp_path_factory):
    """the wide VoxelGrid's reference (tests/voxel_grid_wide_ref.cpp), built for this module"""
    L = voxel_grid_wide_ref.build(tmp_path_factory.mktemp("voxel_grid_wide_ref"))
    return lambda *a, **k: voxel_grid_wide_ref.voxel_grid(L, *a, **k)


def _grid(api, cloud, leaf, wide, form="host", want_membership=True, **kw):
    vg = api.VoxelGrid()
    vg.setLeafSize(leaf)
    vg.setWideIndices(wide)
    if "range_min" in kw:
        vg.setRangeCrop(kw["range_min"])
    if "box" in kw:
        vg.setBoxCrop(kw["box"])
    if "min_pts" in kw:
        vg.setMinimumPointsNumberPerVoxel(kw["min_pts"])
    if form == "torch":
        import torch
        cloud = torch.from_numpy(np.ascontiguousarray(cloud, np.float32)).cuda()
    vg.setInputCloud(cloud)
    out = vg.filter(want_membership)
    if form == "torch":
        out = out.cpu().numpy()
        vg.voxel_idx = vg.voxel_idx.cpu().numpy() if want_membership else None
        vg.member_rank = vg.member_rank.cpu().numpy() if want_membership else None
    return vg, out


def _info(vg):
    i = vg.info
    return (i.status, i.n_kept, i.n_out, list(i.min_b), list(i.max_b), list(i.div_b))


def _assert_wide_equals_narrow(api, cloud, leaf, forms=("host", "torch"), **kw):
    vn, on = _grid(api, cloud, leaf, False, **kw)
    assert vn.info.status == 0
    for form in forms:
        vw, ow = _grid(api, cloud, leaf, True, form=form, **kw)
        assert _info(vw) == _info(vn)
        assert np.array_equal(ow.view(np.uint32), on.view(np.uint32))
        assert vw.voxel_idx.dtype == np.int64 and np.array_equal(vw.voxel_idx, vn.voxel_idx.astype(np.int64))
        assert np.array_equal(vw.member_rank, vn.member_rank)


def _assert_equals_oracle(api, wide, cloud, leaf, form="host", **kw):
    ref = wide(cloud, leaf, min_points_per_voxel=kw.get("min_pts", 0), range_min=kw.get("range_min", -1.0), box=kw.get("box"))
    vg, out = _grid(api, cloud, leaf, True, form=form, **kw)
    assert (vg.info.status, vg.info.n_kept, vg.info.n_out) == (ref["status"], ref["n_kept"], len(ref["points"]))
    assert list(vg.info.min_b) == list(ref["min_b"]) and list(vg.info.max_b) == list(ref["max_b"]) and list(vg.info.div_b) == list(ref["div_b"])
    assert np.array_equal(out.view(np.uint32), ref["points"].view(np.uint32))
    assert np.array_equal(vg.voxel_idx, ref["voxel_idx"])
    assert np.array_equal(vg.member_rank, ref["member_rank"])
    return vg, ref


# 1. wide == narrow below the limit -------------------------------------------------------------------------------------

def test_wide_equals_narrow_velodyne(api, velodyne_pair):
    for leaf in (0.1, 0.2, 0.5):
        _assert_wide_equals_narrow(api, velodyne_pair["target"], leaf)
    src = velodyne_pair["source"]
    _assert_wide_equals_narrow(api, src, 0.2, range_min=1.0)
    _assert_wide_equals_narrow(api, src, 0.1, range_min=2.5, box=[-20, 30, -15, 15, -2, 4])
    _assert_wide_equals_narrow(api, src, 0.5, min_pts=3)


def test_wide_equals_narrow_cfg1_and_pcl_layout(api, velodyne_pair):
    from lidar_graph_slam_b200 import synth
    for sweep in synth.prefilter_sweeps(2):
        _assert_wide_equals_narrow(api, sweep, 0.2, range_min=1.0)
    pts = velodyne_pair["target"]
    aos = np.zeros((len(pts), 8), np.float32)  # pcl::PointXYZI: x y z pad | intensity pad pad pad
    aos[:, :3] = pts[:, :3]
    aos[:, 4] = pts[:, 3]
    _assert_wide_equals_narrow(api, aos, 0.3, forms=("host",))
    vw, ow = _grid(api, aos, 0.3, True)
    vn, on = _grid(api, pts, 0.3, False)
    assert np.array_equal(ow, on) and np.array_equal(vw.voxel_idx, vn.voxel_idx.astype(np.int64))


def test_wide_device_form_and_cube_1290(api):
    below = mc.cube(1290)
    _assert_wide_equals_narrow(api, below, 1.0, range_min=5.0)
    _assert_wide_equals_narrow(api, below, 1.0, min_pts=2)


# 2. beyond the limit: equal to the wide grid's reference ---------------------------------------------------------------

def test_cube_1291_narrow_refuses_wide_matches_oracle(api, wide):
    above = mc.cube(1291)
    vn, on = _grid(api, above, 1.0, False)
    assert vn.info.status == api.VG_REFUSED_OVERFLOW and np.array_equal(on, above)
    for form in ("host", "torch"):
        vg, ref = _assert_equals_oracle(api, wide, above, 1.0, form=form)
        assert vg.info.status == 0 and list(vg.info.div_b) == [1291] * 3 and vg.voxel_idx.max() > mc.INT32_MAX


@pytest.mark.parametrize("case", ["clusters33", "clusters48", "far", "key63"])
def test_wide_keys_match_oracle(api, wide, case):
    cloud, leaf = {"clusters33": (mc.clusters((400, 400, 50)), 0.1), "clusters48": (mc.clusters((2000, 2000, 100)), 0.01),
                   "far": (mc.far_from_origin(), 0.001), "key63": (mc.key63(False), 0.001)}[case]
    assert _grid(api, cloud, leaf, False)[0].info.status == api.VG_REFUSED_OVERFLOW
    vg, ref = _assert_equals_oracle(api, wide, cloud, leaf)
    assert vg.info.status == 0
    bits = int(vg.voxel_idx.max()).bit_length()
    assert bits >= {"clusters33": 33, "clusters48": 47, "far": 40, "key63": 62}[case], bits
    _assert_equals_oracle(api, wide, cloud, leaf, form="torch")
    _assert_equals_oracle(api, wide, cloud, leaf, range_min=3.0, min_pts=2)
    _assert_equals_oracle(api, wide, cloud, leaf, box=[-1.0, 300.0, -1.0, 300.0, -1.0, 300.0], min_pts=3)


def test_edge_clouds_match_oracle(api, wide):
    one = np.array([[1, 2, 3, 4]], np.float32)
    for cloud, kw in ((np.zeros((0, 4), np.float32), {}), (one, {}), (one, {"range_min": 100.0}),
                      (np.array([[np.nan, 0, 0, 1], [0, np.inf, 0, 1]], np.float32), {})):
        for form in ("host", "torch"):
            _assert_equals_oracle(api, wide, cloud, 0.2, form=form, **kw)


# 3. refusals and bad arguments ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("edge", mc.refusal_edges(), ids=lambda e: e[0])
def test_refusal_limits_match_oracle(api, wide, edge):
    name, cloud, leaf, refused = edge
    vg, ref = _assert_equals_oracle(api, wide, cloud, leaf)
    assert vg.info.status == (api.VG_REFUSED_OVERFLOW if refused else 0), name
    vg, ref = _assert_equals_oracle(api, wide, cloud, leaf, form="torch")
    if refused:
        assert (vg.voxel_idx == -1).all() and (vg.member_rank == -1).all()


def test_bad_arguments_launch_nothing(api):
    from lidar_graph_slam_b200 import _lib
    L, ctx = _lib.load(), api.default_context()
    pts = np.zeros((4, 4), np.float32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    out = np.zeros((4, 4), np.float32)
    leaf, bad_leaf, nan_leaf = (np.array(v, np.float32) for v in ([0.1] * 3, [0.1, 0.0, 0.1], [np.nan] * 3))
    info = _lib.VoxelGridInfo()
    calls = [
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, vp(pts), 4, 16, vp(bad_leaf), 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, vp(pts), 4, 16, vp(nan_leaf), 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, None, 4, 16, vp(leaf), 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, vp(pts), 4, 16, None, 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, vp(pts), 4, 16, vp(leaf), 0, -1.0, None, vp(out), None, None, None),
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, vp(pts), 4, 10, vp(leaf), 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, vp(pts), -1, 16, vp(leaf), 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide(ctx._h, vp(pts), 2 ** 31, 16, vp(leaf), 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide(None, vp(pts), 4, 16, vp(leaf), 0, -1.0, None, vp(out), None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide_dev(ctx._h, None, 4, vp(leaf), 0, -1.0, None, None, None, None, C.byref(info)),
        lambda: L.lgs_voxelgrid_filter_wide_dev(ctx._h, None, 4, vp(bad_leaf), 0, -1.0, None, None, None, None, C.byref(info)),
    ]
    kf = api.KeyFrameArray()
    kf.push(pts, np.eye(4))
    o, n = C.c_void_p(), C.c_int64()
    ids_bad, ids_neg = np.array([0, 1], np.int32), np.array([-1], np.int32)
    calls += [
        lambda: L.lgs_keyframes_export_map(kf._h, vp(ids_bad), 2, 0.1, C.byref(o), C.byref(n), None),
        lambda: L.lgs_keyframes_export_map(kf._h, vp(ids_neg), 1, 0.1, C.byref(o), C.byref(n), None),
        lambda: L.lgs_keyframes_export_map(kf._h, None, 1, 0.1, C.byref(o), C.byref(n), None),
        lambda: L.lgs_keyframes_export_map(kf._h, vp(ids_bad), -1, 0.1, C.byref(o), C.byref(n), None),
        lambda: L.lgs_keyframes_export_map(kf._h, None, 0, 0.1, None, C.byref(n), None),
        lambda: L.lgs_keyframes_export_map(None, None, 0, 0.1, C.byref(o), C.byref(n), None),
    ]
    ctx.synchronize()
    before = ctx.launch_count
    for i, call in enumerate(calls):
        assert call() == -1, i
    ctx.synchronize()
    assert ctx.launch_count == before


# 4. the map export on a key-frame array ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def drive_keyframes(api):
    from odometry_reference import make_drive
    sweeps, poses = make_drive(10)
    kf = api.KeyFrameArray()
    for k in range(sweeps.shape[0]):
        s = sweeps[k]
        s = s[(s[:, :3] != 0).any(dim=1)].contiguous()
        kf.push(s, poses[k])
    return kf, poses


def _wide_filter(api, cloud, leaf):
    vg = api.VoxelGrid()
    vg.setLeafSize(leaf)
    vg.setWideIndices(True)
    vg.setInputCloud(cloud)
    return vg.filter(False), vg


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.cpu().numpy().view(np.uint32), b.cpu().numpy().view(np.uint32))


def test_export_map_beyond_and_below_the_limit(api, drive_keyframes):
    kf, poses = drive_keyframes
    ids = list(range(len(kf)))
    raw = kf.assemble(ids, 0.0)
    assert _bits_equal(kf.export_map(None, 0.0), raw) and kf.map_info.n_out == raw.shape[0]
    narrow = api.VoxelGrid()
    narrow.setLeafSize(0.02)
    narrow.setInputCloud(raw)
    narrow.filter(False)
    assert narrow.info.status == api.VG_REFUSED_OVERFLOW  # the 32-bit grid refuses this map at 2 cm
    m = kf.export_map(None, 0.02)
    ref, vg = _wide_filter(api, raw, 0.02)
    assert kf.map_info.status == 0 and vg.info.status == 0 and _bits_equal(m, ref)
    assert list(kf.map_info.div_b) == list(vg.info.div_b) and kf.map_info.n_out == vg.info.n_out
    m5 = kf.export_map(None, 0.5)
    assert kf.map_info.status == 0 and _bits_equal(m5, kf.assemble(ids, 0.5))


def test_export_map_follows_set_pose_and_ids(api, drive_keyframes):
    kf, poses = drive_keyframes
    before = kf.export_map(None, 0.02)
    moved = np.array(poses[3], np.float32).copy()
    moved[0, 3] += 0.37
    kf.set_pose(3, moved)
    try:
        after = kf.export_map(None, 0.02)
        assert not _bits_equal(after, before)
        assert _bits_equal(after, _wide_filter(api, kf.assemble(list(range(len(kf))), 0.0), 0.02)[0])
        sub = [6, 1, 3]
        assert _bits_equal(kf.export_map(sub, 0.02), _wide_filter(api, kf.assemble(sub, 0.0), 0.02)[0])
        assert _bits_equal(kf.export_map(sub, 0.0), kf.assemble(sub, 0.0))
    finally:
        kf.set_pose(3, poses[3])


def test_save_map_writes_the_exported_map(api, drive_keyframes, tmp_path):
    from lidar_graph_slam_b200 import pcd
    kf, _ = drive_keyframes
    path = str(tmp_path / "map.pcd")
    n = kf.save_map(path, resolution=0.05)
    m = kf.export_map(None, 0.05).cpu().numpy()
    back = pcd.read_pcd(path)
    assert n == len(m) == len(back) and np.array_equal(back.view(np.uint32), m.view(np.uint32))


def test_cpp_map_export_shim_runs(tmp_path):
    from test_map_export_reference import build_shim_map_export
    exe = build_shim_map_export(tmp_path)
    out = subprocess.run([exe, "--run"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=dict(os.environ))
    assert out.returncode == 0, out.stdout
    assert "map export" in out.stdout
