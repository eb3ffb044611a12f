"""The wide VoxelGrid's reference (tests/voxel_grid_wide_ref.cpp) on the CPU: equal to the 32-bit grid wherever that one
does not refuse, equal to an independent numpy restatement beyond it, and refused exactly at its limits.  Also builds the
C++ shim's map-export calls against liblgs_b200.so.  No GPU needed."""
import os
import subprocess

import numpy as np
import pytest

import map_export_clouds as mc
import voxel_grid_wide_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def wide(tmp_path_factory):
    """the wide VoxelGrid's reference (tests/voxel_grid_wide_ref.cpp), built for this module"""
    L = voxel_grid_wide_ref.build(tmp_path_factory.mktemp("voxel_grid_wide_ref"))
    return lambda *a, **k: voxel_grid_wide_ref.voxel_grid(L, *a, **k)


def _same(w, n):
    """wide result == narrow result, the narrow index widened"""
    assert w["status"] == n["status"] and w["n_kept"] == n["n_kept"]
    assert np.array_equal(w["points"].view(np.uint32), n["points"].view(np.uint32))
    assert w["voxel_idx"].dtype == np.int64 and np.array_equal(w["voxel_idx"], n["voxel_idx"].astype(np.int64))
    assert np.array_equal(w["member_rank"], n["member_rank"])
    assert np.array_equal(w["out_idx"], n["out_idx"].astype(np.int64)) and np.array_equal(w["out_count"], n["out_count"])
    for k in ("min_b", "max_b", "div_b"):
        assert np.array_equal(w[k], n[k]), k


@pytest.mark.parametrize("leaf", [0.1, 0.2, 0.5])
def test_wide_equals_narrow_on_velodyne(oracle, velodyne_pair, leaf, wide):
    for cloud in (velodyne_pair["target"], velodyne_pair["source"]):
        n = oracle.voxel_grid(cloud, leaf)
        assert n["status"] == 0
        _same(wide(cloud, leaf), n)
    src = velodyne_pair["source"]
    for kw in (dict(range_min=1.0), dict(range_min=2.5, box=[-20, 30, -15, 15, -2, 4]), dict(min_points_per_voxel=3),
               dict(range_min=1.0, min_points_per_voxel=2)):
        _same(wide(src, leaf, **kw), oracle.voxel_grid(src, leaf, **kw))


@pytest.mark.parametrize("name", ["cube1291", "clusters33", "clusters48", "far"])
def test_wide_beyond_int32_equals_numpy_restatement(oracle, name, wide):
    cloud, leaf = {"cube1291": (mc.cube(1291, n=60_000), 1.0), "clusters33": (mc.clusters((400, 400, 50), n=60_000), 0.1),
                   "clusters48": (mc.clusters((2000, 2000, 100), n=60_000), 0.01), "far": (mc.far_from_origin(n=40_000), 0.001)}[name]
    assert oracle.voxel_grid(cloud, leaf)["status"] == 1  # the 32-bit grid refuses all of these
    w = wide(cloud, leaf)
    r = mc.restate_wide(cloud, leaf)
    assert w["status"] == 0
    cells = int(np.prod(r["div_b"]))
    assert cells > mc.INT32_MAX
    assert np.array_equal(w["div_b"], r["div_b"]) and np.array_equal(w["min_b"], r["min_b"])
    assert np.array_equal(w["voxel_idx"], r["keys"])
    assert np.array_equal(w["out_idx"], r["out_idx"]) and np.array_equal(w["out_count"], r["counts"])
    assert np.array_equal(w["member_rank"], r["member_rank"])
    np.testing.assert_allclose(w["points"], r["centroids"], rtol=1e-6, atol=0)
    if name == "far":  # beyond 2^24 leaf units the f32 cell index merges neighbouring cells, as PCL's does
        far = (cloud[:, 0] > 10000) & np.isfinite(cloud[:, :3]).all(axis=1)
        ijk0 = r["keys"][far] % r["div_b"][0]
        assert np.all(ijk0 % 2 == 0)


def test_cube_either_side_of_int32_max(oracle, wide):
    below, above = mc.cube(1290, n=30_000), mc.cube(1291, n=30_000)
    nb = oracle.voxel_grid(below, 1.0)
    assert nb["status"] == 0 and list(nb["div_b"]) == [1290] * 3
    _same(wide(below, 1.0), nb)
    assert oracle.voxel_grid(above, 1.0)["status"] == 1
    wa = wide(above, 1.0)
    assert wa["status"] == 0 and list(wa["div_b"]) == [1291] * 3 and wa["voxel_idx"].max() > mc.INT32_MAX


@pytest.mark.parametrize("edge", mc.refusal_edges(), ids=lambda e: e[0])
def test_refusal_limits(edge, wide):
    name, cloud, leaf, refused = edge
    w = wide(cloud, leaf)
    assert w["status"] == (1 if refused else 0), name
    if refused:  # PCL's convention: the cropped input, original order
        assert np.array_equal(w["points"], cloud) and (w["voxel_idx"] == -1).all() and (w["member_rank"] == -1).all()
    else:
        assert int(np.prod(w["div_b"].astype(object))) <= 2 ** 63 - 1
    if name == "cells_int64_max":
        assert [int(v) for v in w["div_b"]] == list(mc.DIV_AT_INT64_MAX)
        assert list(w["voxel_idx"]) == [0, 2 ** 63 - 2]


def test_key63_cube(wide):
    under = wide(mc.key63(False, n=20_000), 0.001)
    assert under["status"] == 0 and all(2 ** 21 - 8 < d < 2 ** 21 for d in under["div_b"])
    assert int(under["voxel_idx"].max()) >= 2 ** 62
    assert wide(mc.key63(True, n=20_000), 0.001)["status"] == 1


def test_edge_clouds(oracle, wide):
    empty = wide(np.zeros((0, 4), np.float32), 0.2)
    assert empty["status"] == 0 and empty["n_kept"] == 0 and len(empty["points"]) == 0
    one = np.array([[1, 2, 3, 4]], np.float32)
    _same(wide(one, 0.2), oracle.voxel_grid(one, 0.2))
    cropped = wide(one, 0.2, range_min=100.0)
    assert cropped["n_kept"] == 0 and len(cropped["points"]) == 0 and list(cropped["voxel_idx"]) == [-1]


def build_shim_map_export(tmpdir):
    exe = os.path.join(str(tmpdir), "shim_map_export")
    libdir = os.path.join(ROOT, "lidar_graph_slam_b200")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "shim_map_export.cpp"),
                           "-o", exe, "-L" + libdir, "-l:liblgs_b200.so", "-Wl,-rpath," + libdir, "-ldl", "-lpthread", "-lrt"])
    return exe


def test_cpp_map_export_shim_compiles_and_links(tmp_path):
    from lidar_graph_slam_b200 import _lib
    _lib.load()
    exe = build_shim_map_export(tmp_path)
    assert "shim compiled" in subprocess.check_output([exe]).decode()
