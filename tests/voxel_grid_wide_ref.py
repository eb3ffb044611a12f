"""ctypes view of tests/voxel_grid_wide_ref.cpp, the reference of the wide VoxelGrid (int64 voxel index, refused only at
int64's limits) that tests/test_map_export_reference.py and tests/test_gpu_map_export.py compare against.  build() compiles
it into a directory the caller owns (a pytest tmp dir); voxel_grid() returns the dict oracle.voxel_grid returns, with
out_idx / voxel_idx in int64."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build(tmp_dir):
    so = os.path.join(str(tmp_dir), "libvoxel_grid_wide_ref.so")
    # the oracle's flags (oracle/Makefile): no FMA contraction, so f32 products and sums round as in the reference build
    subprocess.check_call(["/usr/bin/g++", "-O3", "-std=c++17", "-fPIC", "-shared", "-msse4.2", "-ffp-contract=off", "-Wall", "-Wextra",
                           "-I" + os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests", "voxel_grid_wide_ref.cpp"), "-o", so])
    L = C.CDLL(so)
    vp = C.c_void_p
    L.vgw_run.restype = vp
    L.vgw_run.argtypes = [vp, C.c_long, vp, C.c_int, C.c_double, vp]
    L.vgw_status.argtypes = [vp]
    L.vgw_out_n.restype = C.c_long
    L.vgw_out_n.argtypes = [vp]
    L.vgw_n_kept.restype = C.c_long
    L.vgw_n_kept.argtypes = [vp]
    L.vgw_get.argtypes = [vp] * 7
    L.vgw_free.argtypes = [vp]
    return L


def voxel_grid(L, pts, leaf, min_points_per_voxel=0, range_min=-1.0, box=None):
    p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    assert pts.ndim == 2 and pts.shape[1] == 4
    n = pts.shape[0]
    leaf3 = np.asarray([leaf] * 3 if np.isscalar(leaf) else leaf, dtype=np.float32)
    boxa = None if box is None else np.asarray(box, dtype=np.float64)
    h = L.vgw_run(p(pts), n, p(leaf3), int(min_points_per_voxel), float(range_min), p(boxa))
    try:
        m = L.vgw_out_n(h)
        status = L.vgw_status(h)
        ok = status == 0
        out = np.empty((m, 4), np.float32)
        out_idx = np.empty(m if ok else 0, np.int64)
        out_cnt = np.empty(m if ok else 0, np.int32)
        vidx = np.empty(n, np.int64)
        rank = np.empty(n, np.int32)
        grid = np.zeros(9, np.int32)
        L.vgw_get(h, p(out), p(out_idx), p(out_cnt), p(vidx), p(rank), p(grid))
        return dict(status=status, points=out, out_idx=out_idx, out_count=out_cnt, voxel_idx=vidx, member_rank=rank,
                    min_b=grid[0:3].copy(), max_b=grid[3:6].copy(), div_b=grid[6:9].copy(), n_kept=L.vgw_n_kept(h))
    finally:
        L.vgw_free(h)
