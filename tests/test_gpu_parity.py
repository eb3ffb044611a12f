"""GPU parity suite (-m gpu): the CUDA path, called through the C-ABI, against the CPU oracle on the same inputs.

Bars (BASELINE.json north_star / SURVEY.md section 8d): voxel indices, occupancy, membership and output order are
bit-exact; voxel mean / inverse covariance rel 1e-9; final transforms within 1e-4 m / 1e-4 rad; fitness and
transformation probability within 1e-5 relative; identical iteration counts and convergence flags."""
import os
import json

import numpy as np
import pytest

from conftest import ROOT, pose_error

pytestmark = pytest.mark.gpu

T_TOL_M, R_TOL_RAD, FIT_RTOL = 1e-4, 1e-4, 1e-5


def _vg(api, pts, leaf, **kw):
    vg = api.VoxelGrid()
    vg.setLeafSize(leaf)
    if "range_min" in kw:
        vg.setRangeCrop(kw["range_min"])
    if "box" in kw:
        vg.setBoxCrop(kw["box"])
    if "min_pts" in kw:
        vg.setMinimumPointsNumberPerVoxel(kw["min_pts"])
    vg.setInputCloud(pts)
    out = vg.filter()
    return vg, out


def _check_vg(api, oracle, pts, leaf, **kw):
    vg, out = _vg(api, pts, leaf, **kw)
    ref = oracle.voxel_grid(pts, leaf, min_points_per_voxel=kw.get("min_pts", 0), range_min=kw.get("range_min", -1.0), box=kw.get("box"))
    assert vg.info.status == ref["status"]
    assert vg.info.n_kept == ref["n_kept"]
    assert out.shape[0] == ref["points"].shape[0]
    if ref["status"] == 0 and ref["n_kept"] > 0:
        assert list(vg.info.min_b) == list(ref["min_b"]) and list(vg.info.div_b) == list(ref["div_b"])
    assert np.array_equal(vg.voxel_idx, ref["voxel_idx"])        # per-point voxel index: bit-exact
    assert np.array_equal(vg.member_rank, ref["member_rank"])    # membership: bit-exact
    # centroids: same f32 summation order as the oracle => expected bit-exact; the contract is rel 1e-5
    np.testing.assert_allclose(out, ref["points"], rtol=1e-5, atol=1e-6)
    return out, ref


def test_voxelgrid_velodyne_bit_exact(api, oracle, velodyne_pair):
    for leaf in (0.1, 0.2, 0.5):
        out, ref = _check_vg(api, oracle, velodyne_pair["target"], leaf)
        assert np.array_equal(out, ref["points"])  # stronger than the contract: identical bits
    _check_vg(api, oracle, velodyne_pair["source"], 0.2, range_min=1.0)
    _check_vg(api, oracle, velodyne_pair["source"], 0.1, range_min=2.5, box=[-20, 30, -15, 15, -2, 4])
    _check_vg(api, oracle, velodyne_pair["source"], 0.5, min_pts=3)


def test_voxelgrid_cfg1_synthetic_128_beam(api, oracle):
    """BASELINE configs[1]: VoxelGrid 0.2 m + min-range crop of 128-beam 262 144-point sweeps, bit-exact membership."""
    from lidar_graph_slam_b200 import synth
    for sweep in synth.prefilter_sweeps(2):
        assert sweep.shape == (262144, 4)
        for leaf in (0.2, 0.1):
            out, ref = _check_vg(api, oracle, sweep, leaf, range_min=1.0)
            assert np.array_equal(out, ref["points"])


def test_voxelgrid_pcl_point_layout_and_edge_cases(api, oracle, velodyne_pair):
    pts = velodyne_pair["target"][:5000]
    aos = np.zeros((len(pts), 8), np.float32)  # pcl::PointXYZI: x y z pad | intensity pad pad pad
    aos[:, :3] = pts[:, :3]
    aos[:, 4] = pts[:, 3]
    vg = api.VoxelGrid()
    vg.setLeafSize(0.3)
    vg.setInputCloud(aos)
    out32 = vg.filter()
    ref = oracle.voxel_grid(pts, 0.3)
    assert np.array_equal(out32, ref["points"])
    # empty, single, all-cropped, overflow refusal
    for cloud, kw in ((np.zeros((0, 4), np.float32), {}), (np.array([[1, 2, 3, 4]], np.float32), {}),
                      (np.array([[1, 2, 3, 4]], np.float32), {"range_min": 100.0})):
        _check_vg(api, oracle, cloud, 0.2, **kw)
    far = np.array([[0, 0, 0, 1], [5000, 5000, 5000, 2]], np.float32)
    vg, out = _vg(api, far, 0.01)
    assert vg.info.status == api.VG_REFUSED_OVERFLOW and np.array_equal(out, far)


def test_voxelgrid_idempotent_at_full_size(api):
    """Size-independent property at BASELINE size: filtering the centroids again with the same leaf keeps one point
    per voxel, and membership counts sum to the kept points."""
    from lidar_graph_slam_b200 import synth
    sweep = synth.prefilter_sweeps(1)[0]
    vg, out = _vg(api, sweep, 0.2, range_min=1.0)
    counts = np.bincount(vg.member_rank[vg.member_rank >= 0], minlength=len(out))
    assert counts.sum() == vg.info.n_kept and counts.min() >= 1
    assert np.all(np.diff(vg.voxel_idx[np.argsort(vg.member_rank, kind="stable")][vg.member_rank[np.argsort(vg.member_rank, kind="stable")] >= 0]) >= 0)
    vg2, out2 = _vg(api, out, 0.2)
    assert len(out2) <= len(out) and len(out2) >= 0.95 * len(out)


# ------------------------------------------------------------------------------------------------------------------
def _ndt_pair(api, oracle, tgt, src, res=1.0, eps=0.01, it=64, method=None):
    g = api.NormalDistributionsTransform()
    o = oracle.NDT()
    for n in (g, o):
        n.setResolution(res)
        n.setTransformationEpsilon(eps)
        n.setMaximumIterations(it)
        n.setStepSize(0.1)
        if method is not None:
            n.setNeighborhoodSearchMethod(method)
        n.setInputTarget(tgt)
        n.setInputSource(src)
    return g, o


def _compare_voxels(g, o):
    vg, vo = g.export_voxels(), o.export_voxels()
    assert np.array_equal(vg["idx"], vo["idx"])          # occupancy: bit-exact
    assert np.array_equal(vg["n"], vo["n"])              # counts and validity flags: bit-exact
    assert list(vg["min_b"]) == list(vo["min_b"]) and list(vg["div_b"]) == list(vo["div_b"])
    valid = vo["n"] >= 6
    assert vg["n_valid"] == valid.sum()
    np.testing.assert_allclose(vg["mean"], vo["mean"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(vg["icov"][valid], vo["icov"][valid], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(vg["cov"][valid], vo["cov"][valid], rtol=1e-9, atol=1e-12)
    return vo, valid


def _compare_align(g, o, guess=None):
    g.align(guess)
    o.align(guess)
    r = g.result
    assert (r.iterations, bool(r.converged)) == (o.nr_iterations, o.converged)
    assert (r.evaluations, r.line_search_trials, r.hessian_recomputes) == (o.stats["derivative_evals"], o.stats["line_search_trials"],
                                                                         o.stats["hessian_recomputes"])
    t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
    assert t_err < T_TOL_M and r_err < R_TOL_RAD
    assert g.getTransformationProbability() == pytest.approx(o.trans_probability, rel=FIT_RTOL)
    assert g.getFitnessScore() == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)


def test_ndt_velodyne_voxels_and_derivatives(api, oracle, velodyne_pair):
    td = oracle.voxel_grid(velodyne_pair["target"], 0.1)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.1)["points"]
    for res in (1.0, 2.0, 0.5):
        g, o = _ndt_pair(api, oracle, td, sd, res=res)
        _compare_voxels(g, o)
        for p in (np.zeros(6), np.array([0.45, 0.12, -0.02, 0.004, -0.008, 0.011])):
            T = oracle.ndt_convert_transform(p)
            for mode in (0, 1, 2):
                so, go, Ho = o.derivatives(T, p, mode)
                sg, gg, Hg = g.derivatives(T, p, mode)
                scale = np.abs(Ho).max() if mode != 1 else 1.0
                if mode != 2:
                    assert sg == pytest.approx(so, rel=1e-12)
                    np.testing.assert_allclose(gg, go, rtol=1e-10, atol=1e-10 * np.abs(go).max())
                if mode == 2:
                    # computeHessian in f64: upper triangle formed like the reference and mirrored (its own (j,i)
                    # entry differs from (i,j) by f64 rounding of the terms only)
                    np.testing.assert_allclose(np.triu(Hg), np.triu(Ho), rtol=1e-9, atol=1e-11 * scale)
                    np.testing.assert_allclose(Hg, Ho, rtol=1e-9, atol=1e-11 * scale)
                    assert np.array_equal(Hg, Hg.T)
                if mode == 0:
                    # all 36 entries exactly as the reference forms them: its (j,i) entry is NOT its (i,j) entry (the f32
                    # products of a term round in the other order, NDT:521-531), and the Newton step sees both triangles
                    np.testing.assert_allclose(Hg, Ho, rtol=1e-12, atol=1e-13 * scale)
                    assert not np.array_equal(Ho, Ho.T) and np.array_equal(Hg == Hg.T, Ho == Ho.T)


def test_ndt_velodyne_align_parity(api, oracle, velodyne_pair):
    td = oracle.voxel_grid(velodyne_pair["target"], 0.1)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.1)["points"]
    for res, eps, it in ((1.0, 0.01, 64), (1.0, 0.1, 35), (2.0, 0.01, 64)):
        g, o = _ndt_pair(api, oracle, td, sd, res=res, eps=eps, it=it)
        _compare_align(g, o)
    g, o = _ndt_pair(api, oracle, td, sd)
    t_err, r_err = None, None
    _compare_align(g, o)
    t_err, r_err = pose_error(velodyne_pair["relative"], g.getFinalTransformation())
    assert t_err < 0.05 and np.degrees(r_err) < 1.0  # the reference's own acceptance band
    # non-identity guess (LSM:165 passes the previous pose), DIRECT1 and DIRECT26 neighbourhoods
    guess = velodyne_pair["relative"].astype(np.float32).copy()
    guess[:3, 3] += np.array([0.2, -0.15, 0.03], np.float32)
    _compare_align(g, o, guess)
    for method in (api.NDT_DIRECT1, api.NDT_DIRECT26):
        g, o = _ndt_pair(api, oracle, td, sd, method=method)
        _compare_align(g, o)


def test_ndt_large_source_multi_tile(api, oracle):
    """A 262 144-point source (cfg 1's 128-beam sweep, unfiltered): every CTA of the evaluator walks several 1024-point
    tiles, in the persistent grid as well as with one launch per evaluation (derivatives hook)."""
    from lidar_graph_slam_b200 import synth
    sweep = synth.prefilter_sweeps(n_sweeps=1)[0]
    tgt = oracle.voxel_grid(synth.drop_invalid(sweep), 0.2)["points"]
    guess = _pose(0.25, -0.2, 0.03, 0.01)
    g, o = _ndt_pair(api, oracle, tgt, sweep, res=1.0, eps=0.01, it=30)
    p = np.array([0.25, -0.2, 0.03, 0.0, 0.0, 0.01])
    T = oracle.ndt_convert_transform(p)
    for mode in (0, 1, 2):
        so, go, Ho = o.derivatives(T, p, mode)
        sg, gg, Hg = g.derivatives(T, p, mode)
        if mode != 2:
            assert sg == pytest.approx(so, rel=1e-12)
            np.testing.assert_allclose(gg, go, rtol=1e-10, atol=1e-10 * np.abs(go).max())
        if mode != 1:
            np.testing.assert_allclose(np.triu(Hg), np.triu(Ho), rtol=1e-9, atol=1e-10 * np.abs(Ho).max())
    _compare_align(g, o, guess)


def test_non_finite_points_are_skipped_like_pcl(api, oracle, velodyne_pair):
    """Clouds that are not is_dense: pcl::VoxelGrid, getMinMax3D and VoxelGridCovariance (VGC:210-215) skip points with a NaN /
    Inf coordinate.  Such rows must not reach the bounding box, a voxel, a centroid or an NDT leaf - with and without a crop."""
    cloud = velodyne_pair["target"][:60000].copy()
    rng = np.random.default_rng(3)
    bad = rng.choice(len(cloud), 500, replace=False)
    cloud[bad[:200], 0] = np.nan
    cloud[bad[200:300], 2] = np.inf
    cloud[bad[300:400], 1] = -np.inf
    cloud[bad[400:], :3] = np.nan
    for crop in (None, 1.0):
        vg = api.VoxelGrid()
        vg.setLeafSize(0.2)
        if crop is not None:
            vg.setRangeCrop(crop)
        vg.setInputCloud(cloud)
        out = vg.filter()
        ref = oracle.voxel_grid(cloud, 0.2, range_min=-1.0 if crop is None else crop)
        assert np.isfinite(out).all()
        assert np.array_equal(vg.voxel_idx, ref["voxel_idx"]) and np.array_equal(vg.member_rank, ref["member_rank"])
        assert np.array_equal(out, ref["points"])
        assert (vg.voxel_idx[bad] == -1).all()
    g, o = _ndt_pair(api, oracle, cloud, velodyne_pair["source"][:30000])
    vo, valid = _compare_voxels(g, o)
    assert np.isfinite(vo["mean"]).all() and valid.sum() > 100
    g.align()
    o.align()
    t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
    assert t_err < T_TOL_M and r_err < R_TOL_RAD and g.result.iterations == o.nr_iterations  # (getFitnessScore's kd-tree over NaN rows is not defined)
    # nothing finite at all: the grid is empty, the align returns the guess without touching the device tables
    g2 = api.NormalDistributionsTransform()
    g2.setInputTarget(np.full((100, 4), np.nan, np.float32))
    g2.setInputSource(velodyne_pair["source"][:1000])
    g2.align()
    assert g2.grid_info().refused and np.array_equal(g2.getFinalTransformation(), np.eye(4, dtype=np.float32))


def test_ndt_device_resident_align_equals_host_stepped(api, velodyne_pair, oracle):
    """The align as ONE cooperative launch (optimiser resident in CTA 0 of ndt_align_kernel) walks the same path as the host
    stepping the same state machine with one launch per evaluation: identical iteration / evaluation / trial / computeHessian
    counts and the same pose, on the bundled pair (several guesses, all three neighbourhoods) and on cfg 0."""
    from lidar_graph_slam_b200 import synth
    td = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    d = synth.ndt_scan_to_map()
    cases = [(td, sd, dict(res=1.0, eps=0.01, it=64), [None, velodyne_pair["relative"].astype(np.float32), _pose(0.3, -0.2, 0.05, 0.03)]),
             (td, sd, dict(res=2.0, eps=0.01, it=64, method=api.NDT_DIRECT1), [None]),
             (td, sd, dict(res=1.0, eps=0.001, it=30, method=api.NDT_DIRECT26), [None]),
             (d["target"], d["source"], dict(res=1.0, eps=0.01, it=64), [d["guess"]])]
    launches = []
    for tgt, src, kw, guesses in cases:
        a, _ = _ndt_pair(api, oracle, tgt, src, **kw)
        b, _ = _ndt_pair(api, oracle, tgt, src, **kw)
        b.profile(1)  # per-evaluation timing: the host steps the optimiser
        for G in guesses:
            l0 = a.ctx.launch_count
            a.align(G)
            launches.append(a.ctx.launch_count - l0)
            b.align(G)
            ra, rb = a.result, b.result
            assert (ra.iterations, ra.converged, ra.evaluations, ra.line_search_trials, ra.hessian_recomputes) == \
                (rb.iterations, rb.converged, rb.evaluations, rb.line_search_trials, rb.hessian_recomputes)
            t_err, r_err = pose_error(b.getFinalTransformation(), a.getFinalTransformation())
            assert t_err < 1e-6 and r_err < 1e-6
            assert ra.trans_probability == pytest.approx(rb.trans_probability, rel=1e-9)
        b.profile(0)
    assert all(l == 1 for l in launches), launches  # one kernel launch per align


def test_ndt_parity_over_many_random_guesses(api, oracle, velodyne_pair):
    """How robust is "same iteration count"?  48 seeded random guesses (up to 0.6 m / 4 deg off the ground truth, every eighth
    four times as far) on the bundled pair at two resolutions: for EVERY one the device-resident align takes the oracle's
    iterations, derivative evaluations, line-search trials and computeHessian calls, and ends on the oracle's transform to
    1e-6 m / 1e-6 rad (in practice the same 16 floats).  The Newton step is a block elimination on the device and a JacobiSVD
    in the oracle, the sines and cosines come from a restatement of the C library's, the sums are added in another order:
    none of these matters.  What does: this test found that the reference's f32-term Hessian is not symmetric (its (i,j) and
    (j,i) entries round their products in different orders, ~1e-8 apart) and that a solver fed one mirrored triangle leaves
    the reference's path on a quarter of these guesses (3 with other iteration counts, 9 more ending up to 2 mm away).  The
    evaluation kernels form all 36 entries since."""
    td = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    rel = velodyne_pair["relative"].astype(np.float64)
    rng = np.random.default_rng(20261018)
    rows = []
    for res in (1.0, 2.0):
        g, o = _ndt_pair(api, oracle, td, sd, res=res, eps=0.01, it=64)
        for k in range(24):
            scale = 4.0 if k % 8 == 7 else 1.0  # every eighth guess is far off
            d = np.eye(4)
            ang = rng.uniform(-1, 1, 3) * np.radians([1.0, 1.0, 4.0]) * scale
            cx, sx, cy, sy, cz, sz = np.cos(ang[0]), np.sin(ang[0]), np.cos(ang[1]), np.sin(ang[1]), np.cos(ang[2]), np.sin(ang[2])
            Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
            Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
            Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
            d[:3, :3] = Rx @ Ry @ Rz
            d[:3, 3] = rng.uniform(-1, 1, 3) * np.array([0.6, 0.6, 0.1]) * scale
            guess = (d @ rel).astype(np.float32)
            g.align(guess)
            o.align(guess)
            r = g.result
            t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
            same = (r.iterations, bool(r.converged), r.evaluations, r.line_search_trials, r.hessian_recomputes) == \
                (o.nr_iterations, o.converged, o.stats["derivative_evals"], o.stats["line_search_trials"], o.stats["hessian_recomputes"])
            fit = abs(g.getTransformationProbability() - o.trans_probability) / abs(o.trans_probability)
            rows.append(dict(res=res, k=k, same=same, it=(r.iterations, o.nr_iterations), conv=(bool(r.converged), bool(o.converged)),
                             t_err=float(t_err), r_err=float(r_err), fit=float(fit)))
    if os.path.isdir(os.path.join(ROOT, "gpurun_out")):
        with open(os.path.join(ROOT, "gpurun_out", "ndt_random_guesses.json"), "w") as f:
            json.dump(rows, f, indent=1)
    assert len(rows) == 48
    for x in rows:
        assert x["same"] and x["t_err"] < 1e-6 and x["r_err"] < 1e-6 and x["fit"] < 1e-9, x
    assert len({x["it"][0] for x in rows}) > 10  # the guesses do exercise different paths (2 to 39 iterations)


def test_gicp_parity_over_many_random_guesses(api, oracle, velodyne_pair):
    """The same for FastGICP (target three times the source, so the lazy target covariances are exercised): 24 random guesses,
    identical nr_iterations / linearisations / error evaluations, poses within 1e-4, fitness within 1e-5."""
    td = oracle.voxel_grid(velodyne_pair["target"], 0.1)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.3)["points"]
    assert len(td) > 2 * len(sd)
    rel = velodyne_pair["relative"].astype(np.float64)
    rng = np.random.default_rng(4242)
    g, o = api.FastGICP(), oracle.FastGICP()
    for x in (g, o):
        x.setMaxCorrespondenceDistance(2.0)
        x.setMaximumIterations(100)
        x.setTransformationEpsilon(0.01)
        x.setInputTarget(td)
        x.setInputSource(sd)
    for k in range(24):
        d = np.eye(4)
        yaw = rng.uniform(-1, 1) * np.radians(5.0)
        d[:2, :2] = [[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]
        d[:3, 3] = rng.uniform(-1, 1, 3) * np.array([1.0, 1.0, 0.1])
        guess = (d @ rel).astype(np.float32)
        g.align(guess)
        o.align(guess)
        assert (g.result.iterations, bool(g.result.converged), g.result.evaluations, g.result.line_search_trials) == \
            (o.nr_iterations, o.converged, o.stats["linearize_calls"], o.stats["error_calls"]), k
        t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
        assert t_err < T_TOL_M and r_err < R_TOL_RAD, (k, t_err, r_err)
        assert g.getFitnessScore() == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)


def test_ndt_rolling_map_incremental_target(api, oracle):
    """SURVEY section 8f-2 / LSM:187-212: the scan matcher's rolling local map as a list of resident key frames, maintained
    incrementally (lgs_ndt_set_target_keyframes).  Sliding the window voxelises only the key frame that entered it; the voxel
    table equals setInputTarget(assembled cloud) - occupancy, counts, validity flags identical, means / covariances to 1e-12 -
    and the oracle's on the same cloud; aligns take the same iterations to the same pose; a moved key frame is re-voxelised."""
    from lidar_graph_slam_b200 import synth
    n_kf, window = 14, 8
    d = synth.loop_keyframes(n_pairs=1, n_keyframes=n_kf, n_azimuth=900, n_unique=1)
    kf = api.KeyFrameArray()
    for c, P in zip(d["clouds"][:n_kf], d["poses"][:n_kf]):
        kf.push(c, P)
    inc = api.NormalDistributionsTransform()
    full = api.NormalDistributionsTransform()
    for x in (inc, full):
        x.setResolution(1.0)
        x.setTransformationEpsilon(0.01)
        x.setMaximumIterations(64)

    def check_same(ids, src, guess, with_oracle=False):
        cloud = kf.assemble(ids)
        full.setInputTarget(cloud)
        vi, vf = inc.export_voxels(), full.export_voxels()
        assert np.array_equal(vi["idx"], vf["idx"]) and np.array_equal(vi["n"], vf["n"]) and vi["n_valid"] == vf["n_valid"]
        assert list(vi["min_b"]) == list(vf["min_b"]) and list(vi["div_b"]) == list(vf["div_b"])
        valid = vf["n"] >= 6
        np.testing.assert_allclose(vi["mean"], vf["mean"], rtol=1e-12, atol=1e-12)
        # the single-pass covariance (VGC:329) cancels sums of ~x^2 n against each other: a 1e-16 relative difference of the
        # sums (per-frame partial sums instead of one running sum) is ~1e-13 absolute at 50 m
        np.testing.assert_allclose(vi["cov"][valid], vf["cov"][valid], rtol=1e-9, atol=1e-11)
        np.testing.assert_allclose(vi["icov"][valid], vf["icov"][valid], rtol=1e-6, atol=1e-6 * np.abs(vf["icov"][valid]).max())
        for x in (inc, full):
            x.setInputSource(src)
            x.align(guess)
        assert (inc.result.iterations, inc.result.converged, inc.result.evaluations) == (full.result.iterations, full.result.converged, full.result.evaluations)
        t_err, r_err = pose_error(full.getFinalTransformation(), inc.getFinalTransformation())
        assert t_err < 1e-6 and r_err < 1e-6
        assert inc.getFitnessScore() == pytest.approx(full.getFitnessScore(), rel=1e-12)  # the cloud is assembled on first use
        if with_oracle:
            o = oracle.NDT()
            o.setResolution(1.0)
            o.setTransformationEpsilon(0.01)
            o.setMaximumIterations(64)
            o.setInputTarget(cloud.cpu().numpy())
            o.setInputSource(src)
            vo = o.export_voxels()
            assert np.array_equal(vi["idx"], vo["idx"]) and np.array_equal(vi["n"], vo["n"])
            np.testing.assert_allclose(vi["mean"], vo["mean"], rtol=1e-9, atol=1e-12)
            o.align(guess)
            t_err, r_err = pose_error(o.final_transformation, inc.getFinalTransformation())
            assert t_err < T_TOL_M and r_err < R_TOL_RAD and inc.result.iterations == o.nr_iterations

    for step in range(n_kf - window + 1):
        ids = list(range(step + window - 1, step - 1, -1))  # newest first, as LSM:199-212 walks the array
        voxelised = inc.setInputTargetKeyFrames(kf, ids)
        assert voxelised == (window if step == 0 else 1), (step, voxelised)
        k = ids[0]
        guess = d["poses"][k].copy()
        guess[:3, 3] += np.array([0.2, -0.15, 0.02], np.float32)
        check_same(ids, d["clouds"][k], guess, with_oracle=step in (0, 3))
    # a pose-graph update moves one key frame of the window: only that frame is voxelised again
    P = d["poses"][ids[3]].copy()
    P[:3, 3] += np.array([0.07, -0.04, 0.01], np.float32)
    kf.set_pose(ids[3], P)
    assert inc.setInputTargetKeyFrames(kf, ids) == 1
    check_same(ids, d["clouds"][ids[0]], guess)
    # a coarser resolution invalidates every cached frame; the same list again costs nothing
    for x in (inc, full):
        x.setResolution(2.0)
    assert inc.setInputTargetKeyFrames(kf, ids) in (0, window)   # setResolution already re-initialised the grid from the frames
    assert inc.setInputTargetKeyFrames(kf, ids) == 0
    check_same(ids, d["clouds"][ids[0]], guess)
    # back to a plain cloud target
    inc.setInputTarget(kf.assemble(ids[:2]))
    full.setInputTarget(kf.assemble(ids[:2]))
    assert np.array_equal(inc.export_voxels()["idx"], full.export_voxels()["idx"])


def test_ndt_cfg0_synthetic_scan_to_map(api, oracle):
    """BASELINE configs[0]: 120 000-point 64-beam sweep against a 1 000 000-point local map, DIRECT7, 1.0 m."""
    from lidar_graph_slam_b200 import synth
    d = synth.ndt_scan_to_map()
    assert d["source"].shape == (120000, 4) and d["target"].shape == (1000000, 4)
    g, o = _ndt_pair(api, oracle, d["target"], d["source"])
    _compare_voxels(g, o)
    _compare_align(g, o, d["guess"])
    t_err, r_err = pose_error(d["T_true"], g.getFinalTransformation())
    assert t_err < 0.05 and r_err < np.radians(0.5)
    # calculateScore (NDT:934-982)
    assert g.calculateScore(g.getFinalTransformation()) == pytest.approx(o.calculateScore(o.final_transformation), rel=1e-9)


@pytest.mark.parametrize("res", [1.0, 0.5])
def test_ndt_cfg3_rolling_map_20m(api, oracle, res):
    """cfg 3 at full size: 120 000-pt sweep against the 20 M-point rolling map at 1.0 m and 0.5 m.  The voxel table of
    all 20 M points equals the oracle's (occupancy, counts and validity bit-exact; means / covariances 1e-9), the
    align takes the same iterations to the same pose."""
    from lidar_graph_slam_b200 import synth
    d = synth.rolling_map()
    assert d["target"].shape == (20_000_000, 4)
    g, o = _ndt_pair(api, oracle, d["target"], d["source"], res=res)
    vo, valid = _compare_voxels(g, o)
    assert valid.sum() > 100_000
    _compare_align(g, o, d["guess"])


def test_ndt_hash_table_path_and_refusal(api, oracle):
    """A sparse, very wide target forces the hashed cell table; results must equal the dense-table oracle semantics.
    A grid above INT32_MAX cells is refused like VGC:79-84 (every lookup misses, align returns the guess)."""
    rs = np.random.RandomState(3)
    centers = rs.uniform(-1000, 1000, size=(300, 3)).astype(np.float32)
    centers[:, 2] = rs.uniform(-100, 100, size=300)
    tgt = (centers[:, None, :] + rs.normal(0, 0.25, size=(300, 40, 3))).reshape(-1, 3).astype(np.float32)
    tgt = np.concatenate([tgt, np.zeros((len(tgt), 1), np.float32)], 1)
    src = tgt[::3].copy()
    src[:, :3] += np.array([0.05, -0.04, 0.02], np.float32)
    g, o = _ndt_pair(api, oracle, tgt, src, res=2.0)
    vo, valid = _compare_voxels(g, o)
    assert valid.sum() > 100 and not g.export_voxels()["dense"] and not g.export_voxels()["refused"]
    _compare_align(g, o)
    big = np.array([[0, 0, 0, 0], [40000, 40000, 4000, 0]], np.float32)
    g, o = _ndt_pair(api, oracle, np.concatenate([tgt, big]), src, res=0.5)
    assert g.export_voxels()["refused"] and o.export_voxels()["refused"]
    _compare_align(g, o)


def test_ndt_set_target_always_rebuilds(api, oracle, velodyne_pair):
    """LSM:187-212 mutates the target cloud in place and re-submits the same pointer: every call must re-voxelise."""
    td = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"].copy()
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g, o = _ndt_pair(api, oracle, td, sd)
    td[:, 0] += 0.37  # in-place mutation of the same buffer
    g.setInputTarget(td)
    o.setInputTarget(td)
    _compare_voxels(g, o)
    _compare_align(g, o)


# ------------------------------------------------------------------------------------------------------------------
def test_statistical_outlier_removal_parity(api, oracle, velodyne_pair):
    """Second prefilter stage (PPF:132-140): per-point mean neighbour distances bit-identical to the oracle's, the same
    threshold (1e-12), the same kept set in the same order; mean_k / multiplier / negative variants; chained after the
    voxel grid on a 128-beam sweep like the node does; device-resident input."""
    import torch
    from lidar_graph_slam_b200 import synth
    clouds = [oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"],
              oracle.voxel_grid(synth.prefilter_sweeps(n_sweeps=1)[0], 0.2, range_min=1.0)["points"]]
    for pts in clouds:
        for mean_k, mul, neg in ((30, 1.2, False), (8, 0.5, False), (30, 1.2, True), (31, 2.0, False)):
            s = api.StatisticalOutlierRemoval()
            s.setMeanK(mean_k)
            s.setStddevMulThresh(mul)
            s.setNegative(neg)
            s.setInputCloud(pts)
            out = s.filter()
            ref = oracle.statistical_outlier_removal(pts, mean_k, mul, neg)
            assert np.array_equal(s.distances, ref["distances"])
            assert s.info.threshold == pytest.approx(ref["threshold"], rel=1e-12)
            assert s.info.mean == pytest.approx(ref["mean"], rel=1e-12) and s.info.stddev == pytest.approx(ref["stddev"], rel=1e-10)
            assert np.array_equal(s.keep, ref["keep"])
            assert np.array_equal(out, ref["points"])
            assert 0 < len(out) < len(pts)
    # device-resident input, outputs stay on the device
    s.setInputCloud(torch.from_numpy(pts).cuda())
    out_d = s.filter()
    assert np.array_equal(out_d.cpu().numpy(), out) and np.array_equal(s.keep.cpu().numpy(), ref["keep"])
    # tiny clouds: fewer points than mean_k + 1, and the empty cloud
    s = api.StatisticalOutlierRemoval()
    s.setMeanK(30)
    s.setStddevMulThresh(1.0)
    s.setInputCloud(pts[:7])
    out = s.filter()
    ref = oracle.statistical_outlier_removal(pts[:7], 30, 1.0)
    assert np.array_equal(s.distances, ref["distances"]) and np.array_equal(out, ref["points"])
    s.setInputCloud(np.zeros((0, 4), np.float32))
    assert len(s.filter()) == 0


@pytest.mark.parametrize("n,bits", [(1, 8), (2, 1), (31, 5), (1024, 8), (1025, 9), (4097, 13), (262144, 21), (1048576 + 77, 30), (3000001, 32)])
def test_radix_sort_pairs_stable_and_exact(api, n, bits):
    """The device sort that orders points by voxel: same permutation as numpy's stable sort (bit-exact, ties in input
    order), for both tile sizes, partial last tiles, clustered keys (long runs of one voxel, as in a sweep) and 1..4
    digit passes."""
    rs = np.random.RandomState(n % 9973)
    mask = np.uint64((1 << bits) - 1)
    keys = (rs.randint(0, 1 << 32, n, dtype=np.uint64) & mask).astype(np.uint32)
    if n > 1000:  # runs of equal keys and a heavily skewed digit
        keys[: n // 3] = np.repeat(keys[: n // 3: 37], 37)[: n // 3]
        keys[n // 2: n // 2 + n // 8] = keys[0]
    vals = np.arange(n, dtype=np.uint32)
    order = np.argsort(keys, kind="stable")
    ks, vs = api.sort_pairs(keys, vals, bits)
    assert np.array_equal(ks, keys[order])
    assert np.array_equal(vs, vals[order])


def test_knn_exact(api, oracle, velodyne_pair):
    pts = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    q = oracle.voxel_grid(velodyne_pair["source"], 0.4)["points"]
    for k in (1, 20):
        ig, dg = api.knn(pts, q, k)
        io, do = oracle.knn(pts, q, k)
        assert np.array_equal(dg, do)   # f32 squared distances: identical bits
        assert np.array_equal(ig, io)   # same tie rule => identical indices
    # far-away queries and duplicates
    qq = np.array([[500, -300, 40, 0], [0, 0, 0, 0]], np.float32)
    dup = np.concatenate([pts[:100], pts[:100]])
    ig, dg = api.knn(dup, qq, 3)
    io, do = oracle.knn(dup, qq, 3)
    assert np.array_equal(ig, io) and np.array_equal(dg, do)


def _gicp_pair(api, oracle, tgt, src, max_corr=None, it=64, eps=5e-4):
    g, o = api.FastGICP(), oracle.FastGICP()
    for x in (g, o):
        x.setMaximumIterations(it)
        x.setTransformationEpsilon(eps)
        if max_corr is not None:
            x.setMaxCorrespondenceDistance(max_corr)
        x.setInputTarget(tgt)
        x.setInputSource(src)
    return g, o


def _compare_gicp_align(g, o, guess=None):
    g.align(guess)
    o.align(guess)
    r = g.result
    assert (r.iterations, bool(r.converged)) == (o.nr_iterations, o.converged)
    assert (r.evaluations, r.line_search_trials) == (o.stats["linearize_calls"], o.stats["error_calls"])
    t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
    assert t_err < T_TOL_M and r_err < R_TOL_RAD
    assert g.getFitnessScore() == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)
    np.testing.assert_allclose(g.getFinalHessian(), o.getFinalHessian(), rtol=1e-6, atol=1e-6 * np.abs(o.getFinalHessian()).max())


def test_gicp_covariances_and_linearize(api, oracle, velodyne_pair):
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g, o = _gicp_pair(api, oracle, t2, s2)
    for which in (0, 1):
        np.testing.assert_allclose(g.covariances(which), o.covariances(which), rtol=1e-6, atol=1e-9)
    T = velodyne_pair["relative"].copy()
    T[:3, 3] += [0.1, -0.05, 0.02]
    cg, Hg, bg, corrg = g.linearize(T)
    co, Ho, bo, corro = o.linearize(T)
    assert np.array_equal(corrg, corro)
    assert cg == pytest.approx(co, rel=1e-10)
    np.testing.assert_allclose(Hg, Ho, rtol=1e-9, atol=1e-9 * np.abs(Ho).max())
    np.testing.assert_allclose(bg, bo, rtol=1e-9, atol=1e-9 * np.abs(bo).max())
    for reg in (api.REG_NONE, api.REG_MIN_EIG, api.REG_NORMALIZED_MIN_EIG, api.REG_FROBENIUS):
        g.setRegularizationMethod(reg)
        o.setRegularizationMethod(reg)
        g.setInputSource(s2[:3000])
        o.setInputSource(s2[:3000])
        cg_, co_ = g.covariances(0), o.covariances(0)
        np.testing.assert_allclose(cg_, co_, rtol=1e-6, atol=1e-7 * np.abs(co_).max())


def test_gicp_set_covariances(api, oracle, velodyne_pair):
    """setSourceCovariances / setTargetCovariances (fast_gicp.hpp:60-70, FG:93-109): supplied covariances are used as they
    are when their count matches the cloud, recomputed otherwise, and dropped by the next setInputSource."""
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g, o = _gicp_pair(api, oracle, t2, s2)
    # covariances of another regularisation, computed by the oracle, handed to both
    alt = oracle.FastGICP()
    alt.setRegularizationMethod(oracle.REG_MIN_EIG)
    alt.setInputSource(s2)
    alt.setInputTarget(t2)
    cs, ct = alt.covariances(0), alt.covariances(1)
    for x in (g, o):
        x.setSourceCovariances(cs)
        x.setTargetCovariances(ct)
    assert np.array_equal(g.getSourceCovariances(), cs) and np.array_equal(g.getTargetCovariances(), ct)
    _compare_gicp_align(g, o)
    # evaluateCost (LSQ:48-50) at the solution and next to it, over the correspondences of the last linearisation
    for dx in (0.0, 0.05):
        T = g.getFinalTransformation().copy()
        T[0, 3] += dx
        assert g.evaluateCost(T) == pytest.approx(o.evaluateCost(T), rel=1e-10)
    assert g.evaluateCost(T) > g.evaluateCost(g.getFinalTransformation())
    with pytest.raises(RuntimeError):
        api.FastGICP().evaluateCost(np.eye(4))
    plane = api.FastGICP()
    plane.setInputTarget(t2)
    plane.setInputSource(s2)
    plane.align()
    assert not np.array_equal(plane.getFinalTransformation(), g.getFinalTransformation())  # the supplied covariances mattered
    # wrong size: ignored, computed at align time (FG:104-109); a new cloud drops them (FG:72-90)
    g.setSourceCovariances(cs[:100])
    g.align()
    assert np.array_equal(g.getFinalTransformation(), _gicp_target_user_source_plane(api, t2, s2, ct))
    g.setInputSource(s2)
    g.setInputTarget(t2)
    g.align()
    assert np.array_equal(g.getFinalTransformation(), plane.getFinalTransformation())


def _gicp_target_user_source_plane(api, t2, s2, ct):
    x = api.FastGICP()
    x.setInputTarget(t2)
    x.setInputSource(s2)
    x.setTargetCovariances(ct)
    x.align()
    return x.getFinalTransformation()


def test_gicp_velodyne_align_parity(api, oracle, velodyne_pair):
    """fast_gicp gtest recipe (gicp_test.cpp:55-65,147-201) + the four set/swap orderings."""
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g, o = _gicp_pair(api, oracle, t2, s2)
    _compare_gicp_align(g, o)
    t_err, r_err = pose_error(velodyne_pair["relative"], g.getFinalTransformation())
    assert t_err < 0.05 and np.degrees(r_err) < 1.0 and g.hasConverged()
    # backward
    g, o = _gicp_pair(api, oracle, s2, t2)
    _compare_gicp_align(g, o)
    t_err, r_err = pose_error(velodyne_pair["relative"], np.linalg.inv(g.getFinalTransformation().astype(np.float64)))
    assert t_err < 0.05 and np.degrees(r_err) < 1.0
    # swap and set source
    g, o = api.FastGICP(), oracle.FastGICP()
    for x in (g, o):
        x.setInputSource(t2)
        x.swapSourceAndTarget()
        x.setInputSource(s2)
    _compare_gicp_align(g, o)
    # swap and set target
    g, o = api.FastGICP(), oracle.FastGICP()
    for x in (g, o):
        x.setInputTarget(s2)
        x.swapSourceAndTarget()
        x.setInputTarget(t2)
    _compare_gicp_align(g, o)
    # product parameters (lidar_scan_matcher.param.yaml: max_corr 2.0, eps 0.01) with a non-identity guess
    g, o = _gicp_pair(api, oracle, t2, s2, max_corr=2.0, eps=0.01)
    guess = np.eye(4, dtype=np.float32)
    guess[:3, 3] = [0.3, 0.0, 0.0]
    _compare_gicp_align(g, o, guess)


def _pc2_message(pts, layout, rng):
    """Packs (N,4) xyzi into a sensor_msgs/PointCloud2-style payload: (point_step, fields) with random filler bytes."""
    point_step, fields = layout
    n = pts.shape[0]
    raw = rng.integers(0, 256, size=(n, point_step), dtype=np.uint8)
    for col, name in enumerate(("x", "y", "z", "intensity")):
        if name not in fields:
            continue
        off, dt = fields[name]
        if dt == 7:
            raw[:, off:off + 4] = np.ascontiguousarray(pts[:, col]).view(np.uint8).reshape(n, 4)
        elif dt == 2:
            raw[:, off] = np.clip(pts[:, col], 0, 255).astype(np.uint8)
    return raw.tobytes()


@pytest.mark.parametrize("layout", [
    (22, {"x": (0, 7), "y": (4, 7), "z": (8, 7), "intensity": (12, 7), "ring": (16, 4), "time": (18, 7)}),    # velodyne_pointcloud PointXYZIRT
    (48, {"x": (0, 7), "y": (4, 7), "z": (8, 7), "intensity": (16, 7), "t": (20, 6), "reflectivity": (24, 4)}),  # ouster-ros
    (16, {"x": (0, 7), "y": (4, 7), "z": (8, 7), "intensity": (12, 7)}),
    (13, {"x": (0, 7), "y": (4, 7), "z": (8, 7), "intensity": (12, 2)}),     # UINT8 intensity: not mapped by fromROSMsg -> 0
    (12, {"x": (0, 7), "y": (4, 7), "z": (8, 7)}),
    (255, {"x": (101, 7), "y": (3, 7), "z": (250, 7), "intensity": (77, 7)}),
], ids=["velodyne22", "ouster48", "packed16", "u8_intensity13", "xyz12", "odd255"])
def test_pointcloud2_ingest_bit_exact(api, oracle, velodyne_pair, layout):
    """sensor_msgs/PointCloud2 payload -> device xyzi (pcl::fromROSMsg, PPF:65-70): every float is copied bit for bit."""
    rng = np.random.default_rng(5)
    point_step, fields = layout
    for n in (0, 1, 255, 256, 257, 69088):
        pts = velodyne_pair["target"][:n].copy()
        if n > 10:
            pts[3] = [np.nan, np.inf, -0.0, 1e-42]  # payload bits travel untouched, denormals and NaN included
        msg = _pc2_message(pts, layout, rng)
        dev = api.from_pointcloud2(msg, n, 1, point_step, fields)
        ref = oracle.from_pointcloud2(msg, n, 1, point_step, fields)
        assert dev.shape == (n, 4)
        assert np.array_equal(dev.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    # organised cloud (height > 1) and the device result feeding the prefilter: same voxels as the host path
    pts = velodyne_pair["target"][:64 * 1024]
    msg = _pc2_message(pts, layout, rng)
    dev = api.from_pointcloud2(msg, 1024, 64, point_step, fields, row_step=1024 * point_step)
    ref = oracle.from_pointcloud2(msg, 1024, 64, point_step, fields)
    assert np.array_equal(dev.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    vg = api.VoxelGrid()
    vg.setLeafSize(0.2)
    vg.setRangeCrop(1.0)
    vg.setInputCloud(dev)
    out = vg.filter()
    out = out.cpu().numpy() if hasattr(out, "cpu") else out
    r = oracle.voxel_grid(ref, 0.2, range_min=1.0)
    assert out.shape == r["points"].shape
    np.testing.assert_allclose(out, r["points"], rtol=1e-5, atol=1e-6)
    with pytest.raises(RuntimeError):
        api.from_pointcloud2(msg, 1024, 64, point_step, dict(fields, x=(fields["x"][0], 8)))  # FLOAT64 x: refused, never guessed


def _pose(x, y, z, yaw, pitch=0.0):
    cy, sy, cp, sp = np.cos(yaw), np.sin(yaw), np.cos(pitch), np.sin(pitch)
    T = np.eye(4, dtype=np.float32)
    T[:3, :3] = np.array([[cy * cp, -sy, cy * sp], [sy * cp, cy, sy * sp], [-sp, 0, cp]], np.float32)
    T[:3, 3] = [x, y, z]
    return T


def test_keyframe_array_submap_assembly(api, oracle, velodyne_pair):
    """Device-resident key_frame_array_ (LSM:196-212, GBS:297-313): the assembled sub-map is bit-identical to transforming
    and concatenating on the host, in both loop orders, across arena chunks, after pose updates, and through VoxelGrid."""
    rng = np.random.default_rng(11)
    base = [velodyne_pair["target"], velodyne_pair["source"]]
    kf = api.KeyFrameArray()
    clouds, poses = [], []
    for i in range(70):  # 70 x ~69 k points: crosses the 4 Mi-point arena chunk
        c = base[i % 2][: 69000 - 137 * i] if i != 5 else base[0][:0]  # key frame 5 is empty
        P = _pose(0.9 * i, 0.05 * i * i / 70, 0.01 * i, 0.02 * i, 0.001 * i)
        assert kf.push(c if i % 3 else np.ascontiguousarray(np.pad(c, ((0, 0), (0, 4)))[:, [0, 1, 2, 7, 3, 4, 5, 6]]), P) == i  # every third as 32-byte PointXYZI
        clouds.append(c)
        poses.append(P)
    assert len(kf) == 70
    # scan matcher order: the newest 20, newest first (LSM:199-208)
    ids = [69 - k for k in range(20)]
    got = kf.assemble(ids).cpu().numpy()
    ref = oracle.assemble_submap(clouds, poses, ids)
    assert got.shape == ref.shape and np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    # graph SLAM order: min_id +- 20 ascending (GBS:297-309), then VoxelGrid 0.5 (GBS:61,311-313)
    ids = list(range(0, 41))
    got = kf.assemble(ids, leaf=0.5).cpu().numpy()
    ref = oracle.assemble_submap(clouds, poses, ids, leaf=0.5)
    assert got.shape == ref.shape
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-6)
    # a pose-graph update moves key frames
    for i in (3, 40):
        poses[i] = _pose(*rng.normal(size=3), 0.3)
        kf.set_pose(i, poses[i])
    got = kf.assemble(ids).cpu().numpy()
    ref = oracle.assemble_submap(clouds, poses, ids)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    # more key frames than one launch takes (96), repeated ids, tiny frames; and the empty selections
    small = api.KeyFrameArray()
    sc = [base[0][1000 * i: 1000 * i + 1 + (i * 37) % 200] for i in range(30)]
    sp = [_pose(i, -i, 0.1 * i, 0.1 * i) for i in range(30)]
    for c, P in zip(sc, sp):
        small.push(c, P)
    ids = [int(v) for v in rng.integers(0, 30, size=250)]
    got = small.assemble(ids).cpu().numpy()
    ref = oracle.assemble_submap(sc, sp, ids)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert small.assemble([]).shape == (0, 4) and kf.assemble([5]).shape == (0, 4)
    with pytest.raises(RuntimeError):
        small.assemble([30])
    # the sub-map never leaves the GPU: NDT on the device sub-map == NDT on the host-assembled one
    ids = [69 - k for k in range(20)]
    target_dev = kf.assemble(ids)
    target_host = oracle.assemble_submap(clouds, poses, ids)
    src = oracle.transform_point_cloud(clouds[69][::4], poses[69] @ _pose(0.2, -0.1, 0.0, 0.01))
    res = []
    for tgt in (target_dev, target_host):
        n = api.NormalDistributionsTransform()
        n.setResolution(1.0)
        n.setTransformationEpsilon(0.01)
        n.setMaximumIterations(30)
        n.setInputTarget(tgt)
        n.setInputSource(src)
        n.align()
        res.append((n.getFinalTransformation().copy(), n.result.iterations, n.getTransformationProbability()))
    assert np.array_equal(res[0][0], res[1][0]) and res[0][1] == res[1][1] and res[0][2] == res[1][2]


def _gicp_omp_pair(api, oracle, target, source, **kw):
    g, o = api.GeneralizedIterativeClosestPoint(), oracle.GeneralizedIterativeClosestPoint()
    for x in (g, o):
        if "max_corr" in kw:
            x.setMaxCorrespondenceDistance(kw["max_corr"])
        if "eps" in kw:
            x.setTransformationEpsilon(kw["eps"])
        if "max_iter" in kw:
            x.setMaximumIterations(kw["max_iter"])
        if "max_inner" in kw:
            x.setMaximumOptimizerIterations(kw["max_inner"])
        if "k" in kw:
            x.setCorrespondenceRandomness(kw["k"])
        x.setInputTarget(target)
        x.setInputSource(source)
    return g, o


def test_fuzzed_clouds_and_parameters_against_the_oracle():
    """tests/diag_fuzz.py, 140 seeded cases x (VoxelGrid, NDT, FastGICP): random clouds (clusters, walls, collinear and duplicated
    points, far-away coordinates) with random leaf sizes, resolutions, neighbourhoods, step sizes and guesses; centroids and
    membership bit-exact, voxel tables 1e-9, aligns with identical counts and transforms within 1e-6 (NDT) / 1e-4 (GICP).
    Seed 1 contains the two cases that once disagreed: an align whose terms are all f32 denormals (case 31: the f64 emulation
    of the f32 roundings now rounds denormals like a float), and one with cond(H) = 4e8 (case 138: ill-conditioned Newton
    systems go to the JacobiSVD restatement)."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "diag_fuzz.py"), "140", "1"], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "140 cases x 3 fuzzers, 0 disagreements" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]


def test_ndt_exact_newton_step_mode_is_bit_identical_to_the_oracle(api, oracle, velodyne_pair):
    """Parity mode (lgs_ndt_set_exact_newton_step / LGS_NDT_EXACT_SOLVE=1): every Newton step of the device-resident align goes
    through the JacobiSVD restatement instead of the block elimination.  Then the whole align repeats the reference's arithmetic
    and the final transform is the oracle's bit for bit - on the bundled pair through the setter, and on 60 fuzzed problems
    (where the default mode ends one f32 ulp away in ~1.5 % of the aligns) through the environment switch."""
    import subprocess
    import sys
    td = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.3)["points"]
    g, o = _ndt_pair(api, oracle, td, sd, res=1.0, eps=0.01, it=64)
    g.setExactNewtonStep(True)
    for guess in _random_guesses(velodyne_pair["relative"], 7, 6):
        g.align(guess)
        o.align(guess)
        r = g.result
        assert (r.iterations, bool(r.converged), r.evaluations, r.line_search_trials, r.hessian_recomputes) == \
            (o.nr_iterations, o.converged, o.stats["derivative_evals"], o.stats["line_search_trials"], o.stats["hessian_recomputes"])
        assert np.array_equal(g.getFinalTransformation(), o.final_transformation)
    env = dict(os.environ, LGS_NDT_EXACT_SOLVE="1", LGS_FUZZ_BITWISE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "diag_fuzz.py"), "60", "31"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0 and "0 disagreements" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]


def _random_guesses(rel, seed, count, yaw_deg=4.0, xy=0.6):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        d = np.eye(4)
        yaw = rng.uniform(-1, 1) * np.radians(yaw_deg)
        d[:2, :2] = [[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]
        d[:3, 3] = rng.uniform(-1, 1, 3) * np.array([xy, xy, 0.1])
        out.append((d @ rel.astype(np.float64)).astype(np.float32))
    return out


@pytest.mark.parametrize("method", [1, 3])  # DIRECT26, DIRECT1 (DIRECT7 has its own test; KDTREE is refused, DESIGN section 8)
def test_ndt_search_methods_over_random_guesses(api, oracle, velodyne_pair, method):
    """The other neighbourhood searches of pclomp NDT (ndt_omp.h:52-57) over 12 random guesses each: identical counts, the
    oracle's transform.  (DIRECT26: 27 cells; DIRECT1: the point's own cell.)"""
    td = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.3)["points"]
    g, o = _ndt_pair(api, oracle, td, sd, res=1.0, eps=0.01, it=40, method=method)
    for k, guess in enumerate(_random_guesses(velodyne_pair["relative"], 77 + method, 12)):
        g.align(guess)
        o.align(guess)
        r = g.result
        assert (r.iterations, bool(r.converged), r.evaluations, r.line_search_trials, r.hessian_recomputes) == \
            (o.nr_iterations, o.converged, o.stats["derivative_evals"], o.stats["line_search_trials"], o.stats["hessian_recomputes"]), (method, k)
        t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
        assert t_err < 1e-6 and r_err < 1e-6, (method, k, t_err, r_err)
        assert g.getTransformationProbability() == pytest.approx(o.trans_probability, rel=1e-9)


def test_gicp_omp_parity_over_random_guesses(api, oracle, velodyne_pair):
    """pclomp GICP (BFGS) over 12 random guesses: identical outer iterations, functor / gradient evaluation counts and inner
    iterations (the exact fixed-point sums make every evaluation bit-identical), poses within 1e-4."""
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.25)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.25)["points"]
    g, o = _gicp_omp_pair(api, oracle, t2, s2, max_corr=2.0, eps=0.01, max_iter=30, max_inner=10)
    for guess in _random_guesses(velodyne_pair["relative"], 99, 12):
        _compare_gicp_omp_align(g, o, guess)


def test_icp_parity_over_random_guesses(api, oracle, velodyne_pair):
    """pcl::IterativeClosestPoint with the loop-closure parameters (GBS:145-149) over 12 random guesses on the same pair of
    objects (PCL's convergence criteria carry state from align to align, reproduced): identical iteration counts and
    convergence states, poses within 1e-4."""
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.25)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.25)["points"]
    g, o = _icp_pair(api, oracle, t2, s2)
    for guess in _random_guesses(velodyne_pair["relative"], 123, 12):
        _compare_icp_align(g, o, guess)


def test_gicp_omp_covariances_and_functor(api, oracle, velodyne_pair):
    """pclomp::GeneralizedIterativeClosestPoint pieces: computeCovariances (GO:48-122), the correspondence / Mahalanobis
    set-up of one outer iteration (GO:404-474) and the three BFGS functor evaluations (GO:245-367)."""
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g, o = _gicp_omp_pair(api, oracle, t2, s2)
    for which in (0, 1):
        cg, co = g.covariances(which), o.covariances(which)
        np.testing.assert_allclose(cg, co, rtol=1e-6, atol=1e-8)
    guess = np.eye(4, dtype=np.float32)
    guess[:3, 3] = [0.2, -0.1, 0.05]
    trans = np.eye(4, dtype=np.float32)
    trans[:3, 3] = [0.05, 0.02, -0.01]
    x = np.array([0.4, 0.1, -0.02, 0.003, -0.004, 0.01])
    rg, ro = g.functor(guess, trans, x), o.functor(guess, trans, x)
    assert np.array_equal(rg["corr"], ro["corr"])            # correspondence indices: bit-exact
    assert rg["n_corr"] == ro["n_corr"] > 7000
    valid = ro["corr"] >= 0
    np.testing.assert_allclose(rg["mahal"][valid], ro["mahal"][valid], rtol=1e-6, atol=1e-6)
    assert rg["f"] == pytest.approx(ro["f"], rel=1e-9)         # f32 terms are bit-identical; only the f64 sum order differs
    assert rg["fdf_f"] == pytest.approx(ro["fdf_f"], rel=1e-10)
    np.testing.assert_allclose(rg["df"], ro["df"], rtol=1e-9, atol=1e-10 * np.abs(ro["df"]).max())
    np.testing.assert_allclose(rg["fdf_g"], ro["fdf_g"], rtol=1e-9, atol=1e-10 * np.abs(ro["fdf_g"]).max())
    np.testing.assert_allclose(rg["fdf_g"], rg["df"], rtol=1e-12, atol=1e-14)


def _compare_gicp_omp_align(g, o, guess=None):
    og = o.align(guess)
    gg = g.align(guess, want_output=True)
    assert g.result.iterations == o.nr_iterations
    assert bool(g.result.converged) == o.converged
    # the BFGS trajectory: identical numbers of functor evaluations and inner iterations
    assert g.result.line_search_trials == o.stats["f_calls"]
    assert g.result.evaluations == o.stats["df_calls"] + o.stats["fdf_calls"]
    assert g.result.hessian_recomputes == o.stats["inner_iterations"]
    t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
    assert t_err < T_TOL_M and r_err < R_TOL_RAD
    assert g.getFitnessScore() == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)
    np.testing.assert_allclose(gg, og, atol=2e-4)


def test_gicp_omp_velodyne_align_parity(api, oracle, velodyne_pair):
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g, o = _gicp_omp_pair(api, oracle, t2, s2)
    _compare_gicp_omp_align(g, o)
    t_err, r_err = pose_error(velodyne_pair["relative"], g.getFinalTransformation())
    assert t_err < 0.05 and np.degrees(r_err) < 1.0 and g.hasConverged()
    # the same objects again (covariances are kept, GO:381-392), with a non-identity guess and the scan matcher's parameters
    guess = np.eye(4, dtype=np.float32)
    guess[:3, 3] = [0.3, 0.0, 0.0]
    _compare_gicp_omp_align(g, o, guess)
    g, o = _gicp_omp_pair(api, oracle, t2, s2, max_corr=2.0, eps=0.01, max_iter=30, max_inner=10)
    _compare_gicp_omp_align(g, o, guess)
    # backward
    g, o = _gicp_omp_pair(api, oracle, s2, t2)
    _compare_gicp_omp_align(g, o)
    t_err, r_err = pose_error(velodyne_pair["relative"], np.linalg.inv(g.getFinalTransformation().astype(np.float64)))
    assert t_err < 0.05 and np.degrees(r_err) < 1.0
    # fewer points than k: the reference logs an error and cannot proceed; here a state error, never a fallback
    g = api.GeneralizedIterativeClosestPoint()
    g.setInputTarget(t2)
    g.setInputSource(s2[:10])
    with pytest.raises(RuntimeError):
        g.align()


def _icp_pair(api, oracle, target, source, gbs=True, **kw):
    g, o = api.IterativeClosestPoint(), oracle.IterativeClosestPoint()
    for x in (g, o):
        if gbs:  # GBS:145-149
            x.setMaxCorrespondenceDistance(30)
            x.setMaximumIterations(100)
            x.setTransformationEpsilon(1e-8)
            x.setEuclideanFitnessEpsilon(1e-6)
            x.setRANSACIterations(0)
        if "max_corr" in kw:
            x.setMaxCorrespondenceDistance(kw["max_corr"])
        if "max_iter" in kw:
            x.setMaximumIterations(kw["max_iter"])
        x.setInputTarget(target)
        x.setInputSource(source)
    return g, o


def _compare_icp_align(g, o, guess=None):
    og = o.align(guess)
    gg = g.align(guess, want_output=True)
    assert g.result.iterations == o.nr_iterations
    assert bool(g.result.converged) == o.converged
    assert g.result.line_search_trials == o.stats["convergence_state"]
    if o.nr_iterations:
        assert g.result.trans_probability == pytest.approx(o.stats["mse"], rel=1e-6)
    t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
    assert t_err < T_TOL_M and r_err < R_TOL_RAD
    assert g.getFitnessScore() == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)
    np.testing.assert_allclose(gg, og, atol=2e-4)


def test_icp_step_and_align_parity(api, oracle, velodyne_pair):
    """pcl::IterativeClosestPoint (the default loop-closure method, GBS:142-151): correspondence sums and the Umeyama step,
    then whole aligns with identical iteration counts and convergence states."""
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g, o = _icp_pair(api, oracle, t2, s2)
    guess = np.eye(4, dtype=np.float32)
    guess[:3, 3] = [0.2, -0.1, 0.05]
    for G in (np.eye(4, dtype=np.float32), guess):
        okg, sg, Tg = g.step(G)
        oko, so, To = o.step(G)
        assert okg and oko and sg[0] == so[0]
        np.testing.assert_allclose(sg, so, rtol=1e-12)       # f64 sums of identical terms: only the order differs
        assert np.array_equal(Tg, To)                         # rounded to f32 before the SVD: bit-identical
    _compare_icp_align(g, o)
    assert g.hasConverged() and g.result.line_search_trials == 2  # CONVERGENCE_CRITERIA_TRANSFORM
    _compare_icp_align(g, o, guess)
    # gated correspondences (FAST_GICP-like 2 m), full-resolution clouds, iteration cap of the PCL defaults
    g, o = _icp_pair(api, oracle, velodyne_pair["target"], velodyne_pair["source"], max_corr=2.0)
    _compare_icp_align(g, o)
    g, o = _icp_pair(api, oracle, t2, s2, gbs=False)
    _compare_icp_align(g, o)
    assert g.result.iterations == 10 and g.result.line_search_trials == 1
    # nothing within reach: not converged, final transformation = guess
    far = s2 + np.array([500, 0, 0, 0], np.float32)
    g, o = _icp_pair(api, oracle, t2, far, max_corr=0.5)
    _compare_icp_align(g, o, guess)
    assert not g.hasConverged() and g.result.line_search_trials == 5 and np.array_equal(g.getFinalTransformation(), guess)


def test_gicp_cfg2_synthetic_odometry(api, oracle):
    """BASELINE configs[2] in miniature: scan-to-scan GICP over consecutive synthetic 64-beam sweeps, VoxelGrid 0.25 m
    (kitti.cpp:80-82), covariance reuse through swapSourceAndTarget (kitti.cpp:115-125)."""
    from lidar_graph_slam_b200 import synth
    sweeps, poses = synth.odometry_sequence(4)
    ds = [oracle.voxel_grid(s, 0.25, range_min=1.0)["points"] for s in sweeps]
    g, o = api.FastGICP(), oracle.FastGICP()
    for x in (g, o):
        x.setMaxCorrespondenceDistance(1.0)
        x.setInputTarget(ds[0])
    for k in range(1, len(ds)):
        for x in (g, o):
            x.setInputSource(ds[k])
        _compare_gicp_align(g, o)
        rel_true = np.linalg.inv(poses[k - 1]) @ poses[k]
        t_err, r_err = pose_error(rel_true, g.getFinalTransformation())
        assert t_err < 0.1 and r_err < np.radians(1.0)
        for x in (g, o):
            x.swapSourceAndTarget()


def test_gicp_clear_source_and_target(api, oracle, velodyne_pair):
    """clearSource / clearTarget (FG:60-69): the cloud, its tree and its covariances are gone - align refuses to run - and setting
    the clouds again gives the registration of a fresh object, bit for bit."""
    t2 = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    s2 = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g = api.FastGICP()
    g.setInputTarget(t2)
    g.setInputSource(s2)
    g.align()
    T0, it0 = g.getFinalTransformation().copy(), g.result.iterations
    g.clearSource()
    with pytest.raises(RuntimeError):
        g.align()
    g.setInputSource(s2)
    g.clearTarget()
    with pytest.raises(RuntimeError):
        g.align()
    g.setInputTarget(t2)
    g.align()
    assert np.array_equal(g.getFinalTransformation(), T0) and g.result.iterations == it0
    g.clearSource()
    g.clearTarget()
    g.setInputSource(t2)   # the roles swapped after a full clear
    g.setInputTarget(s2)
    g.align()
    o = oracle.FastGICP()
    o.setInputSource(t2)
    o.setInputTarget(s2)
    o.align()
    t_err, r_err = pose_error(o.final_transformation, g.getFinalTransformation())
    assert t_err < T_TOL_M and r_err < R_TOL_RAD and g.result.iterations == o.nr_iterations


def test_ndt_align_fills_the_output_cloud(api, oracle, velodyne_pair):
    """align(output, guess) (LSM:164-165): the output cloud is the source transformed by the final transformation with
    pcl::transformPointCloud's arithmetic - bit for bit, intensities carried over - for the device-resident align and the
    host-stepped one."""
    td = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    for stepped in (False, True):
        g, _ = _ndt_pair(api, oracle, td, sd)
        if stepped:
            g.profile(1)
        out = g.align(_pose(0.2, -0.1, 0.02, 0.01), want_output=True)
        assert out.shape == sd.shape
        assert np.array_equal(out, oracle.transform_point_cloud(sd, g.getFinalTransformation()))
        if stepped:
            g.profile(0)


def test_keyframe_loop_detection_uses_f64_positions(api):
    """detect_loop_with_accum_dist compares the f64 positions of geometry_msgs poses (GBS:163-171): a key frame 15 m - 1e-9 away
    is a candidate, which the f32 pose matrix alone (15.000000 exactly) would reject (dist < threshold is strict)."""
    kf = api.KeyFrameArray()
    pts = np.zeros((10, 4), np.float32)
    pos = [(0.0, 0.0), (60.0, 0.0), (120.0, 0.0), (15.0 - 1e-9, 0.0)]
    acc = [0.0, 60.0, 120.0, 225.0]
    for (x, y), a in zip(pos, acc):
        P = np.eye(4, dtype=np.float32)
        P[:3, 3] = [x, y, 0.0]
        kid = kf.push(pts, P)
        kf.set_accum_distance(kid, a)
    cand, nearest = kf.detect_loop(3, accumulate_distance_threshold=100.0, search_for_candidate_threshold=15.0)
    assert list(cand) == [] and nearest == -1          # f32: |15.0 - 0.0| < 15 is false
    for kid, (x, y) in enumerate(pos):
        kf.set_position(kid, [x, y, 0.0])
    cand, nearest = kf.detect_loop(3, accumulate_distance_threshold=100.0, search_for_candidate_threshold=15.0)
    assert list(cand) == [0] and nearest == 0


def test_gicp_cfg2_long_drive_1000_sweeps(api, oracle):
    """BASELINE configs[2] at its full size (kitti.cpp:80-82, 115-138): scan-to-scan FastGICP odometry over 1000 consecutive
    120 000-ray sweeps of a 1 km drive, VoxelGrid 0.25 m + range crop, max_corr 1.0, covariance reuse through
    swapSourceAndTarget, pose accumulated as poses[i] = poses[i-1] * T.
      * every frame: converged, per-frame pose within 3 cm / 0.1 deg of the synthetic ground truth (the accumulated
        trajectory's drift is whatever scan-to-scan GICP drifts on this scene - it is compared with the oracle, not the truth);
      * a sample of frames (every 25th + a contiguous run of 24) against the oracle at the full tolerances - per-frame T within
        1e-4 m / 1e-4 rad, same nr_iterations - and the trajectory accumulated over the contiguous run within 5e-4 m."""
    import torch
    from lidar_graph_slam_b200 import synth
    n = int(os.environ.get("LGS_CFG2_SWEEPS", 1000))
    sweeps, poses = synth.long_drive(n, device="cuda")
    vg = api.VoxelGrid()
    vg.setLeafSize(0.25)
    vg.setRangeCrop(1.0)
    g = api.FastGICP()
    g.setMaxCorrespondenceDistance(1.0)
    run0 = n // 2
    sample = sorted(set(range(25, n, 25)) | set(range(run0, min(run0 + 24, n))))
    need = set(sample) | {k - 1 for k in sample}
    host, rel, iters, n_pts = {}, [None], [0], []
    for k in range(n):
        vg.setInputCloud(sweeps[k])
        ds = vg.filter(want_membership=False)
        n_pts.append(int(ds.shape[0]))
        if k in need:
            host[k] = ds.cpu().numpy()
        if k == 0:
            g.setInputTarget(ds)
            continue
        g.setInputSource(ds)
        g.align()
        assert g.hasConverged(), k
        rel.append(g.getFinalTransformation().astype(np.float64))
        iters.append(g.result.iterations)
        g.swapSourceAndTarget()
    assert min(n_pts) > 15000
    # ground truth: per-frame and accumulated
    X = np.eye(4)
    worst_t = worst_r = 0.0
    for k in range(1, n):
        true_rel = np.linalg.inv(poses[k - 1]) @ poses[k]
        t_err, r_err = pose_error(true_rel, rel[k])
        worst_t, worst_r = max(worst_t, t_err), max(worst_r, r_err)
        X = X @ rel[k]
    assert worst_t < 0.03 and worst_r < np.radians(0.1), (worst_t, worst_r)
    assert np.isfinite(X).all()
    # the oracle on the sampled frames
    acc_g, acc_o = np.eye(4), np.eye(4)
    for k in sample:
        o = oracle.FastGICP()
        o.setMaxCorrespondenceDistance(1.0)
        o.setInputTarget(host[k - 1])
        o.setInputSource(host[k])
        o.align()
        t_err, r_err = pose_error(o.final_transformation, rel[k])
        assert t_err < T_TOL_M and r_err < R_TOL_RAD, (k, t_err, r_err)
        assert iters[k] == o.nr_iterations and o.converged, k
        if run0 <= k < run0 + 24:
            acc_g = acc_g @ rel[k]
            acc_o = acc_o @ o.final_transformation.astype(np.float64)
    t_err, r_err = pose_error(acc_o, acc_g)
    assert t_err < 5e-4 and r_err < 5e-4, (t_err, r_err)
    del sweeps
    torch.cuda.empty_cache()


def test_batch_loop_closure_matches_single_pair_runs(api, oracle):
    """BASELINE configs[4] in miniature: the batch API equals per-pair runs of the oracle (VoxelGrid 0.5 m on the
    submap, FastGICP with graph_based_slam.param.yaml parameters, fitness), independent of worker count."""
    from lidar_graph_slam_b200 import synth
    scans, submaps, corrections = synth.loop_pairs(n_pairs=4, n_keyframes=9, n_unique=2)
    recs1 = api.batch_align(scans, submaps, method=api.METHOD_GICP, n_workers=1)
    recs3 = api.batch_align(scans, submaps, method=api.METHOD_GICP, n_workers=3, pair_id0=100)
    for i, (r1, r3) in enumerate(zip(recs1, recs3)):
        assert list(r1.T) == list(r3.T) and r1.fitness == r3.fitness and r1.iterations == r3.iterations  # bitwise
        assert r1.pair_id == i and r3.pair_id == 100 + i
        o = oracle.FastGICP()
        o.setMaximumIterations(100)
        o.setTransformationEpsilon(0.01)
        o.setMaxCorrespondenceDistance(2.0)
        o.setInputTarget(oracle.voxel_grid(submaps[i], 0.5)["points"])
        o.setInputSource(scans[i])
        o.align()
        T = np.array(r1.T, np.float32).reshape(4, 4, order="F")
        t_err, r_err = pose_error(o.final_transformation, T)
        assert t_err < T_TOL_M and r_err < R_TOL_RAD
        assert (r1.iterations, bool(r1.converged)) == (o.nr_iterations, o.converged)
        assert r1.fitness == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)
        t_err, r_err = pose_error(corrections[i], T)
        assert t_err < 0.1 and r_err < np.radians(0.5)
    # NDT through the same batch entry point.  NDT at 1 m resolution cannot recover the 2 m / 5 deg offsets of the
    # candidates (it wanders, and a wandering optimiser is chaotic in its last digits), so it gets a close guess.
    guesses = []
    for i in range(2):
        g = corrections[i].copy()
        g[:3, 3] += [0.08, -0.05, 0.02]
        guesses.append(g.astype(np.float32))
    recs_ndt = api.batch_align(scans[:2], submaps[:2], method=api.METHOD_NDT, n_workers=2, guesses=guesses)
    for i, r in enumerate(recs_ndt):
        o = oracle.NDT()
        o.setMaximumIterations(100)
        o.setTransformationEpsilon(0.01)
        o.setInputTarget(oracle.voxel_grid(submaps[i], 0.5)["points"])
        o.setInputSource(scans[i])
        o.align(guesses[i])
        T = np.array(r.T, np.float32).reshape(4, 4, order="F")
        t_err, r_err = pose_error(o.final_transformation, T)
        assert t_err < T_TOL_M and r_err < R_TOL_RAD and r.iterations == o.nr_iterations
        assert r.fitness == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)


def test_batch_loop_closure_icp_and_gicp_omp_methods(api, oracle):
    """The node's other two loop-closure methods through the batch entry point: pcl::IterativeClosestPoint with the
    GBS:142-151 settings (the YAML default) and pclomp::GeneralizedIterativeClosestPoint with GBS:120-141's."""
    from lidar_graph_slam_b200 import synth
    scans, submaps, corrections = synth.loop_pairs(n_pairs=3, n_keyframes=9, n_unique=2)
    recs = api.batch_align(scans, submaps, method=api.METHOD_ICP, n_workers=2, max_iterations=100, transformation_epsilon=1e-8,
                           max_correspondence_distance=30.0, euclidean_fitness_epsilon=1e-6)
    recs1 = api.batch_align(scans, submaps, method=api.METHOD_ICP, n_workers=1, max_iterations=100, transformation_epsilon=1e-8,
                            max_correspondence_distance=30.0, euclidean_fitness_epsilon=1e-6)
    for i, r in enumerate(recs):
        assert list(r.T) == list(recs1[i].T) and r.fitness == recs1[i].fitness  # bitwise independent of the worker count
        o = oracle.IterativeClosestPoint()
        o.setMaxCorrespondenceDistance(30)
        o.setMaximumIterations(100)
        o.setTransformationEpsilon(1e-8)
        o.setEuclideanFitnessEpsilon(1e-6)
        o.setInputTarget(oracle.voxel_grid(submaps[i], 0.5)["points"])
        o.setInputSource(scans[i])
        o.align()
        T = np.array(r.T, np.float32).reshape(4, 4, order="F")
        t_err, r_err = pose_error(o.final_transformation, T)
        assert t_err < T_TOL_M and r_err < R_TOL_RAD
        assert (r.iterations, bool(r.converged), r.line_search_trials) == (o.nr_iterations, o.converged, o.stats["convergence_state"])
        assert r.fitness == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)
    recs = api.batch_align(scans, submaps, method=api.METHOD_GICP_OMP, n_workers=2, max_iterations=100, transformation_epsilon=0.01,
                           max_correspondence_distance=2.0, max_optimizer_iterations=20)
    for i, r in enumerate(recs):
        o = oracle.GeneralizedIterativeClosestPoint()
        o.setMaxCorrespondenceDistance(2.0)
        o.setMaximumIterations(100)
        o.setMaximumOptimizerIterations(20)
        o.setTransformationEpsilon(0.01)
        o.setInputTarget(oracle.voxel_grid(submaps[i], 0.5)["points"])
        o.setInputSource(scans[i])
        o.align()
        T = np.array(r.T, np.float32).reshape(4, 4, order="F")
        t_err, r_err = pose_error(o.final_transformation, T)
        assert t_err < T_TOL_M and r_err < R_TOL_RAD
        assert (r.iterations, bool(r.converged)) == (o.nr_iterations, o.converged)
        assert r.fitness == pytest.approx(o.getFitnessScore(), rel=FIT_RTOL)
        t_err, r_err = pose_error(corrections[i], T)
        assert t_err < 0.1 and r_err < np.radians(0.5)


def test_batch_loop_closure_from_keyframe_array(api, oracle):
    """optimization_callback for a list of candidates with every cloud already in HBM (lgs_batch_align_keyframes): the
    records are bit-identical to the host-array batch fed with the oracle's transformed / assembled clouds, for the GICP
    and ICP methods; and detect_loop_with_accum_dist (GBS:157-187) picks the reference's candidates."""
    from lidar_graph_slam_b200 import synth
    K = 4
    d = synth.loop_keyframes(n_pairs=3, n_keyframes=2 * K + 1, n_azimuth=900, n_unique=2)
    kf = api.KeyFrameArray()
    for c, P in zip(d["clouds"], d["poses"]):
        kf.push(c, P)
    n_kf = len(kf)
    scans, submaps = [], []
    for sid, cid in zip(d["scan_ids"], d["center_ids"]):
        ids = [j for j in range(cid - K, cid + K + 1) if 0 <= j < n_kf]
        scans.append(oracle.transform_point_cloud(d["clouds"][sid], d["poses"][sid]))
        submaps.append(oracle.assemble_submap(d["clouds"], d["poses"], ids))
    for method, kw in ((api.METHOD_GICP, {}), (api.METHOD_ICP, dict(max_correspondence_distance=30.0, transformation_epsilon=1e-8,
                                                                      euclidean_fitness_epsilon=1e-6))):
        a = kf.batch_align(d["scan_ids"], d["center_ids"], search_key_frame_num=K, method=method, n_workers=2, **kw)
        b = api.batch_align(scans, submaps, method=method, n_workers=2, **kw)
        for ra, rb in zip(a, b):
            assert list(ra.T) == list(rb.T) and ra.fitness == rb.fitness and ra.iterations == rb.iterations and ra.converged == rb.converged
        if method == api.METHOD_GICP:
            for r, corr in zip(a, d["corrections"]):
                t_err, r_err = pose_error(corr, np.array(r.T, np.float32).reshape(4, 4, order="F"))
                assert r.converged and t_err < 0.1 and r_err < np.radians(0.5)
    # the clipped neighbourhood at the ends of the array (GBS:299: ids outside [0, size) are skipped)
    a = kf.batch_align([d["scan_ids"][0]], [1], search_key_frame_num=K, n_workers=1)
    ids = [j for j in range(1 - K, 1 + K + 1) if 0 <= j < n_kf]
    b = api.batch_align([scans[0]], [oracle.assemble_submap(d["clouds"], d["poses"], ids)], n_workers=1)
    assert list(a[0].T) == list(b[0].T) and a[0].fitness == b[0].fitness
    with pytest.raises(RuntimeError):
        kf.batch_align([n_kf], [0])
    # the GICP methods take at most 32 neighbours: a larger k fails the call instead of running with the k a worker had
    for method in (api.METHOD_GICP, api.METHOD_GICP_OMP):
        with pytest.raises(RuntimeError, match="k_correspondences"):
            kf.batch_align(d["scan_ids"], d["center_ids"], search_key_frame_num=K, method=method, k_correspondences=33)
        with pytest.raises(RuntimeError, match="k_correspondences"):
            api.batch_align(scans, submaps, method=method, k_correspondences=33)
    # candidate search: key frames along a loop, 2 m apart, the latest one back near the start
    loop = api.KeyFrameArray()
    pts = d["clouds"][0][:100]
    pos = [(2.0 * i, 0.0) for i in range(60)] + [(3.0, 4.0)]
    acc = 0.0
    for i, (x, y) in enumerate(pos):
        if i:
            acc += float(np.hypot(x - pos[i - 1][0], y - pos[i - 1][1]))
        P = np.eye(4, dtype=np.float32)
        P[:3, 3] = [x, y, 0.0]
        loop.set_accum_distance(loop.push(pts, P), acc)
    cand, nearest = loop.detect_loop(60, accumulate_distance_threshold=100.0, search_for_candidate_threshold=15.0)
    dist = np.array([np.hypot(3.0 - x, 4.0 - y) for x, y in pos[:60]])
    accd = np.concatenate([[0.0], np.cumsum(np.hypot(np.diff([p[0] for p in pos]), np.diff([p[1] for p in pos])))])
    want = [i for i in range(61) if accd[60] - accd[i] >= 100.0 and np.hypot(3.0 - pos[i][0], 4.0 - pos[i][1]) < 15.0]
    assert list(cand) == want and len(want) > 3
    assert nearest == want[int(np.argmin(dist[want]))]
    cand, nearest = loop.detect_loop(10)
    assert len(cand) == 0 and nearest == -1


def test_loop_closure_cfg4_full_size_properties(api):
    """BASELINE configs[4] at its full size: 4096 (scan, 41-key-frame sub-map) candidates verified from the device
    key-frame array.  The oracle needs seconds per pair, so this checks size-independent properties: every candidate
    that passes the node's fitness gate sits on its known correction (and at least 99 % pass), and a record does not depend on the worker count, on the order of the batch, or
    on the shard (rank) it is dealt to - bit for bit."""
    from lidar_graph_slam_b200 import synth
    from lidar_graph_slam_b200.distributed import partition_pairs
    n_pairs = 4096
    d = synth.loop_keyframes(n_pairs=n_pairs, n_keyframes=41, n_azimuth=900, n_unique=2)
    kf = api.KeyFrameArray()
    for c, P in zip(d["clouds"], d["poses"]):
        kf.push(c, P)
    assert len(kf) == 2 * 41 + n_pairs
    recs = kf.batch_align(d["scan_ids"], d["center_ids"], search_key_frame_num=20, n_workers=4)
    assert [r.pair_id for r in recs] == list(range(n_pairs))
    assert all(r.converged for r in recs)
    # GBS:328 accepts a candidate iff it converged and fitness <= score_threshold_ (0.3, graph_based_slam.param.yaml:6).
    # Every accepted candidate sits on its known correction (no false loop closure); the few that GICP drags into a wrong
    # basin from a 2 m / 5 deg offset have a fitness ten times the threshold and are rejected.
    accepted = 0
    for r, corr in zip(recs, d["corrections"]):
        t_err, r_err = pose_error(corr, np.array(r.T, np.float32).reshape(4, 4, order="F"))
        if r.fitness <= 0.3:
            accepted += 1
            assert t_err < 0.1 and r_err < np.radians(0.5)
        else:
            assert t_err > 0.5 and r.fitness > 1.0
    assert accepted >= 0.99 * n_pairs
    # shard 3 of 8 (what rank 3 of an 8-GPU job verifies), shuffled, one worker: the same records
    mine = partition_pairs([1] * n_pairs, 3, 8)[:48]
    rng = np.random.default_rng(2)
    order = [mine[i] for i in rng.permutation(len(mine))]
    sub = kf.batch_align([d["scan_ids"][i] for i in order], [d["center_ids"][i] for i in order], search_key_frame_num=20, n_workers=1)
    for r, i in zip(sub, order):
        assert list(r.T) == list(recs[i].T) and r.fitness == recs[i].fitness and r.iterations == recs[i].iterations


def test_registrations_survive_degenerate_clouds(api, velodyne_pair):
    """Empty or tiny clouds never take the process or the GPU down: the calls return (an error or a not-converged
    result, as the reference's objects would report), and the same objects work normally afterwards."""
    s2 = velodyne_pair["source"][:5000]
    t2 = velodyne_pair["target"][:5000]
    empty = np.zeros((0, 4), np.float32)
    g = api.FastGICP()
    g.setInputTarget(empty)
    g.setInputSource(s2)
    g.align()                       # no target points: no correspondences at any LM iteration (seeded search included)
    g.align()
    g.setInputTarget(t2)
    g.setInputSource(empty)
    g.align()
    assert g.result.iterations == 0
    for cls in (api.IterativeClosestPoint, api.GeneralizedIterativeClosestPoint):
        x = cls()
        x.setInputTarget(empty)
        x.setInputSource(s2)
        with pytest.raises(RuntimeError):
            x.align()
        x.setInputTarget(t2)
        x.align()
        assert x.result.iterations >= 1
    n = api.NormalDistributionsTransform()
    n.setInputTarget(t2)
    n.setInputSource(empty)
    n.align()
    n.setInputSource(s2)
    n.align()
    assert n.result.iterations >= 1
    g.setInputSource(s2)
    g.align()
    assert g.hasConverged()


def test_device_resident_inputs(api, oracle, velodyne_pair):
    """_dev entry points: clouds already in HBM (torch tensors) give the same results as host uploads."""
    import torch
    td = oracle.voxel_grid(velodyne_pair["target"], 0.2)["points"]
    sd = oracle.voxel_grid(velodyne_pair["source"], 0.2)["points"]
    g1 = api.NormalDistributionsTransform()
    g2 = api.NormalDistributionsTransform()
    g1.setInputTarget(td)
    g1.setInputSource(sd)
    g2.setInputTarget(torch.from_numpy(td).cuda())
    g2.setInputSource(torch.from_numpy(sd).cuda())
    g1.align()
    g2.align()
    assert np.array_equal(g1.getFinalTransformation(), g2.getFinalTransformation())
    vg = api.VoxelGrid()
    vg.setLeafSize(0.2)
    vg.setInputCloud(torch.from_numpy(velodyne_pair["target"]).cuda())
    out = vg.filter().cpu().numpy()
    assert np.array_equal(out, td)


def test_cpp_shim_runs_reference_call_sequence(api, tmp_path):
    """The header-only C++ shim drives VoxelGrid + NDT through the reference's call order on the GPU."""
    import subprocess
    from test_oracle_cpu import _build_shim
    exe = _build_shim(tmp_path)
    out = subprocess.check_output([exe, "--run"]).decode()
    assert "converged 1" in out, out
