"""Restatement of the offline odometry loop of lgs_odometry_run (DESIGN section 8; the scan matcher's callback_cloud,
LSM:122-250) over a pluggable backend, so that one statement of the bookkeeping drives three checks:

- a scripted fake registration (CPU tests of the key-frame decisions, windows, accum_distance and dropped frames);
- the oracle (`OracleBackend`: oracle/pyoracle.py's VoxelGrid, outlier filter, registrations and sub-map assembly);
- the library's public per-call API (the GPU composition test builds that backend).

A backend provides prefilter(cloud) -> base-frame cloud, set_source(cloud), align(T) -> dict(T, converged, iterations,
evaluations, trans_probability), push_keyframe(cloud, T, accum_distance) -> id and set_target(ids).
"""
import numpy as np


def keyframe_delta(T, T_kf):
    """LSM:183 as the library computes it: the f32 norm ((dx*dx + dy*dy) + dz*dz) of the f32 translation difference."""
    d = [np.float32(np.float32(T[a, 3]) - np.float32(T_kf[a, 3])) for a in range(3)]
    s = np.float32(np.float32(np.float32(d[0] * d[0]) + np.float32(d[1] * d[1])) + np.float32(d[2] * d[2]))
    return np.float32(np.sqrt(s))


def window(latest_id, max_scan_accumulate_num):
    """LSM:199-212: the newest max_scan_accumulate_num key frames, newest first."""
    return list(range(latest_id, max(-1, latest_id - max_scan_accumulate_num), -1))


def run_sequence(frames, backend, keyframe_displacement=1.0, max_scan_accumulate_num=20, initial_pose=None, sequence=0):
    """Returns one dict per frame with the fields of lgs_odometry_frame (T as a 4x4 float32) plus `delta` (the key-frame
    test's distance, None where no test ran)."""
    T = np.eye(4, dtype=np.float32) if initial_pose is None else np.asarray(initial_pose, np.float32).reshape(4, 4).copy()
    T_kf, accum, out = None, 0.0, []
    for k, cloud in enumerate(frames):
        base = backend.prefilter(cloud)
        rec = dict(sequence=sequence, frame=k, n_source=int(len(base)), keyframe_id=-1, converged=0, iterations=0, evaluations=0,
                   trans_probability=0.0, delta=None)
        if k == 0:  # LSM:133-160: key frame 0 and the first target, at the initial pose
            kid = backend.push_keyframe(base, T, accum)
            backend.set_target(window(kid, max_scan_accumulate_num))
            T_kf = T.copy()
            rec.update(converged=1, keyframe_id=kid)
        else:
            backend.set_source(base)
            r = backend.align(T)
            rec.update(converged=int(r["converged"]), iterations=int(r["iterations"]), evaluations=r["evaluations"],
                       trans_probability=r["trans_probability"])
            if r["converged"]:  # LSM:167-170: otherwise the frame is dropped
                T = np.asarray(r["T"], np.float32).copy()
                delta = keyframe_delta(T, T_kf)
                rec["delta"] = float(delta)
                if float(delta) >= keyframe_displacement:
                    accum += float(delta)
                    kid = backend.push_keyframe(base, T, accum)
                    backend.set_target(window(kid, max_scan_accumulate_num))
                    T_kf = T.copy()
                    rec["keyframe_id"] = kid
        rec["T"] = T.copy()
        rec["accum_distance"] = accum
        out.append(rec)
    return out


class OracleBackend:
    """The loop on the oracle: VoxelGrid + range crop, outlier filter, pcl::transformPointCloud and the sub-map assembly of
    LSM:199-208, with the registration settings lgs_odometry_run resolves by default (SURVEY Appendix C)."""

    def __init__(self, method, leaf=0.1, range_min=1.0, sor_mean_k=0, sor_stddev_mul=1.0, base_from_sensor=None):
        from oracle import pyoracle as O
        self.O = O
        self.leaf, self.range_min, self.sor_mean_k, self.sor_stddev_mul = leaf, range_min, sor_mean_k, sor_stddev_mul
        self.E = np.eye(4, dtype=np.float32) if base_from_sensor is None else np.asarray(base_from_sensor, np.float32)
        if method == "ndt":
            r = O.NDT()
            r.setResolution(2.0)
            r.setStepSize(0.1)
        else:
            r = O.FastGICP() if method == "gicp" else O.GeneralizedIterativeClosestPoint()
            r.setCorrespondenceRandomness(20)
            r.setMaxCorrespondenceDistance(2.0)
            if method == "gicp_omp":
                r.setMaximumOptimizerIterations(20)
        r.setTransformationEpsilon(0.01)
        r.setMaximumIterations(64)
        self.reg, self.clouds, self.poses = r, [], []

    def prefilter(self, cloud):
        pts = np.ascontiguousarray(cloud, np.float32)
        if self.leaf and self.leaf > 0 and len(pts):
            pts = self.O.voxel_grid(pts, self.leaf, range_min=-1.0 if self.range_min is None else self.range_min)["points"]
        if self.sor_mean_k > 0 and len(pts):
            pts = self.O.statistical_outlier_removal(pts, self.sor_mean_k, self.sor_stddev_mul)["points"]
        return self.O.transform_point_cloud(pts, self.E)

    def set_source(self, cloud):
        self.reg.setInputSource(cloud)

    def align(self, T):
        self.reg.align(T)
        return dict(T=self.reg.final_transformation, converged=self.reg.converged, iterations=self.reg.nr_iterations, evaluations=None,
                    trans_probability=getattr(self.reg, "trans_probability", 0.0))

    def push_keyframe(self, cloud, T, accum):
        self.clouds.append(cloud)
        self.poses.append(np.asarray(T, np.float32).copy())
        return len(self.clouds) - 1

    def set_target(self, ids):
        self.reg.setInputTarget(self.O.assemble_submap(self.clouds, self.poses, ids))


def make_drive(n_frames, n_azimuth=900, spacing=0.4, seed=None, device="cuda"):
    """A recorded drive for the tests: synth.long_drive sweeps (sensor frame, invalid rays as zeros) `spacing` metres apart,
    as a CUDA tensor (n_frames, rays, 4), with the true poses."""
    from lidar_graph_slam_b200 import synth
    kw = {} if seed is None else dict(seed=seed)
    return synth.long_drive(n_frames, device=device, n_azimuth=n_azimuth, spacing=spacing, **kw)
