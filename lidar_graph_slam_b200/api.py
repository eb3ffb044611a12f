"""Host-side mirror of the reference's call surface for the LiDAR front-end hot path.

Class and method names follow pcl::VoxelGrid / pcl::Registration as the reference uses them
(SURVEY.md section 8b): `VoxelGrid.setLeafSize/setInputCloud/filter` (PPF:118-120, GBS:311-313),
`NormalDistributionsTransform` (LSM:56-72) and `FastGICP` (LSM:38-54) with `setInputTarget / setInputSource /
align / hasConverged / getFinalTransformation / getFitnessScore`.  Everything computes in liblgs_b200.so on the GPU.

Clouds are numpy float32 arrays of shape (N, 4) [x, y, z, intensity] (16-byte records) or (N, 8) (the 32-byte
pcl::PointXYZI layout), or CUDA torch tensors of shape (N, 4) for the device-resident variants.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import (AlignResult, BatchDistInfo, BatchParams, NdtGridInfo, OdometryDistInfo, OdometryFrame, OdometryParams, Pc2Layout, SorInfo,
                   VoxelGridInfo, check)

NDT_KDTREE, NDT_DIRECT26, NDT_DIRECT7, NDT_DIRECT1 = 0, 1, 2, 3
REG_NONE, REG_MIN_EIG, REG_NORMALIZED_MIN_EIG, REG_PLANE, REG_FROBENIUS = 0, 1, 2, 3, 4
METHOD_NDT, METHOD_GICP, METHOD_ICP, METHOD_GICP_OMP = 0, 1, 2, 3
VG_OK, VG_REFUSED_OVERFLOW = 0, 1
DBL_MAX = float(np.finfo(np.float64).max)


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _host_cloud(pts):
    a = np.ascontiguousarray(pts, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4, 8):
        raise ValueError("cloud must be (N,3), (N,4) xyzi or (N,8) PointXYZI float32")
    return a, a.ctypes.data_as(C.c_void_p), a.shape[0], a.shape[1] * 4


def _dev_cloud(t, ctx=None):
    """Device-resident cloud.  The library works on the context's stream: when that is not torch's current stream
    (the default context owns a non-blocking stream), torch's pending work on the tensor is waited for first."""
    if not (t.is_cuda and t.dim() == 2 and t.shape[1] == 4 and t.is_contiguous() and str(t.dtype) == "torch.float32"):
        raise ValueError("device cloud must be a contiguous CUDA float32 tensor of shape (N, 4)")
    if ctx is not None and not ctx.shares_torch_stream(t.device):
        import torch
        torch.cuda.current_stream(t.device).synchronize()
    return C.c_void_p(t.data_ptr()), t.shape[0]


class _CudaArray:
    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": "<f4", "data": (int(ptr), False), "version": 2}


def _device_view(ptr, n, device):
    """torch view of a library-owned packed xyzi device cloud (no copy)."""
    import torch
    return torch.as_tensor(_CudaArray(ptr, (int(n), 4)), device="cuda:%d" % device)


def _mat_to_c(T):
    if T is None:
        return None, None
    a = np.asarray(T, dtype=np.float32).reshape(4, 4).ravel(order="F").copy()
    return a, a.ctypes.data_as(C.c_void_p)


def _result_T(res):
    return np.array(res.T, dtype=np.float32).reshape(4, 4, order="F")


class Context:
    """One CUDA device + one stream (include/lgs_c.h lgs_ctx).  stream: a raw cudaStream_t handle or None."""

    def __init__(self, device=0, stream=None):
        self._L = _lib.load()
        h = C.c_void_p()
        check(self._L.lgs_ctx_create(int(device), C.c_void_p(stream) if stream else None, C.byref(h)))
        self._h = h
        self.device = device
        self.stream = int(stream) if stream else None

    def shares_torch_stream(self, device=None):
        """True when the context runs on torch's current stream (stream-ordered with torch work, no sync needed)."""
        if self.stream is None:
            return False
        import torch
        return torch.cuda.current_stream(device).cuda_stream == self.stream

    def synchronize(self):
        check(self._L.lgs_ctx_synchronize(self._h))

    @property
    def launch_count(self):
        return int(self._L.lgs_ctx_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._L.lgs_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


PC2_INT8, PC2_UINT8, PC2_INT16, PC2_UINT16, PC2_INT32, PC2_UINT32, PC2_FLOAT32, PC2_FLOAT64 = range(1, 9)


def from_pointcloud2(data, width, height, point_step, fields, row_step=0, is_bigendian=False, ctx=None):
    """pcl::fromROSMsg<pcl::PointXYZI> on the GPU (PPF:65-70): `data` is the message's byte payload, `fields` maps a
    field name to (offset, datatype) as in sensor_msgs/PointField.  Returns a CUDA float32 tensor (N, 4) xyzi that the
    device-resident entry points take (VoxelGrid / StatisticalOutlierRemoval / setInputSource / setInputTarget)."""
    import torch
    ctx = ctx or default_context()
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data).view(np.uint8).ravel()
    n = int(width) * int(height)
    if buf.size < n * int(point_step):
        raise ValueError("payload shorter than width * height * point_step")
    L = Pc2Layout()
    L.width, L.height, L.point_step, L.row_step = int(width), int(height), int(point_step), int(row_step)
    for name in ("x", "y", "z"):
        if name not in fields:
            raise ValueError("PointCloud2 has no field %r" % name)
    L.offset_x, L.offset_y, L.offset_z = (int(fields[k][0]) for k in ("x", "y", "z"))
    dts = {int(fields[k][1]) for k in ("x", "y", "z")}
    L.datatype_xyz = dts.pop() if len(dts) == 1 else 0
    L.offset_intensity, L.datatype_intensity = (int(fields["intensity"][0]), int(fields["intensity"][1])) if "intensity" in fields else (-1, 0)
    L.is_bigendian = 1 if is_bigendian else 0
    out = torch.empty((max(n, 1), 4), dtype=torch.float32, device="cuda:%d" % ctx.device)
    if not ctx.shares_torch_stream(out.device):
        torch.cuda.current_stream(out.device).synchronize()
    cnt = C.c_int64()
    check(ctx._L.lgs_cloud_from_pointcloud2(ctx._h, buf.ctypes.data_as(C.c_void_p), C.byref(L), C.c_void_p(out.data_ptr()), C.byref(cnt)))
    if not ctx.shares_torch_stream(out.device):
        ctx.synchronize()
    return out[:n]


class VoxelGrid:
    """pcl::VoxelGrid<PointXYZI> plus the prefilter's crop predicates (PPF:89-121)."""

    def __init__(self, ctx=None):
        self.ctx = ctx or default_context()
        self._L = self.ctx._L
        self._leaf = np.array([0.01, 0.01, 0.01], np.float32)
        self._min_pts = 0
        self._range_min = -1.0
        self._box = None
        self._cloud = None
        self.info = None
        self.voxel_idx = None
        self.member_rank = None

    def setLeafSize(self, lx, ly=None, lz=None):
        ly = lx if ly is None else ly
        lz = lx if lz is None else lz
        self._leaf = np.array([lx, ly, lz], dtype=np.float32)  # double -> float as VoxelGrid::setLeafSize(float,...)

    def setMinimumPointsNumberPerVoxel(self, n):
        self._min_pts = int(n)

    def setRangeCrop(self, min_distance):
        """distance_filter of the prefilter node (PPF:102-112); None disables."""
        self._range_min = -1.0 if min_distance is None else float(min_distance)

    def setBoxCrop(self, box6):
        """crop of the prefilter node (PPF:89-100): (min_x, max_x, min_y, max_y, min_z, max_z) or None."""
        self._box = None if box6 is None else np.asarray(box6, dtype=np.float64).copy()

    def setInputCloud(self, cloud):
        self._cloud = cloud

    def filter(self, want_membership=True):
        """Returns the downsampled cloud (M, 4).  Per-point voxel_idx / member_rank land in attributes."""
        leaf_p = self._leaf.ctypes.data_as(C.c_void_p)
        box_p = self._box.ctypes.data_as(C.c_void_p) if self._box is not None else None
        info = VoxelGridInfo()
        if _is_torch(self._cloud):
            import torch
            p, n = _dev_cloud(self._cloud, self.ctx)
            out = torch.empty((max(n, 1), 4), dtype=torch.float32, device=self._cloud.device)
            vidx = torch.empty(max(n, 1), dtype=torch.int32, device=self._cloud.device) if want_membership else None
            rank = torch.empty(max(n, 1), dtype=torch.int32, device=self._cloud.device) if want_membership else None
            check(self._L.lgs_voxelgrid_filter_dev(self.ctx._h, p, n, leaf_p, self._min_pts, self._range_min, box_p, C.c_void_p(out.data_ptr()),
                                                   C.c_void_p(vidx.data_ptr()) if want_membership else None,
                                                   C.c_void_p(rank.data_ptr()) if want_membership else None, C.byref(info)))
            if not self.ctx.shares_torch_stream(self._cloud.device):
                self.ctx.synchronize()  # outputs are written on the context's stream; torch reads them on its own
            self.info = info
            self.voxel_idx = vidx[:n] if want_membership else None
            self.member_rank = rank[:n] if want_membership else None
            return out[: info.n_out]
        a, p, n, stride = _host_cloud(self._cloud)
        out = np.empty((max(n, 1), 4), np.float32)
        vidx = np.empty(max(n, 1), np.int32) if want_membership else None
        rank = np.empty(max(n, 1), np.int32) if want_membership else None
        check(self._L.lgs_voxelgrid_filter(self.ctx._h, p, n, stride, leaf_p, self._min_pts, self._range_min, box_p,
                                           out.ctypes.data_as(C.c_void_p), vidx.ctypes.data_as(C.c_void_p) if want_membership else None,
                                           rank.ctypes.data_as(C.c_void_p) if want_membership else None, C.byref(info)))
        self.info = info
        self.voxel_idx = vidx[:n] if want_membership else None
        self.member_rank = rank[:n] if want_membership else None
        return out[: info.n_out].copy()


class StatisticalOutlierRemoval:
    """pcl::StatisticalOutlierRemoval<PointXYZI> as the prefilter node drives it right after the voxel grid
    (PPF:79-80,132-140)."""

    def __init__(self, ctx=None):
        self.ctx = ctx or default_context()
        self._L = self.ctx._L
        h = C.c_void_p()
        check(self._L.lgs_sor_create(self.ctx._h, C.byref(h)))
        self._h = h
        self._cloud = None
        self.info = None
        self.keep = None
        self.distances = None

    def setMeanK(self, k): check(self._L.lgs_sor_set_mean_k(self._h, int(k)))
    def setStddevMulThresh(self, m): check(self._L.lgs_sor_set_stddev_mul_thresh(self._h, float(m)))
    def setNegative(self, negative): check(self._L.lgs_sor_set_negative(self._h, 1 if negative else 0))
    def setInputCloud(self, cloud): self._cloud = cloud

    def filter(self):
        """Returns the kept points (M, 4) in input order; the per-point decision and mean neighbour distance land in
        the attributes `keep` and `distances`."""
        info = SorInfo()
        if _is_torch(self._cloud):
            import torch
            p, n = _dev_cloud(self._cloud, self.ctx)
            dev = self._cloud.device
            out = torch.empty((max(n, 1), 4), dtype=torch.float32, device=dev)
            keep = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
            dist = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
            check(self._L.lgs_sor_filter_dev(self._h, p, n, C.c_void_p(out.data_ptr()), C.c_void_p(keep.data_ptr()), C.c_void_p(dist.data_ptr()),
                                             C.byref(info)))
            if not self.ctx.shares_torch_stream(dev):
                self.ctx.synchronize()
            self.info, self.keep, self.distances = info, keep[:n].bool(), dist[:n]
            return out[: info.n_out]
        a, p, n, stride = _host_cloud(self._cloud)
        out = np.empty((max(n, 1), 4), np.float32)
        keep = np.empty(max(n, 1), np.uint8)
        dist = np.empty(max(n, 1), np.float32)
        vp = lambda x: x.ctypes.data_as(C.c_void_p)
        check(self._L.lgs_sor_filter(self._h, p, n, stride, vp(out), vp(keep), vp(dist), C.byref(info)))
        self.info, self.keep, self.distances = info, keep[:n].astype(bool), dist[:n]
        return out[: info.n_out].copy()

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._L.lgs_sor_destroy(self._h)
                self._h = None
        except Exception:
            pass


class _Registration:
    """Shared pcl::Registration surface."""

    _prefix = ""

    def __init__(self, ctx=None):
        self.ctx = ctx or default_context()
        self._L = self.ctx._L
        h = C.c_void_p()
        check(self._fn("create")(self.ctx._h, C.byref(h)))
        self._h = h
        self._ns = self._nt = 0

    def _fn(self, name):
        return getattr(self._L, "lgs_%s_%s" % (self._prefix, name))

    def _set_cloud(self, which, cloud):
        if _is_torch(cloud):
            p, n = _dev_cloud(cloud, self.ctx)
            check(self._fn("set_%s_dev" % which)(self._h, p, n))
            if not self.ctx.shares_torch_stream(cloud.device):
                # the library copies the tensor on its own stream, which torch's caching allocator does not know: finish the
                # copy before the caller can drop the tensor and have its memory recycled
                self.ctx.synchronize()
        else:
            _, p, n, stride = _host_cloud(cloud)
            check(self._fn("set_%s" % which)(self._h, p, n, stride))
        return n

    def setInputTarget(self, cloud):
        self._nt = self._set_cloud("target", cloud)

    def setInputSource(self, cloud):
        self._ns = self._set_cloud("source", cloud)

    def align(self, guess=None, want_output=False, out=None):
        """Runs the registration (pcl::Registration::align(output, guess)).  Returns the aligned source cloud when want_output
        (written into `out`, a C-contiguous float32 (>= n_source, 4) host array, when the caller supplies one), else None."""
        keep, gp = _mat_to_c(guess)
        res = AlignResult()
        if want_output and out is None:
            out = np.empty((max(self._ns, 1), 4), np.float32)
        if want_output:
            assert out.dtype == np.float32 and out.flags["C_CONTIGUOUS"] and out.shape[0] >= self._ns and out.shape[1] == 4
        check(self._fn("align")(self._h, gp, C.byref(res), out.ctypes.data_as(C.c_void_p) if want_output else None))
        self.result = res
        self.final_transformation = _result_T(res)
        return out[: self._ns] if want_output else None

    def hasConverged(self):
        return bool(self.result.converged)

    def getFinalTransformation(self):
        return self.final_transformation

    def getFitnessScore(self, max_range=DBL_MAX):
        f = C.c_double()
        check(self._fn("fitness")(self._h, float(max_range), C.byref(f)))
        return f.value

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._fn("destroy")(self._h)
                self._h = None
        except Exception:
            pass


class NormalDistributionsTransform(_Registration):
    """pclomp::NormalDistributionsTransform (NDT.h:71-502)."""

    _prefix = "ndt"

    def __init__(self, ctx=None):
        super().__init__(ctx)
        self._resolution, self._step, self._outlier = 1.0, 0.1, 0.55

    def setResolution(self, r): check(self._L.lgs_ndt_set_resolution(self._h, float(r))); self._resolution = float(r)
    def getResolution(self): return self._resolution
    def setStepSize(self, s): check(self._L.lgs_ndt_set_step_size(self._h, float(s))); self._step = float(s)
    def getStepSize(self): return self._step
    def setOutlierRatio(self, o): check(self._L.lgs_ndt_set_outlier_ratio(self._h, float(o))); self._outlier = float(o)
    def getOutlierRatio(self): return self._outlier
    def setTransformationEpsilon(self, e): check(self._L.lgs_ndt_set_transformation_epsilon(self._h, float(e)))
    def setMaximumIterations(self, n): check(self._L.lgs_ndt_set_maximum_iterations(self._h, int(n)))
    def setNeighborhoodSearchMethod(self, m): check(self._L.lgs_ndt_set_search_method(self._h, int(m)))

    def setExactNewtonStep(self, on):
        """Parity mode: every Newton step through the restated JacobiSVD of the reference instead of the block elimination."""
        check(self._L.lgs_ndt_set_exact_newton_step(self._h, 1 if on else 0))

    def setNumThreads(self, n): pass  # OpenMP knob of the reference (NDT.h:113-115); meaningless on the GPU

    @staticmethod
    def convertTransform(x):
        """static convertTransform (NDT.h:214-238): (x, y, z, roll, pitch, yaw) -> 4x4 float32."""
        x = np.ascontiguousarray(x, np.float64)
        T = np.empty(16, np.float32)
        check(_lib.load().lgs_ndt_convert_transform(x.ctypes.data_as(C.c_void_p), T.ctypes.data_as(C.c_void_p)))
        return T.reshape(4, 4, order="F").copy()

    def getTransformationProbability(self): return self.result.trans_probability
    def getFinalNumIteration(self): return int(self.result.iterations)

    def calculateScore(self, T):
        keep, tp = _mat_to_c(T)
        s = C.c_double()
        check(self._L.lgs_ndt_calculate_score(self._h, tp, C.byref(s)))
        return s.value

    def profile(self, enable):
        """Measurement hook: returns the CUDA-event timings gathered so far and (re)arms / disarms timing.  enable = 1 (True):
        one launch per evaluation (the host steps the optimiser), each launch timed; enable = 2: the device-resident align
        (one ndt_align_kernel launch per align) timed as a whole.  The returned dict describes the mode that WAS armed."""
        was = getattr(self, "_profiling", 0)
        out = np.zeros(8)
        check(self._L.lgs_ndt_profile(self._h, int(enable), out.ctypes.data_as(C.c_void_p)))
        self._profiling = int(enable)
        if was == 2:
            return dict(align_launches=int(out[0]), align_ms=out[1], evaluations=out[2], terms=out[3], terms_last_eval=out[6], n_source=int(out[7]))
        return dict(hess_launches=int(out[0]), hess_ms=out[1], grad_launches=int(out[2]), grad_ms=out[3], h64_launches=int(out[4]),
                    h64_ms=out[5], terms_last_eval=out[6], n_source=int(out[7]))

    def setInputTargetKeyFrames(self, kf, ids):
        """The rolling local map (LSM:187-212) as a list of key frames of a device-resident KeyFrameArray, maintained
        incrementally (lgs_ndt_set_target_keyframes).  Returns the number of key frames voxelised from their points."""
        ids = np.ascontiguousarray(ids, np.int32)
        nv = C.c_int32()
        check(self._L.lgs_ndt_set_target_keyframes(self._h, kf._h, ids.ctypes.data_as(C.c_void_p), int(ids.size), C.byref(nv)))
        self._nt = -1
        return nv.value

    def align_guesses(self, guesses, fitness_max_range=None):
        """One map, many seeds: align this source from every 4x4 guess in one resident launch per wave (ndt_align_many).
        Record k is bit-identical to align(guesses[k]); afterwards the object holds the last guess's result."""
        return ndt_align_many([self] * len(guesses), guesses, fitness_max_range)

    def align_breakdown(self):
        """SM cycles CTA 0 spent per phase of the last device-resident align (lgs_ndt_align_breakdown)."""
        out = np.zeros(16)
        check(self._L.lgs_ndt_align_breakdown(self._h, out.ctypes.data_as(C.c_void_p)))
        return dict(evaluate=out[0], wait_grid=out[1], add_rows=out[2], optimiser=out[3], publish=out[4], total=out[5],
                    opt_decide=out[8], opt_solve=out[9], opt_after_solve=out[10], opt_trig=out[11], opt_pose_tables=out[12], raw=out.tolist())

    # parity hooks -------------------------------------------------------------------------------
    def grid_info(self):
        gi = NdtGridInfo()
        check(self._L.lgs_ndt_grid_info_get(self._h, C.byref(gi)))
        return gi

    def export_voxels(self):
        gi = self.grid_info()
        v = int(gi.n_voxels)
        idx, npts = np.empty(v, np.int32), np.empty(v, np.int32)
        mean, cov, icov = np.empty((v, 3)), np.empty((v, 9)), np.empty((v, 9))
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        check(self._L.lgs_ndt_export_voxels(self._h, vp(idx), vp(npts), vp(mean), vp(cov), vp(icov)))
        return dict(idx=idx, n=npts, mean=mean, cov=cov, icov=icov, min_b=np.array(gi.min_b), max_b=np.array(gi.max_b),
                    div_b=np.array(gi.div_b), refused=bool(gi.refused), dense=bool(gi.dense), n_valid=int(gi.n_valid))

    def derivatives(self, T, p, mode=0):
        keep, tp = _mat_to_c(T)
        p = np.asarray(p, np.float64).copy()
        s = C.c_double()
        g, H = np.zeros(6), np.zeros(36)
        check(self._L.lgs_ndt_derivatives(self._h, tp, p.ctypes.data_as(C.c_void_p), int(mode), C.byref(s), g.ctypes.data_as(C.c_void_p),
                                          H.ctypes.data_as(C.c_void_p)))
        return s.value, g, H.reshape(6, 6)


class FastGICP(_Registration):
    """fast_gicp::FastGICP (fast_gicp.hpp:48-70 over lsq_registration.hpp:48-60)."""

    _prefix = "gicp"

    def setCorrespondenceRandomness(self, k): check(self._L.lgs_gicp_set_correspondence_randomness(self._h, int(k)))
    def setMaxCorrespondenceDistance(self, d): check(self._L.lgs_gicp_set_max_correspondence_distance(self._h, float(d)))
    def setTransformationEpsilon(self, e): check(self._L.lgs_gicp_set_transformation_epsilon(self._h, float(e)))
    def setRotationEpsilon(self, e): check(self._L.lgs_gicp_set_rotation_epsilon(self._h, float(e)))
    def setMaximumIterations(self, n): check(self._L.lgs_gicp_set_maximum_iterations(self._h, int(n)))
    def setRegularizationMethod(self, m): check(self._L.lgs_gicp_set_regularization_method(self._h, int(m)))
    def setInitialLambdaFactor(self, f): check(self._L.lgs_gicp_set_initial_lambda_factor(self._h, float(f)))
    def setNumThreads(self, n): pass

    def swapSourceAndTarget(self):
        check(self._L.lgs_gicp_swap_source_and_target(self._h))
        self._ns, self._nt = self._nt, self._ns

    def clearSource(self): check(self._L.lgs_gicp_clear_source(self._h)); self._ns = 0
    def clearTarget(self): check(self._L.lgs_gicp_clear_target(self._h)); self._nt = 0

    def getFinalHessian(self):
        H = np.empty(36)
        check(self._L.lgs_gicp_final_hessian(self._h, H.ctypes.data_as(C.c_void_p)))
        return H.reshape(6, 6)

    def covariances(self, which):
        n = self._ns if which == 0 else self._nt
        c = np.empty((n, 9))
        check(self._L.lgs_gicp_export_covariances(self._h, int(which), c.ctypes.data_as(C.c_void_p)))
        return c.reshape(n, 3, 3)

    def setDebugPrint(self, flag): pass  # lsq_registration.hpp:36: console output of the LM steps; nothing to print here

    def evaluateCost(self, relative_pose):
        """LsqRegistration::evaluateCost (LSQ:48-50): cost at a pose over the correspondences of the last linearisation."""
        keep, tp = _mat_to_c(relative_pose)
        cost = C.c_double()
        check(self._L.lgs_gicp_evaluate_cost(self._h, tp, C.byref(cost)))
        return cost.value

    def _set_covariances(self, which, covs):
        c = np.ascontiguousarray(np.asarray(covs, np.float64).reshape(-1, 9))
        check(self._L.lgs_gicp_set_covariances(self._h, which, c.ctypes.data_as(C.c_void_p), c.shape[0]))

    def setSourceCovariances(self, covs): self._set_covariances(0, covs)
    def setTargetCovariances(self, covs): self._set_covariances(1, covs)
    def getSourceCovariances(self): return self.covariances(0)
    def getTargetCovariances(self): return self.covariances(1)

    def linearize(self, T):
        Tr = np.ascontiguousarray(np.asarray(T, np.float64).reshape(4, 4))
        cost = C.c_double()
        H, b = np.zeros(36), np.zeros(6)
        corr = np.empty(max(self._ns, 1), np.int32)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        check(self._L.lgs_gicp_linearize(self._h, vp(Tr), C.byref(cost), vp(H), vp(b), vp(corr)))
        return cost.value, H.reshape(6, 6), b, corr[: self._ns]


class GeneralizedIterativeClosestPoint(_Registration):
    """pclomp::GeneralizedIterativeClosestPoint (gicp_omp.h:116-270; BFGS), the "GICP" method of LSM:73-96 / GBS:120-141."""

    _prefix = "gicp_omp"

    def setCorrespondenceRandomness(self, k): check(self._L.lgs_gicp_omp_set_correspondence_randomness(self._h, int(k)))
    def setMaxCorrespondenceDistance(self, d): check(self._L.lgs_gicp_omp_set_max_correspondence_distance(self._h, float(d)))
    def setTransformationEpsilon(self, e): check(self._L.lgs_gicp_omp_set_transformation_epsilon(self._h, float(e)))
    def setRotationEpsilon(self, e): check(self._L.lgs_gicp_omp_set_rotation_epsilon(self._h, float(e)))
    def setMaximumIterations(self, n): check(self._L.lgs_gicp_omp_set_maximum_iterations(self._h, int(n)))
    def setMaximumOptimizerIterations(self, n): check(self._L.lgs_gicp_omp_set_maximum_optimizer_iterations(self._h, int(n)))
    # accepted and ignored, as by the reference's computeTransformation (GO:370-516 never reads them)
    def setUseReciprocalCorrespondences(self, flag): pass
    def setEuclideanFitnessEpsilon(self, e): pass
    def setRANSACIterations(self, n): pass
    def setNumThreads(self, n): pass

    def covariances(self, which):
        n = self._ns if which == 0 else self._nt
        c = np.empty((n, 9))
        check(self._L.lgs_gicp_omp_export_covariances(self._h, int(which), c.ctypes.data_as(C.c_void_p)))
        return c.reshape(n, 3, 3)

    def functor(self, guess, transformation, x):
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        gc = np.asarray(guess, np.float32).reshape(4, 4).ravel(order="F").copy()
        tc = np.asarray(transformation, np.float32).reshape(4, 4).ravel(order="F").copy()
        x = np.ascontiguousarray(x, np.float64)
        out = np.zeros(15)
        corr = np.empty(max(self._ns, 1), np.int32)
        mahal = np.empty((max(self._ns, 1), 9), np.float32)
        check(self._L.lgs_gicp_omp_functor(self._h, vp(gc), vp(tc), vp(x), vp(out), vp(corr), vp(mahal)))
        return dict(f=out[0], df=out[1:7].copy(), fdf_f=out[7], fdf_g=out[8:14].copy(), n_corr=int(out[14]), corr=corr[: self._ns],
                    mahal=mahal[: self._ns])


class KeyFrameArray:
    """Device-resident key_frame_array_ of the scan matcher / graph SLAM nodes (LSM:196-212, GBS:297-313): key frames are
    uploaded once; `assemble` returns the transformed, concatenated (and optionally voxel-filtered) sub-map as a CUDA
    tensor that setInputTarget takes without leaving the GPU."""

    def __init__(self, ctx=None):
        self.ctx = ctx or default_context()
        self._L = self.ctx._L
        h = C.c_void_p()
        check(self._L.lgs_keyframes_create(self.ctx._h, C.byref(h)))
        self._h = h

    def push(self, cloud, pose):
        _, pp = _mat_to_c(pose)
        kid = C.c_int32()
        if _is_torch(cloud):
            p, n = _dev_cloud(cloud, self.ctx)
            check(self._L.lgs_keyframes_push_dev(self._h, p, n, pp, C.byref(kid)))
        else:
            _, p, n, stride = _host_cloud(cloud)
            check(self._L.lgs_keyframes_push(self._h, p, n, stride, pp, C.byref(kid)))
        return kid.value

    def set_pose(self, kid, pose):
        _, pp = _mat_to_c(pose)
        check(self._L.lgs_keyframes_set_pose(self._h, int(kid), pp))

    def __len__(self):
        c = C.c_int64()
        check(self._L.lgs_keyframes_size(self._h, C.byref(c), None))
        return c.value

    def set_position(self, kid, xyz):
        """key_frame.pose.position in f64 (what detect_loop_with_accum_dist compares, GBS:163-171)."""
        p = np.ascontiguousarray(xyz, np.float64)
        check(self._L.lgs_keyframes_set_position(self._h, int(kid), p.ctypes.data_as(C.c_void_p)))

    def set_accum_distance(self, kid, accum_distance):
        check(self._L.lgs_keyframes_set_accum_distance(self._h, int(kid), float(accum_distance)))

    def detect_loop(self, latest_id, accumulate_distance_threshold=100.0, search_for_candidate_threshold=15.0):
        """detect_loop_with_accum_dist (GBS:157-187; defaults of graph_based_slam.param.yaml): (candidate ids, nearest id or -1)."""
        cap = max(len(self), 1)
        cand = np.empty(cap, np.int32)
        n, best = C.c_int32(), C.c_int32()
        check(self._L.lgs_keyframes_detect_loop(self._h, int(latest_id), float(accumulate_distance_threshold), float(search_for_candidate_threshold),
                                                cand.ctypes.data_as(C.c_void_p), cap, C.byref(n), C.byref(best)))
        return cand[: n.value].copy(), best.value

    def batch_align(self, scan_ids, center_ids, search_key_frame_num=20, method=METHOD_GICP, guesses=None, pair_id0=0, records_dev=None,
                    max_iterations=100, transformation_epsilon=0.01, max_correspondence_distance=2.0, k_correspondences=20, ndt_resolution=1.0,
                    ndt_step_size=0.1, submap_leaf=0.5, fitness_max_range=-1.0, n_workers=0, max_optimizer_iterations=0, euclidean_fitness_epsilon=0.0):
        """Loop-closure verification of (key frame, neighbourhood) candidates without leaving the GPU (lgs_batch_align_keyframes)."""
        sid = np.ascontiguousarray(scan_ids, np.int32)
        cid = np.ascontiguousarray(center_ids, np.int32)
        n = int(sid.size)
        assert cid.size == n
        g = _pack_guesses(guesses)
        bp = _batch_params(method, max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution,
                           ndt_step_size, submap_leaf, fitness_max_range, n_workers, max_optimizer_iterations, euclidean_fitness_epsilon)
        recs = (AlignResult * max(n, 1))()
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        check(self._L.lgs_batch_align_keyframes(self._h, None, C.byref(bp), n, vp(sid), vp(cid), int(search_key_frame_num),
                                                vp(g) if g is not None else None, int(pair_id0), recs, C.c_void_p(records_dev) if records_dev else None))
        return [recs[i] for i in range(n)]

    def batch_align_dist(self, comm, scan_ids, center_ids, search_key_frame_num=20, method=METHOD_GICP, guesses=None, max_iterations=100,
                         transformation_epsilon=0.01, max_correspondence_distance=2.0, k_correspondences=20, ndt_resolution=1.0, ndt_step_size=0.1,
                         submap_leaf=0.5, fitness_max_range=-1.0, n_workers=0, max_optimizer_iterations=0, euclidean_fitness_epsilon=0.0):
        """lgs_batch_align_keyframes_dist (collective over `comm`): the candidate list is the same on every rank, each rank
        verifies its share from its own resident key-frame array, one ncclAllGather returns all records everywhere."""
        sid = np.ascontiguousarray(scan_ids, np.int32)
        cid = np.ascontiguousarray(center_ids, np.int32)
        n = int(sid.size)
        assert cid.size == n
        g = _pack_guesses(guesses)
        bp = _batch_params(method, max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution,
                           ndt_step_size, submap_leaf, fitness_max_range, n_workers, max_optimizer_iterations, euclidean_fitness_epsilon)
        recs = (AlignResult * max(n, 1))()
        info = BatchDistInfo()
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        check(self._L.lgs_batch_align_keyframes_dist(self._h, comm._h, C.byref(bp), n, vp(sid), vp(cid), int(search_key_frame_num),
                                                     vp(g) if g is not None else None, recs, C.byref(info)))
        return [recs[i] for i in range(n)], _dist_info(info)

    def assemble(self, ids, leaf=0.0):
        """Returns a CUDA float32 tensor (N, 4): a copy of the library's sub-map buffer."""
        import torch
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        out, n = C.c_void_p(), C.c_int64()
        check(self._L.lgs_keyframes_assemble(self._h, ids.ctypes.data_as(C.c_void_p), int(ids.size), float(leaf), C.byref(out), C.byref(n)))
        self.ctx.synchronize()
        t = torch.empty((n.value, 4), dtype=torch.float32, device="cuda:%d" % self.ctx.device)
        if n.value:
            t.copy_(_device_view(out.value, n.value, self.ctx.device))
            torch.cuda.current_stream(t.device).synchronize()
        return t

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._L.lgs_keyframes_destroy(self._h)
                self._h = None
        except Exception:
            pass


class IterativeClosestPoint(_Registration):
    """pcl::IterativeClosestPoint<PointXYZI, PointXYZI>, the graph SLAM node's default loop-closure method (GBS:142-151)."""

    _prefix = "icp"

    def setMaxCorrespondenceDistance(self, d): check(self._L.lgs_icp_set_max_correspondence_distance(self._h, float(d)))
    def setMaximumIterations(self, n): check(self._L.lgs_icp_set_maximum_iterations(self._h, int(n)))
    def setTransformationEpsilon(self, e): check(self._L.lgs_icp_set_transformation_epsilon(self._h, float(e)))
    def setTransformationRotationEpsilon(self, e): check(self._L.lgs_icp_set_transformation_rotation_epsilon(self._h, float(e)))
    def setEuclideanFitnessEpsilon(self, e): check(self._L.lgs_icp_set_euclidean_fitness_epsilon(self._h, float(e)))
    def setRANSACIterations(self, n): pass  # GBS:149; PCL's ICP installs no rejector by default, the value is never read

    def step(self, guess):
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        gc = np.asarray(guess, np.float32).reshape(4, 4).ravel(order="F").copy()
        sums, T, ok = np.zeros(17), np.zeros(16, np.float32), C.c_int32()
        check(self._L.lgs_icp_step(self._h, vp(gc), vp(sums), vp(T), C.byref(ok)))
        return bool(ok.value), sums, T.reshape(4, 4, order="F").copy()


def ndt_align_many(ndts, guesses=None, fitness_max_range=None, want_output=False):
    """Aligns N NDT problems in one resident launch per wave (lgs_ndt_align_many): ndts[i] from guesses[i] (4x4, or identity
    when guesses is None).  Handles may repeat and must share one Context.  Each record is bit-identical to ndts[i].align(
    guesses[i]) run alone, and every object ends with the result and final transformation of its last occurrence, as after
    those calls in order.  fitness_max_range: records[i].fitness = getFitnessScore(fitness_max_range) at record i's
    transform.  Returns the list of records, or (records, aligned clouds) when want_output."""
    n = len(ndts)
    if guesses is not None and len(guesses) != n:
        raise ValueError("need one guess per problem")
    L = _lib.load()
    hs = (C.c_void_p * max(n, 1))(*[x._h.value for x in ndts])
    g = _pack_guesses(guesses) if n else None
    recs = (AlignResult * max(n, 1))()
    fmr = C.c_double(float(fitness_max_range)) if fitness_max_range is not None else None
    outs = [np.empty((max(x._ns, 1), 4), np.float32) for x in ndts] if want_output else None
    op = (C.c_void_p * max(n, 1))(*[o.ctypes.data for o in outs]) if want_output else None
    check(L.lgs_ndt_align_many(hs, n, g.ctypes.data_as(C.c_void_p) if g is not None else None, C.byref(fmr) if fmr is not None else None,
                               recs, op))
    out = [recs[i] for i in range(n)]
    for x, r in zip(ndts, out):
        x.result = r
        x.final_transformation = _result_T(r)
    if want_output:
        return out, [o[: x._ns] for o, x in zip(outs, ndts)]
    return out


def knn(pts, queries, k, ctx=None):
    """Exact k-NN of `queries` in `pts` (the search behind FG:133 / FG:254).  Returns (idx (m,k) int32, d2 (m,k) f32)."""
    ctx = ctx or default_context()
    a, pa, n, sa = _host_cloud(pts)
    q, pq, m, sq = _host_cloud(queries)
    idx = np.empty((max(m, 1), k), np.int32)
    d2 = np.empty((max(m, 1), k), np.float32)
    check(ctx._L.lgs_knn(ctx._h, pa, n, sa, pq, m, sq, int(k), idx.ctypes.data_as(C.c_void_p), d2.ctypes.data_as(C.c_void_p)))
    return idx[:m], d2[:m]


def nn_search1(pts, queries, seeds=None, ctx=None):
    """Exact 1-NN of `queries` in `pts` by the search of the correspondence steps (FG:133, ICP), started from seeds[t] (an
    index into pts; outside [0, n) = no seed) or unseeded when seeds is None.  Returns (idx (m,) int32, d2 (m,) f32);
    idx -1 and d2 +inf for an empty cloud."""
    ctx = ctx or default_context()
    a, pa, n, sa = _host_cloud(pts)
    q, pq, m, sq = _host_cloud(queries)
    s = None
    if seeds is not None:
        s = np.ascontiguousarray(seeds, dtype=np.int32).ravel()
        if s.size != m:
            raise ValueError("need one seed per query")
    idx = np.empty(max(m, 1), np.int32)
    d2 = np.empty(max(m, 1), np.float32)
    vp = lambda x: x.ctypes.data_as(C.c_void_p)
    check(ctx._L.lgs_nn_search1(ctx._h, pa, n, sa, pq, m, sq, vp(s) if s is not None else None, vp(idx), vp(d2)))
    return idx[:m], d2[:m]


def sort_pairs(keys, vals, bits=32, ctx=None):
    """Stable device radix sort of (uint32 key, uint32 value) pairs by the low `bits` key bits (parity hook for the
    sort that orders points by voxel).  Returns sorted copies."""
    ctx = ctx or default_context()
    k = np.array(keys, dtype=np.uint32, copy=True).ravel()
    v = np.array(vals, dtype=np.uint32, copy=True).ravel()
    assert k.shape == v.shape
    check(ctx._L.lgs_sort_pairs(ctx._h, k.ctypes.data_as(C.c_void_p), v.ctypes.data_as(C.c_void_p), k.shape[0], int(bits)))
    return k, v


def batch_align(scans, submaps, method=METHOD_GICP, guesses=None, device=0, stream=None, pair_id0=0, records_dev=None, max_iterations=100,
                transformation_epsilon=0.01, max_correspondence_distance=2.0, k_correspondences=20, ndt_resolution=1.0, ndt_step_size=0.1,
                submap_leaf=0.5, fitness_max_range=-1.0, n_workers=0, max_optimizer_iterations=0, euclidean_fitness_epsilon=0.0):
    """Batched loop-closure verification (GBS:297-322 for a list of pairs).  scans / submaps: lists of (N,4) float32
    numpy arrays.  Returns a numpy structured view of lgs_align_result records."""
    L = _lib.load()
    n = len(scans)
    assert len(submaps) == n
    sc = [np.ascontiguousarray(s, np.float32) for s in scans]
    sm = [np.ascontiguousarray(s, np.float32) for s in submaps]
    sp = (C.c_void_p * n)(*[s.ctypes.data for s in sc])
    mp = (C.c_void_p * n)(*[s.ctypes.data for s in sm])
    ns = (C.c_int64 * n)(*[s.shape[0] for s in sc])
    nm = (C.c_int64 * n)(*[s.shape[0] for s in sm])
    g = _pack_guesses(guesses)
    bp = _batch_params(method, max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution, ndt_step_size,
                       submap_leaf, fitness_max_range, n_workers, max_optimizer_iterations, euclidean_fitness_epsilon)
    recs = (AlignResult * max(n, 1))()
    check(L.lgs_batch_align(int(device), C.c_void_p(stream) if stream else None, C.byref(bp), n, sp, ns, mp, nm, 16,
                            g.ctypes.data_as(C.c_void_p) if g is not None else None, int(pair_id0), recs,
                            C.c_void_p(records_dev) if records_dev else None))
    return [recs[i] for i in range(n)]


def _pack_guesses(guesses):
    """(K, 16) float32 column-major transforms, or None."""
    if guesses is None:
        return None
    return np.ascontiguousarray(np.stack([np.asarray(T, np.float32).reshape(4, 4).ravel(order="F") for T in guesses]))


def _batch_params(method, max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution, ndt_step_size,
                  submap_leaf, fitness_max_range, n_workers, max_optimizer_iterations, euclidean_fitness_epsilon):
    return BatchParams(method=method, max_iterations=max_iterations, transformation_epsilon=transformation_epsilon,
                       max_correspondence_distance=max_correspondence_distance, k_correspondences=k_correspondences,
                       ndt_resolution=ndt_resolution, ndt_step_size=ndt_step_size, submap_leaf=submap_leaf,
                       fitness_max_range=fitness_max_range, n_workers=n_workers, max_optimizer_iterations=max_optimizer_iterations,
                       euclidean_fitness_epsilon=euclidean_fitness_epsilon)


def partition_pairs(sizes, rank, world):
    """lgs_batch_partition: the pair indices rank `rank` of `world` verifies (descending size, dealt round-robin)."""
    L = _lib.load()
    sz = np.ascontiguousarray(sizes, np.int64)
    out = np.empty(max(sz.size, 1), np.int32)
    n = C.c_int64()
    check(L.lgs_batch_partition(sz.ctypes.data_as(C.c_void_p), int(sz.size), int(rank), int(world), out.ctypes.data_as(C.c_void_p), int(out.size), C.byref(n)))
    return out[: n.value].tolist()


def _prefer_bundled_nccl():
    """liblgs_b200.so binds NCCL at run time (dlopen).  In a Python process that also imports PyTorch the copy PyTorch ships
    (site-packages/nvidia/nccl) must be the one that gets loaded: a different libnccl.so.2 loaded first would satisfy
    PyTorch's own dependency by soname and miss symbols it needs.  Points LGS_NCCL_LIB at the bundled file if there is one."""
    import os
    if os.environ.get("LGS_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for d in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
            cand = os.path.join(d, "lib", "libnccl.so.2")
            if os.path.exists(cand):
                os.environ["LGS_NCCL_LIB"] = cand
                return
    except Exception:
        pass


class Comm:
    """NCCL communicator of the distributed loop-closure batch (lgs_comm): one process per GPU.  Rank 0 draws the 128-byte
    unique id (Comm.unique_id()) and the caller carries it to the other ranks (Comm.from_torch_distributed does that with a
    torch.distributed broadcast); the gather of the records is then a single ncclAllGather issued by the C++ host."""

    def __init__(self, unique_id, rank, world, device):
        _prefer_bundled_nccl()
        self._L = _lib.load()
        idb = np.frombuffer(bytes(unique_id), np.uint8).copy()
        assert idb.size == 128
        h = C.c_void_p()
        check(self._L.lgs_comm_init_rank(idb.ctypes.data_as(C.c_void_p), int(rank), int(world), int(device), C.byref(h)))
        self._h = h
        self.rank, self.world, self.device = int(rank), int(world), int(device)

    @staticmethod
    def unique_id():
        _prefer_bundled_nccl()
        idb = np.zeros(128, np.uint8)
        check(_lib.load().lgs_comm_get_unique_id(idb.ctypes.data_as(C.c_void_p)))
        return idb.tobytes()

    @classmethod
    def from_torch_distributed(cls, device):
        """One communicator per rank of the default torch.distributed process group (the id travels by broadcast)."""
        import torch
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return cls(cls.unique_id(), 0, 1, device)
        rank, world = dist.get_rank(), dist.get_world_size()
        dev = "cuda:%d" % device if dist.get_backend() == "nccl" else "cpu"
        t = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(cls.unique_id()), dtype=torch.uint8))
        dist.broadcast(t, 0)
        return cls(bytes(t.cpu().numpy().tobytes()), rank, world, device)

    @property
    def nccl_version(self):
        v = C.c_int32()
        check(self._L.lgs_comm_info(self._h, None, None, C.byref(v)))
        return v.value

    def close(self):
        if getattr(self, "_h", None):
            self._L.lgs_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _dist_info(info):
    return dict(rank=info.rank, world=info.world, n_local=info.n_local, n_received=info.n_received, gather_bytes=info.gather_bytes,
                verify_ms=info.verify_ms, gather_ms=info.gather_ms)


def batch_align_dist(comm, scans, submaps, method=METHOD_GICP, guesses=None, max_iterations=100, transformation_epsilon=0.01,
                     max_correspondence_distance=2.0, k_correspondences=20, ndt_resolution=1.0, ndt_step_size=0.1, submap_leaf=0.5, fitness_max_range=-1.0,
                     n_workers=0, max_optimizer_iterations=0, euclidean_fitness_epsilon=0.0, sizes=None):
    """lgs_batch_align_dist (collective): every rank passes the same pair list; entries of scans / submaps this rank does not
    own may be None when `sizes` = [(n_scan, n_submap), ...] is given.  Returns (all records, info dict)."""
    L = _lib.load()
    n = len(scans)
    assert len(submaps) == n
    sc = [None if s is None else np.ascontiguousarray(s, np.float32) for s in scans]
    sm = [None if s is None else np.ascontiguousarray(s, np.float32) for s in submaps]
    sp = (C.c_void_p * max(n, 1))(*[None if s is None else s.ctypes.data for s in sc])
    mp = (C.c_void_p * max(n, 1))(*[None if s is None else s.ctypes.data for s in sm])
    if sizes is None:
        sizes = [(a.shape[0], b.shape[0]) for a, b in zip(sc, sm)]
    ns = (C.c_int64 * max(n, 1))(*[int(a) for a, _ in sizes])
    nm = (C.c_int64 * max(n, 1))(*[int(b) for _, b in sizes])
    g = _pack_guesses(guesses)
    bp = _batch_params(method, max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution, ndt_step_size,
                       submap_leaf, fitness_max_range, n_workers, max_optimizer_iterations, euclidean_fitness_epsilon)
    recs = (AlignResult * max(n, 1))()
    info = BatchDistInfo()
    check(L.lgs_batch_align_dist(comm._h, C.byref(bp), n, sp, ns, mp, nm, 16, g.ctypes.data_as(C.c_void_p) if g is not None else None, recs, C.byref(info)))
    return [recs[i] for i in range(n)], _dist_info(info)


# lgs_odometry_frame as a numpy record (T is column-major: T.reshape(4, 4, order="F") is the 4x4 pose)
ODOMETRY_FRAME = np.dtype([("T", "<f4", (16,)), ("trans_probability", "<f8"), ("accum_distance", "<f8"), ("sequence", "<i4"), ("frame", "<i4"),
                           ("converged", "<i4"), ("iterations", "<i4"), ("evaluations", "<i4"), ("keyframe_id", "<i4"), ("n_source", "<i8")])


def odometry_poses(records):
    """The (N, 4, 4) float32 poses of odometry records."""
    return np.ascontiguousarray(records["T"].reshape(-1, 4, 4).transpose(0, 2, 1))


def _odometry_params(method, keyframe_displacement, max_scan_accumulate_num, range_min, leaf, sor_mean_k, sor_stddev_mul, base_from_sensor,
                     max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution, ndt_step_size,
                     max_optimizer_iterations):
    p = OdometryParams(method=method, max_iterations=max_iterations, transformation_epsilon=transformation_epsilon,
                       max_correspondence_distance=max_correspondence_distance, k_correspondences=k_correspondences, ndt_resolution=ndt_resolution,
                       ndt_step_size=ndt_step_size, max_optimizer_iterations=max_optimizer_iterations, max_scan_accumulate_num=max_scan_accumulate_num,
                       keyframe_displacement=keyframe_displacement, range_min=-1.0 if range_min is None else float(range_min),
                       leaf=0.0 if leaf is None else float(leaf), sor_mean_k=sor_mean_k, sor_stddev_mul=sor_stddev_mul)
    E = np.eye(4, dtype=np.float32) if base_from_sensor is None else np.asarray(base_from_sensor, np.float32).reshape(4, 4)
    p.base_from_sensor[:] = [float(v) for v in E.ravel(order="F")]
    return p


class _OdometryInput:
    """The flat frame list of lgs_odometry_run*: host clouds (numpy, one record width for all) or packed xyzi CUDA tensors.
    Sequences that are None (allowed for the distributed run) contribute their frame counts from `n_points`."""

    def __init__(self, sequences, n_points=None, ctx=None):
        self.n_seq = len(sequences)
        self.n_frames, self.sizes, ptrs, self._keep = [], [], [], []
        self.device = None
        stride = None
        for s, seq in enumerate(sequences):
            if seq is None:
                if n_points is None:
                    raise ValueError("sequence %d is None: pass n_points" % s)
                self.n_frames.append(len(n_points[s]))
                self.sizes += [int(v) for v in n_points[s]]
                ptrs += [None] * len(n_points[s])
                continue
            self.n_frames.append(len(seq))
            for cloud in seq:
                if _is_torch(cloud):
                    if self.device is False:
                        raise ValueError("a call takes host clouds or CUDA tensors, not both")
                    p, n = _dev_cloud(cloud, ctx)
                    self.device = True
                    self._keep.append(cloud)
                    ptrs.append(p.value)
                else:
                    if self.device is True:
                        raise ValueError("a call takes host clouds or CUDA tensors, not both")
                    a, p, n, st = _host_cloud(cloud)
                    if stride not in (None, st):
                        raise ValueError("all host clouds of a call need the same record width")
                    self.device, stride = False, st
                    self._keep.append(a)
                    ptrs.append(p.value)
                self.sizes.append(int(n))
        if n_points is not None:
            want = [int(v) for seq in n_points for v in seq]
            if want != self.sizes:
                raise ValueError("n_points does not match the clouds")
        self.device = bool(self.device)
        self.stride = stride or 16
        self.total = len(self.sizes)
        self.nf = (C.c_int32 * max(self.n_seq, 1))(*self.n_frames)
        self.np = (C.c_int64 * max(self.total, 1))(*self.sizes)
        self.ptrs = (C.c_void_p * max(self.total, 1))(*ptrs)


def _initial_poses(initial_poses, n_seq):
    if initial_poses is None:
        return None
    if len(initial_poses) != n_seq:
        raise ValueError("need one initial pose per sequence")
    return _pack_guesses(initial_poses)


def odometry(sequences, method=METHOD_NDT, keyframe_displacement=1.0, max_scan_accumulate_num=20, range_min=1.0, leaf=0.1, sor_mean_k=0,
             sor_stddev_mul=1.0, base_from_sensor=None, initial_poses=None, keyframes=None, max_iterations=0, transformation_epsilon=0.0,
             max_correspondence_distance=0.0, k_correspondences=0, ndt_resolution=0.0, ndt_step_size=0.0, max_optimizer_iterations=0, ctx=None):
    """Offline odometry (lgs_odometry_run / _dev): the scan matcher's key-frame loop (LSM:122-250) over each sequence of sweeps in
    the sensor frame.  sequences: a list of sequences, each a list (or a stacked array / tensor) of clouds, all numpy host clouds
    or all CUDA (N, 4) tensors.  leaf / range_min None disable the VoxelGrid / range crop (the crop needs the VoxelGrid);
    sor_mean_k 0 disables the outlier filter.  Registration settings left at 0 take the scan-matcher YAML defaults.
    keyframes: None or one entry per sequence, each None or an empty KeyFrameArray on the same context, which the run fills.
    Returns a numpy structured array (ODOMETRY_FRAME) with one record per frame, in (sequence, frame) order."""
    ctx = ctx or default_context()
    inp = _OdometryInput(sequences, ctx=ctx)
    p = _odometry_params(method, keyframe_displacement, max_scan_accumulate_num, range_min, leaf, sor_mean_k, sor_stddev_mul, base_from_sensor,
                         max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution, ndt_step_size,
                         max_optimizer_iterations)
    g = _initial_poses(initial_poses, inp.n_seq)
    gp = g.ctypes.data_as(C.c_void_p) if g is not None else None
    kfs = None
    if keyframes is not None:
        if len(keyframes) != inp.n_seq:
            raise ValueError("need one keyframes entry per sequence")
        kfs = (C.c_void_p * max(inp.n_seq, 1))(*[None if k is None else k._h.value for k in keyframes])
    recs = np.zeros(max(inp.total, 1), ODOMETRY_FRAME)
    rp = recs.ctypes.data_as(C.c_void_p)
    if inp.device:
        check(ctx._L.lgs_odometry_run_dev(ctx._h, C.byref(p), inp.n_seq, inp.nf, inp.ptrs, inp.np, gp, kfs, rp))
    else:
        check(ctx._L.lgs_odometry_run(ctx._h, C.byref(p), inp.n_seq, inp.nf, inp.ptrs, inp.np, inp.stride, gp, kfs, rp))
    return recs[: inp.total]


def odometry_dist(comm, sequences, n_points=None, method=METHOD_NDT, keyframe_displacement=1.0, max_scan_accumulate_num=20, range_min=1.0, leaf=0.1,
                  sor_mean_k=0, sor_stddev_mul=1.0, base_from_sensor=None, initial_poses=None, max_iterations=0, transformation_epsilon=0.0,
                  max_correspondence_distance=0.0, k_correspondences=0, ndt_resolution=0.0, ndt_step_size=0.0, max_optimizer_iterations=0, ctx=None):
    """lgs_odometry_run_dist / _dev (collective over `comm`, ctx on comm's device): every rank passes the same sequence list;
    a sequence this rank does not own may be None when n_points (per sequence, the point count of every frame) is given.
    Returns (records of every frame of every sequence, info dict)."""
    ctx = ctx or default_context()
    inp = _OdometryInput(sequences, n_points, ctx=ctx)
    p = _odometry_params(method, keyframe_displacement, max_scan_accumulate_num, range_min, leaf, sor_mean_k, sor_stddev_mul, base_from_sensor,
                         max_iterations, transformation_epsilon, max_correspondence_distance, k_correspondences, ndt_resolution, ndt_step_size,
                         max_optimizer_iterations)
    g = _initial_poses(initial_poses, inp.n_seq)
    gp = g.ctypes.data_as(C.c_void_p) if g is not None else None
    recs = np.zeros(max(inp.total, 1), ODOMETRY_FRAME)
    rp = recs.ctypes.data_as(C.c_void_p)
    info = OdometryDistInfo()
    if inp.device:
        check(ctx._L.lgs_odometry_run_dist_dev(ctx._h, comm._h, C.byref(p), inp.n_seq, inp.nf, inp.ptrs, inp.np, gp, rp, C.byref(info)))
    else:
        check(ctx._L.lgs_odometry_run_dist(ctx._h, comm._h, C.byref(p), inp.n_seq, inp.nf, inp.ptrs, inp.np, inp.stride, gp, rp, C.byref(info)))
    return recs[: inp.total], dict(rank=info.rank, world=info.world, n_local_sequences=info.n_local_sequences, n_local_frames=info.n_local_frames,
                                   n_received=info.n_received, gather_bytes=info.gather_bytes, run_ms=info.run_ms, gather_ms=info.gather_ms)


def odometry_profile():
    """lgs_odometry_profile: with LGS_ODOMETRY_PROFILE=1 set before the runs, the CUDA-event split of this thread's odometry frames
    since the last call (which clears it)."""
    out = np.zeros(4)
    check(_lib.load().lgs_odometry_profile(out.ctypes.data_as(C.c_void_p)))
    return dict(frames=int(out[0]), prefilter_ms=out[1], align_ms=out[2], keyframe_ms=out[3])


def batch_release():
    """Frees the worker state batch_align keeps between calls (streams, registration objects, device buffers)."""
    _lib.load().lgs_batch_release()
