"""ORACLE (test infrastructure) -- ctypes view of oracle/_build/liblgs_oracle.so.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
It is the checker, never the product path.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liblgs_oracle.so")

SEARCH_KDTREE, SEARCH_DIRECT26, SEARCH_DIRECT7, SEARCH_DIRECT1 = 0, 1, 2, 3
REG_NONE, REG_MIN_EIG, REG_NORMALIZED_MIN_EIG, REG_PLANE, REG_FROBENIUS = 0, 1, 2, 3, 4


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".cpp", ".hpp", "Makefile"))]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE], stdout=subprocess.DEVNULL)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        vp, f32p, f64p, i32p = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.orc_max_threads.restype = C.c_int
        L.orc_vg_run.restype = vp
        L.orc_vg_run.argtypes = [vp, C.c_long, vp, C.c_int, C.c_double, vp]
        L.orc_vg_status.argtypes = [vp]
        L.orc_vg_out_n.restype = C.c_long
        L.orc_vg_out_n.argtypes = [vp]
        L.orc_vg_n_kept.restype = C.c_long
        L.orc_vg_n_kept.argtypes = [vp]
        L.orc_vg_get.argtypes = [vp] * 7
        L.orc_vg_free.argtypes = [vp]
        L.orc_ndt_create.restype = vp
        L.orc_ndt_destroy.argtypes = [vp]
        L.orc_ndt_set_params.argtypes = [vp, C.c_float, C.c_double, C.c_double, C.c_int, C.c_double, C.c_int, C.c_int]
        L.orc_ndt_set_target.argtypes = [vp, vp, C.c_long]
        L.orc_ndt_set_source.argtypes = [vp, vp, C.c_long]
        L.orc_ndt_align.argtypes = [vp] * 8
        L.orc_ndt_fitness.restype = C.c_double
        L.orc_ndt_fitness.argtypes = [vp, C.c_double]
        L.orc_ndt_voxel_count.restype = C.c_long
        L.orc_ndt_voxel_count.argtypes = [vp]
        L.orc_ndt_refused.argtypes = [vp]
        L.orc_ndt_export_voxels.argtypes = [vp] * 7
        L.orc_ndt_derivatives.restype = C.c_double
        L.orc_ndt_derivatives.argtypes = [vp, vp, vp, C.c_int, vp, vp]
        L.orc_ndt_convert_transform.argtypes = [vp, vp]
        L.orc_ndt_calculate_score.restype = C.c_double
        L.orc_ndt_calculate_score.argtypes = [vp, vp]
        L.orc_gicp_create.restype = vp
        L.orc_gicp_destroy.argtypes = [vp]
        L.orc_gicp_set_params.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int]
        L.orc_gicp_set_source.argtypes = [vp, vp, C.c_long]
        L.orc_gicp_set_target.argtypes = [vp, vp, C.c_long]
        L.orc_gicp_swap.argtypes = [vp]
        L.orc_gicp_align.argtypes = [vp] * 7
        L.orc_gicp_fitness.restype = C.c_double
        L.orc_gicp_fitness.argtypes = [vp, C.c_double]
        L.orc_gicp_final_hessian.argtypes = [vp, vp]
        L.orc_gicp_covariances.argtypes = [vp, C.c_int, vp]
        L.orc_gicp_evaluate_cost.restype = C.c_double
        L.orc_gicp_evaluate_cost.argtypes = [vp, vp]
        L.orc_gicp_set_covariances.argtypes = [vp, C.c_int, vp, C.c_long]
        L.orc_gicp_linearize.restype = C.c_double
        L.orc_gicp_linearize.argtypes = [vp, vp, vp, vp, vp]
        L.orc_pgicp_create.restype = vp
        L.orc_pgicp_destroy.argtypes = [vp]
        L.orc_pgicp_set_params.argtypes = [vp, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double, C.c_int]
        L.orc_pgicp_set_source.argtypes = [vp, vp, C.c_long]
        L.orc_pgicp_set_target.argtypes = [vp, vp, C.c_long]
        L.orc_pgicp_align.argtypes = [vp] * 7
        L.orc_pgicp_fitness.restype = C.c_double
        L.orc_pgicp_fitness.argtypes = [vp, C.c_double]
        L.orc_pgicp_covariances.argtypes = [vp, C.c_int, vp]
        L.orc_pgicp_functor.argtypes = [vp] * 7
        L.orc_icp_create.restype = vp
        L.orc_icp_destroy.argtypes = [vp]
        L.orc_icp_set_params.argtypes = [vp, C.c_double, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int]
        L.orc_icp_set_source.argtypes = [vp, vp, C.c_long]
        L.orc_icp_set_target.argtypes = [vp, vp, C.c_long]
        L.orc_icp_align.argtypes = [vp] * 8
        L.orc_icp_fitness.restype = C.c_double
        L.orc_icp_fitness.argtypes = [vp, C.c_double]
        L.orc_icp_step.argtypes = [vp] * 4
        L.orc_transform_cloud.argtypes = [vp, C.c_long, vp, vp]
        L.orc_knn.argtypes = [vp, C.c_long, vp, C.c_long, C.c_int, vp, vp, C.c_int]
        L.orc_fitness.restype = C.c_double
        L.orc_fitness.argtypes = [vp, C.c_long, vp, C.c_long, vp, C.c_double, C.c_int]
        L.orc_sor_run.restype = vp
        L.orc_sor_run.argtypes = [vp, C.c_long, C.c_int, C.c_double, C.c_int]
        L.orc_sor_out_n.restype = C.c_long
        L.orc_sor_out_n.argtypes = [vp]
        L.orc_sor_get.argtypes = [vp] * 5
        L.orc_sor_free.argtypes = [vp]
        L.orc_linalg_batch.restype = C.c_int
        L.orc_linalg_batch.argtypes = [C.c_int, C.c_long, vp, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] == 4, "points are N x 4 float32 (x, y, z, intensity)"
    return a


def max_threads():
    return lib().orc_max_threads()


def voxel_grid(pts, leaf, min_points_per_voxel=0, range_min=-1.0, box=None):
    """Oracle of the prefilter: crop (PPF:89-112) + pcl::VoxelGrid (PPF:114-121).  Returns a dict."""
    L = lib()
    pts = _pts(pts)
    n = pts.shape[0]
    leaf3 = np.asarray([leaf] * 3 if np.isscalar(leaf) else leaf, dtype=np.float32)
    boxa = None if box is None else np.asarray(box, dtype=np.float64)
    h = L.orc_vg_run(_p(pts), n, _p(leaf3), int(min_points_per_voxel), float(range_min), _p(boxa))
    try:
        m = L.orc_vg_out_n(h)
        status = L.orc_vg_status(h)
        out = np.empty((m, 4), np.float32)
        ok = status == 0
        out_idx = np.empty(m if ok else 0, np.int32)
        out_cnt = np.empty(m if ok else 0, np.int32)
        vidx = np.empty(n, np.int32)
        rank = np.empty(n, np.int32)
        grid = np.zeros(9, np.int32)
        L.orc_vg_get(h, _p(out), _p(out_idx), _p(out_cnt), _p(vidx), _p(rank), _p(grid))
        return dict(status=status, points=out, out_idx=out_idx, out_count=out_cnt, voxel_idx=vidx, member_rank=rank,
                    min_b=grid[0:3].copy(), max_b=grid[3:6].copy(), div_b=grid[6:9].copy(), n_kept=L.orc_vg_n_kept(h))
    finally:
        L.orc_vg_free(h)


def statistical_outlier_removal(pts, mean_k=30, stddev_mul=1.2, negative=False):
    """Oracle of pcl::StatisticalOutlierRemoval as the prefilter node uses it (PPF:132-140).  Returns a dict."""
    L = lib()
    pts = _pts(pts)
    n = pts.shape[0]
    h = L.orc_sor_run(_p(pts), n, int(mean_k), float(stddev_mul), 1 if negative else 0)
    try:
        m = L.orc_sor_out_n(h)
        out = np.empty((m, 4), np.float32)
        dist = np.empty(n, np.float32)
        keep = np.empty(n, np.uint8)
        stats = np.zeros(3)
        L.orc_sor_get(h, _p(out), _p(dist), _p(keep), _p(stats))
    finally:
        L.orc_sor_free(h)
    return dict(points=out, distances=dist, keep=keep.astype(bool), mean=stats[0], stddev=stats[1], threshold=stats[2])


class NDT:
    """Oracle of pclomp::NormalDistributionsTransform (PCL method names)."""

    def __init__(self):
        self._L = lib()
        self._h = self._L.orc_ndt_create()
        self.params = dict(resolution=1.0, step_size=0.1, trans_eps=0.1, max_iter=35, outlier_ratio=0.55,
                           search_method=SEARCH_DIRECT7, num_threads=0)
        self._ns = 0
        self.stats = None

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.orc_ndt_destroy(self._h)
            self._h = None

    def _push(self):
        p = self.params
        self._L.orc_ndt_set_params(self._h, p["resolution"], p["step_size"], p["trans_eps"], p["max_iter"], p["outlier_ratio"],
                                   p["search_method"], p["num_threads"])

    def setResolution(self, r): self.params["resolution"] = float(r); self._push()
    def setStepSize(self, s): self.params["step_size"] = float(s); self._push()
    def setTransformationEpsilon(self, e): self.params["trans_eps"] = float(e); self._push()
    def setMaximumIterations(self, n): self.params["max_iter"] = int(n); self._push()
    def setOutlierRatio(self, o): self.params["outlier_ratio"] = float(o); self._push()
    def setNeighborhoodSearchMethod(self, m): self.params["search_method"] = int(m); self._push()
    def setNumThreads(self, n): self.params["num_threads"] = int(n); self._push()

    def setInputTarget(self, pts):
        pts = _pts(pts)
        self._push()
        self._L.orc_ndt_set_target(self._h, _p(pts), pts.shape[0])

    def setInputSource(self, pts):
        pts = _pts(pts)
        self._ns = pts.shape[0]
        self._L.orc_ndt_set_source(self._h, _p(pts), pts.shape[0])

    def align(self, guess=None):
        g = np.eye(4, dtype=np.float32) if guess is None else np.asarray(guess, dtype=np.float32)
        gc = np.asfortranarray(g).ravel(order="F").copy()
        T = np.empty(16, np.float32)
        it, cv = C.c_int(), C.c_int()
        tp = C.c_double()
        out = np.empty((self._ns, 4), np.float32)
        st = np.zeros(3, np.int32)
        self._L.orc_ndt_align(self._h, _p(gc), _p(T), C.addressof(it), C.addressof(cv), C.addressof(tp), _p(out), _p(st))
        self.final_transformation = T.reshape(4, 4, order="F").copy()
        self.nr_iterations, self.converged, self.trans_probability = it.value, bool(cv.value), tp.value
        self.stats = dict(derivative_evals=int(st[0]), line_search_trials=int(st[1]), hessian_recomputes=int(st[2]))
        return out

    def hasConverged(self): return self.converged
    def getFinalTransformation(self): return self.final_transformation
    def getFinalNumIteration(self): return self.nr_iterations
    def getTransformationProbability(self): return self.trans_probability
    def getFitnessScore(self, max_range=np.finfo(np.float64).max): return self._L.orc_ndt_fitness(self._h, float(max_range))

    def export_voxels(self):
        v = self._L.orc_ndt_voxel_count(self._h)
        idx, npts = np.empty(v, np.int32), np.empty(v, np.int32)
        mean, cov, icov = np.empty((v, 3)), np.empty((v, 9)), np.empty((v, 9))
        grid = np.zeros(9, np.int32)
        self._L.orc_ndt_export_voxels(self._h, _p(idx), _p(npts), _p(mean), _p(cov), _p(icov), _p(grid))
        return dict(idx=idx, n=npts, mean=mean, cov=cov, icov=icov, min_b=grid[0:3].copy(), max_b=grid[3:6].copy(),
                    div_b=grid[6:9].copy(), refused=bool(self._L.orc_ndt_refused(self._h)))

    def derivatives(self, T, p, mode=0):
        Tc = np.asarray(T, np.float32).ravel(order="F").copy()
        p = np.asarray(p, np.float64).copy()
        g, H = np.zeros(6), np.zeros(36)
        s = self._L.orc_ndt_derivatives(self._h, _p(Tc), _p(p), int(mode), _p(g), _p(H))
        return s, g, H.reshape(6, 6)

    def calculateScore(self, T):
        Tc = np.asarray(T, np.float32).ravel(order="F").copy()
        return self._L.orc_ndt_calculate_score(self._h, _p(Tc))


def ndt_convert_transform(p):
    p = np.asarray(p, np.float64).copy()
    T = np.empty(16, np.float32)
    lib().orc_ndt_convert_transform(_p(p), _p(T))
    return T.reshape(4, 4, order="F").copy()


class FastGICP:
    """Oracle of fast_gicp::FastGICP (PCL method names)."""

    def __init__(self):
        self._L = lib()
        self._h = self._L.orc_gicp_create()
        self.params = dict(k=20, max_corr_dist=-1.0, trans_eps=5e-4, rot_eps=2e-3, max_iter=64, regularization=REG_PLANE, num_threads=0)
        self._ns = self._nt = 0

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.orc_gicp_destroy(self._h)
            self._h = None

    def _push(self):
        p = self.params
        self._L.orc_gicp_set_params(self._h, p["k"], p["max_corr_dist"], p["trans_eps"], p["rot_eps"], p["max_iter"], p["regularization"],
                                    p["num_threads"])

    def setCorrespondenceRandomness(self, k): self.params["k"] = int(k); self._push()
    def setMaxCorrespondenceDistance(self, d): self.params["max_corr_dist"] = float(d); self._push()
    def setTransformationEpsilon(self, e): self.params["trans_eps"] = float(e); self._push()
    def setRotationEpsilon(self, e): self.params["rot_eps"] = float(e); self._push()
    def setMaximumIterations(self, n): self.params["max_iter"] = int(n); self._push()
    def setRegularizationMethod(self, m): self.params["regularization"] = int(m); self._push()
    def setNumThreads(self, n): self.params["num_threads"] = int(n); self._push()

    def setInputSource(self, pts):
        pts = _pts(pts)
        self._ns = pts.shape[0]
        self._L.orc_gicp_set_source(self._h, _p(pts), pts.shape[0])

    def setInputTarget(self, pts):
        pts = _pts(pts)
        self._nt = pts.shape[0]
        self._L.orc_gicp_set_target(self._h, _p(pts), pts.shape[0])

    def swapSourceAndTarget(self):
        self._L.orc_gicp_swap(self._h)
        self._ns, self._nt = self._nt, self._ns

    def align(self, guess=None):
        g = np.eye(4, dtype=np.float32) if guess is None else np.asarray(guess, dtype=np.float32)
        gc = g.ravel(order="F").copy()
        T = np.empty(16, np.float32)
        it, cv = C.c_int(), C.c_int()
        out = np.empty((self._ns, 4), np.float32)
        st = np.zeros(2, np.int32)
        self._L.orc_gicp_align(self._h, _p(gc), _p(T), C.addressof(it), C.addressof(cv), _p(out), _p(st))
        self.final_transformation = T.reshape(4, 4, order="F").copy()
        self.nr_iterations, self.converged = it.value, bool(cv.value)
        self.stats = dict(linearize_calls=int(st[0]), error_calls=int(st[1]))
        return out

    def hasConverged(self): return self.converged
    def getFinalTransformation(self): return self.final_transformation
    def getFitnessScore(self, max_range=np.finfo(np.float64).max): return self._L.orc_gicp_fitness(self._h, float(max_range))

    def getFinalHessian(self):
        H = np.empty(36)
        self._L.orc_gicp_final_hessian(self._h, _p(H))
        return H.reshape(6, 6)

    def covariances(self, which):
        n = self._ns if which == 0 else self._nt
        c = np.empty((n, 9))
        self._L.orc_gicp_covariances(self._h, int(which), _p(c))
        return c.reshape(n, 3, 3)

    def evaluateCost(self, relative_pose):
        Tc = np.asarray(relative_pose, np.float32).ravel(order="F").copy()
        return self._L.orc_gicp_evaluate_cost(self._h, _p(Tc))

    def _set_covariances(self, which, covs):
        c = np.ascontiguousarray(np.asarray(covs, np.float64).reshape(-1, 9))
        self._L.orc_gicp_set_covariances(self._h, which, _p(c), c.shape[0])

    def setSourceCovariances(self, covs): self._set_covariances(0, covs)
    def setTargetCovariances(self, covs): self._set_covariances(1, covs)

    def linearize(self, T):
        Tr = np.ascontiguousarray(np.asarray(T, np.float64))
        H, b = np.zeros(36), np.zeros(6)
        corr = np.empty(self._ns, np.int32)
        c = self._L.orc_gicp_linearize(self._h, _p(Tr), _p(H), _p(b), _p(corr))
        return c, H.reshape(6, 6), b, corr


class GeneralizedIterativeClosestPoint:
    """Oracle of pclomp::GeneralizedIterativeClosestPoint (BFGS; PCL method names, defaults of gicp_omp.h:116-126)."""

    def __init__(self):
        self._L = lib()
        self._h = self._L.orc_pgicp_create()
        self.params = dict(k=20, max_corr_dist=5.0, trans_eps=5e-4, rot_eps=2e-3, max_iter=200, max_inner=20, gicp_eps=1e-3, num_threads=0)
        self._ns = self._nt = 0

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.orc_pgicp_destroy(self._h)
            self._h = None

    def _push(self):
        p = self.params
        self._L.orc_pgicp_set_params(self._h, p["k"], p["max_corr_dist"], p["trans_eps"], p["rot_eps"], p["max_iter"], p["max_inner"], p["gicp_eps"],
                                     p["num_threads"])

    def setCorrespondenceRandomness(self, k): self.params["k"] = int(k); self._push()
    def setMaxCorrespondenceDistance(self, d): self.params["max_corr_dist"] = float(d); self._push()
    def setTransformationEpsilon(self, e): self.params["trans_eps"] = float(e); self._push()
    def setRotationEpsilon(self, e): self.params["rot_eps"] = float(e); self._push()
    def setMaximumIterations(self, n): self.params["max_iter"] = int(n); self._push()
    def setMaximumOptimizerIterations(self, n): self.params["max_inner"] = int(n); self._push()
    def setNumThreads(self, n): self.params["num_threads"] = int(n); self._push()

    def setInputSource(self, pts):
        pts = _pts(pts)
        self._ns = pts.shape[0]
        self._L.orc_pgicp_set_source(self._h, _p(pts), pts.shape[0])

    def setInputTarget(self, pts):
        pts = _pts(pts)
        self._nt = pts.shape[0]
        self._L.orc_pgicp_set_target(self._h, _p(pts), pts.shape[0])

    def align(self, guess=None):
        g = np.eye(4, dtype=np.float32) if guess is None else np.asarray(guess, dtype=np.float32)
        gc = g.ravel(order="F").copy()
        T = np.empty(16, np.float32)
        it, cv = C.c_int(), C.c_int()
        out = np.empty((self._ns, 4), np.float32)
        st = np.zeros(5, np.int32)
        self._L.orc_pgicp_align(self._h, _p(gc), _p(T), C.addressof(it), C.addressof(cv), _p(out), _p(st))
        self.final_transformation = T.reshape(4, 4, order="F").copy()
        self.nr_iterations, self.converged = it.value, bool(cv.value)
        self.stats = dict(f_calls=int(st[0]), df_calls=int(st[1]), fdf_calls=int(st[2]), inner_iterations=int(st[3]), correspondences=int(st[4]))
        return out

    def hasConverged(self): return self.converged
    def getFinalTransformation(self): return self.final_transformation
    def getFitnessScore(self, max_range=np.finfo(np.float64).max): return self._L.orc_pgicp_fitness(self._h, float(max_range))

    def covariances(self, which):
        n = self._ns if which == 0 else self._nt
        c = np.empty((n, 9))
        self._L.orc_pgicp_covariances(self._h, int(which), _p(c))
        return c.reshape(n, 3, 3)

    def functor(self, guess, transformation, x):
        """One outer-iteration set-up at (transformation_, guess), then f(x), df(x), fdf(x) (gicp_omp_impl.hpp:245-367)."""
        gc = np.asarray(guess, np.float32).ravel(order="F").copy()
        tc = np.asarray(transformation, np.float32).ravel(order="F").copy()
        x = np.ascontiguousarray(x, np.float64)
        out = np.zeros(15)
        corr = np.empty(self._ns, np.int32)
        mahal = np.empty((self._ns, 9), np.float32)
        self._L.orc_pgicp_functor(self._h, _p(gc), _p(tc), _p(x), _p(out), _p(corr), _p(mahal))
        return dict(f=out[0], df=out[1:7].copy(), fdf_f=out[7], fdf_g=out[8:14].copy(), n_corr=int(out[14]), corr=corr, mahal=mahal)


class IterativeClosestPoint:
    """Oracle of pcl::IterativeClosestPoint<PointXYZI, PointXYZI> (PCL defaults; GBS:142-151 sets 30 / 100 / 1e-8 / 1e-6)."""

    def __init__(self):
        self._L = lib()
        self._h = self._L.orc_icp_create()
        self.params = dict(max_corr_dist=float(np.sqrt(np.finfo(np.float64).max)), max_iter=10, trans_eps=0.0, rot_eps=0.0,
                           fitness_eps=-float(np.finfo(np.float64).max), num_threads=0)
        self._ns = 0

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.orc_icp_destroy(self._h)
            self._h = None

    def _push(self):
        p = self.params
        self._L.orc_icp_set_params(self._h, p["max_corr_dist"], p["max_iter"], p["trans_eps"], p["rot_eps"], p["fitness_eps"], p["num_threads"])

    def setMaxCorrespondenceDistance(self, d): self.params["max_corr_dist"] = float(d); self._push()
    def setMaximumIterations(self, n): self.params["max_iter"] = int(n); self._push()
    def setTransformationEpsilon(self, e): self.params["trans_eps"] = float(e); self._push()
    def setTransformationRotationEpsilon(self, e): self.params["rot_eps"] = float(e); self._push()
    def setEuclideanFitnessEpsilon(self, e): self.params["fitness_eps"] = float(e); self._push()
    def setRANSACIterations(self, n): pass  # no rejector is installed by default: never read
    def setNumThreads(self, n): self.params["num_threads"] = int(n); self._push()

    def setInputSource(self, pts):
        pts = _pts(pts)
        self._ns = pts.shape[0]
        self._L.orc_icp_set_source(self._h, _p(pts), pts.shape[0])

    def setInputTarget(self, pts):
        pts = _pts(pts)
        self._L.orc_icp_set_target(self._h, _p(pts), pts.shape[0])

    def align(self, guess=None):
        g = np.eye(4, dtype=np.float32) if guess is None else np.asarray(guess, dtype=np.float32)
        gc = g.ravel(order="F").copy()
        T = np.empty(16, np.float32)
        it, cv = C.c_int(), C.c_int()
        out = np.empty((self._ns, 4), np.float32)
        st = np.zeros(2, np.int64)
        mse = C.c_double()
        self._L.orc_icp_align(self._h, _p(gc), _p(T), C.addressof(it), C.addressof(cv), _p(out), _p(st), C.addressof(mse))
        self.final_transformation = T.reshape(4, 4, order="F").copy()
        self.nr_iterations, self.converged = it.value, bool(cv.value)
        self.stats = dict(convergence_state=int(st[0]), correspondences=int(st[1]), mse=mse.value)
        return out

    def hasConverged(self): return self.converged
    def getFinalTransformation(self): return self.final_transformation
    def getFitnessScore(self, max_range=np.finfo(np.float64).max): return self._L.orc_icp_fitness(self._h, float(max_range))

    def step(self, guess):
        gc = np.asarray(guess, np.float32).ravel(order="F").copy()
        sums, T = np.zeros(17), np.zeros(16, np.float32)
        ok = self._L.orc_icp_step(self._h, _p(gc), _p(sums), _p(T))
        return bool(ok), sums, T.reshape(4, 4, order="F").copy()


def from_pointcloud2(data, width, height, point_step, fields):
    """ORACLE of pcl::fromROSMsg<pcl::PointXYZI> (called at PPF:65-70, LSM:122-130): numpy restatement of PCL's field
    mapping (pcl/conversions.h createMapping / fromPCLPointCloud2: a message field is copied only when its name and
    datatype equal the point type's, FLOAT32 = 7 for x, y, z, intensity; unmatched point fields keep their default 0).
    `fields`: name -> (offset, datatype).  Returns (N, 4) float32 xyzi."""
    n = int(width) * int(height)
    raw = np.frombuffer(data, dtype=np.uint8, count=n * int(point_step)).reshape(n, int(point_step))
    out = np.zeros((n, 4), np.float32)
    for col, name in enumerate(("x", "y", "z", "intensity")):
        if name in fields and int(fields[name][1]) == 7:
            off = int(fields[name][0])
            out[:, col] = np.ascontiguousarray(raw[:, off:off + 4]).view("<f4")[:, 0]
    return out


def transform_point_cloud(pts, T):
    """pcl::transformPointCloud with an Eigen::Matrix4f (lidar_graph_slam_utils transform_point_cloud, LSM:206, GBS:305)."""
    pts = _pts(pts)
    Tc = np.asarray(T, np.float32).reshape(4, 4).ravel(order="F").copy()
    out = np.empty_like(pts)
    lib().orc_transform_cloud(_p(pts), pts.shape[0], _p(Tc), _p(out))
    return out


def assemble_submap(clouds, poses, ids, leaf=0.0):
    """The sub-map loops of LSM:199-208 / GBS:297-313: transform each key frame by its pose, concatenate in the order of
    ids, optionally pcl::VoxelGrid(leaf)."""
    parts = [transform_point_cloud(clouds[i], poses[i]) for i in ids]
    cat = np.concatenate(parts, axis=0) if parts else np.zeros((0, 4), np.float32)
    if leaf > 0 and cat.shape[0]:
        return voxel_grid(cat, leaf)["points"]
    return cat


def knn(pts, queries, k, num_threads=0):
    pts, queries = _pts(pts), _pts(queries)
    m = queries.shape[0]
    idx = np.empty((m, k), np.int32)
    d2 = np.empty((m, k), np.float32)
    lib().orc_knn(_p(pts), pts.shape[0], _p(queries), m, int(k), _p(idx), _p(d2), num_threads or max_threads())
    return idx, d2


LINALG_SVD3, LINALG_EIG3, LINALG_INV3, LINALG_SVD_SOLVE6, LINALG_SVD3_F32, LINALG_LDLT6 = 0, 1, 2, 3, 16, 17
_LINALG_SHAPES = {0: (9, 21), 1: (9, 13), 2: (9, 9), 3: (42, 6), 16: (9, 21), 17: (42, 6)}


def linalg_batch(op, inputs):
    """The solvers of linalg.hpp over a batch: inputs (n, 9) for the 3x3 ops, (n, 42) = H row-major + b for the 6x6
    ones.  Returns (n, width) f64 in the layout of lgs_linalg_batch (LINALG_SVD3_F32: f32 inputs and results, exactly
    widened)."""
    nin, nout = _LINALG_SHAPES[op]
    a = np.ascontiguousarray(inputs, dtype=np.float64).reshape(-1, nin)
    out = np.empty((a.shape[0], nout))
    if lib().orc_linalg_batch(int(op), a.shape[0], _p(a), _p(out)) != 0:
        raise ValueError("unknown linalg op %d" % op)
    return out


def fitness(target, source, T, max_range=np.finfo(np.float64).max, num_threads=0):
    target, source = _pts(target), _pts(source)
    Tc = np.asarray(T, np.float32).ravel(order="F").copy()
    return lib().orc_fitness(_p(target), target.shape[0], _p(source), source.shape[0], _p(Tc), float(max_range), num_threads or max_threads())
