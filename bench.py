#!/usr/bin/env python
"""bench.py -- headline benchmark of the LiDAR front-end hot path (see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): NDT scan-to-map aligns per second, 120 000-point 64-beam sweep against a 1 000 000-point
local map (configs[0]: DIRECT7, 1.0 m, step 0.1, eps 0.01, max_iter 64), synthetic data (SURVEY.md section 8d).
One step = one align of one sweep against the resident map.  At N > 1 every rank runs its own sequence against its
own map ("offline multi-sequence odometry", the north_star's partitioning of odometry): weak scaling, no data-path
collective; the loop-closure batch (configs[4]) is measured next to it with its NCCL result gather and reported
under "loop_closure".

  value  aligns/s, sweeps already resident in HBM (set_source_dev + align), per-step CUDA events, L2 flushed
         between steps outside the event pairs
  e2e    aligns/s through the reference-facing call sequence with HOST buffers: setInputSource(pinned host sweep)
         -> align(aligned cloud, guess) -> getFinalTransformation; H2D of the sweep and D2H of the aligned cloud and of
         the result inside the timed region
  roofline  the dominant kernel (ndt_align_kernel: one launch per align): algorithmic bytes of all its evaluations /
         its CUDA-event duration, timed live in the timed region
  cpu_baseline  the oracle (CPU restatement of the reference's OpenMP path) on this box's host cores, bounded sample

--impl reference times the reference's CPU path (the oracle port: the reference cannot be compiled here) on the
same workload with all host threads.

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float32 / float64), so that
two builds can be compared output for output on identical inputs (the workload is seeded):
  final_transformation (4x4 f32), fitness_score, transformation_probability, align_counts (iterations, converged,
  derivative evaluations, line-search trials, computeHessian calls)   the headline path (sweep resident in HBM)
  e2e_<same names>, e2e_aligned_cloud (n_source x 4 f32)              the e2e path (host buffers)
--impl reference writes the headline names and aligned_cloud.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "cfg0: NDT DIRECT7 res 1.0 m, 120000-pt 64-beam sweep -> 1000000-pt local map (20 keyframes, 0.2 m filtered)"
NDT_PARAMS = dict(resolution=1.0, step=0.1, eps=0.01, max_iter=64)
N_SWEEP_POOL = 6


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def make_workload(rank):
    """Target map + a pool of source sweeps with perturbed guesses, distinct per rank (multi-sequence)."""
    from lidar_graph_slam_b200 import synth
    seed = synth.SEED + 7919 * rank
    d = synth.ndt_scan_to_map(perturb_seed=1 + rank, seed=seed)
    # further scans of the sequence: sweeps physically re-cast 0.5 m apart with fresh noise and their own guesses
    sweeps, guesses, poses = synth.ndt_sweep_pool(d, N_SWEEP_POOL, seed=seed, perturb_seed=1 + rank)
    return d["target"], sweeps, guesses, poses


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self._kill)  # the sampler must not outlive a benchmark that fails before stop()
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def _kill(self):
        if self.proc and self.proc.poll() is None:
            self.proc.kill()
            self.proc.wait()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads():
    """Host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm must not inherit that)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            j = json.load(f)
        return float(j["dram_bytes_per_launch"]), j.get("source")
    except Exception:
        return None, None


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ndt_outputs(ndt, counts, prefix=""):
    """What the caller of one NDT align receives (the product's and the oracle's NDT share these getters).  `counts`:
    iterations, converged, derivative evaluations, line-search trials, computeHessian calls."""
    return {prefix + "final_transformation": np.array(ndt.getFinalTransformation(), np.float32),
            prefix + "fitness_score": np.array([ndt.getFitnessScore()], np.float64),
            prefix + "transformation_probability": np.array([ndt.getTransformationProbability()], np.float64),
            prefix + "align_counts": np.array(counts, np.float64)}


def write_outputs(directory, arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def cpu_baseline(target, sweeps, guesses, budget_s=20.0, threads=0):
    """The oracle (kind 'port': CPU restatement of the reference's ndt_omp path) on the host cores, bounded sample."""
    from oracle import pyoracle as O
    nthreads = threads or host_threads()
    n = O.NDT()
    n.setNumThreads(nthreads)
    n.setResolution(NDT_PARAMS["resolution"])
    n.setStepSize(NDT_PARAMS["step"])
    n.setTransformationEpsilon(NDT_PARAMS["eps"])
    n.setMaximumIterations(NDT_PARAMS["max_iter"])
    t0 = time.perf_counter()
    n.setInputTarget(target)
    t_build = time.perf_counter() - t0
    done, t_align = 0, 0.0
    while done < len(sweeps) and (done == 0 or t_align < budget_s):
        n.setInputSource(sweeps[done])
        t0 = time.perf_counter()
        n.align(guesses[done])
        t_align += time.perf_counter() - t0
        done += 1
    # the reference's own default thread count (lidar_scan_matcher.param.yaml:10 omp_num_thread: 4), two aligns
    n.setNumThreads(min(4, nthreads))
    t4, d4 = 0.0, 0
    for k in range(min(2, len(sweeps))):
        n.setInputSource(sweeps[k])
        t0 = time.perf_counter()
        n.align(guesses[k])
        t4 += time.perf_counter() - t0
        d4 += 1
    return dict(value=done / t_align, unit="aligns/s", cores=nthreads, kind="port", value_at_4_threads=d4 / t4,
                sample="%d aligns of the cfg0 workload (oracle NDT, %d OpenMP threads); target build %.3f s not included" % (done, nthreads, t_build),
                target_build_s=t_build, iterations_last=n.nr_iterations)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port) on the host cores, all threads, same workload."""
    if rank != 0:
        return
    from oracle import pyoracle as O
    target, sweeps, guesses, _ = make_workload(0)
    nthreads = host_threads()
    n = O.NDT()
    n.setNumThreads(nthreads)
    n.setResolution(NDT_PARAMS["resolution"])
    n.setStepSize(NDT_PARAMS["step"])
    n.setTransformationEpsilon(NDT_PARAMS["eps"])
    n.setMaximumIterations(NDT_PARAMS["max_iter"])
    n.setInputTarget(target)
    n.setInputSource(sweeps[0])
    t0 = time.perf_counter()
    n.align(guesses[0])
    t_one = time.perf_counter() - t0
    warm = min(args.warmup, 1 if t_one > 5 else args.warmup)
    steps = max(1, args.steps)
    for w in range(max(0, warm - 1)):
        n.setInputSource(sweeps[w % len(sweeps)])
        n.align(guesses[w % len(sweeps)])
    t0 = time.perf_counter()
    for s in range(steps):
        n.setInputSource(sweeps[s % len(sweeps)])
        aligned = n.align(guesses[s % len(sweeps)])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        st = n.stats
        out = ndt_outputs(n, (n.nr_iterations, n.converged, st["derivative_evals"], st["line_search_trials"], st["hessian_recomputes"]))
        out["aligned_cloud"] = aligned
        write_outputs(args.dump_outputs, out)
    val = steps / dt
    line = {"impl": "reference", "metric": "ndt_scan_to_map_aligns_per_sec", "value": val, "unit": "aligns/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": WORKLOAD, "arithmetic": "f32 terms, f64 accumulation and optimiser state", "impl_note": "oracle port of pclomp::NDT (reference needs PCL/Eigen, unbuildable here)"},
            "cpu_baseline": {"value": val, "unit": "aligns/s", "cores": nthreads, "kind": "port",
                             "sample": "%d aligns of the cfg0 workload, %d OpenMP threads" % (steps, nthreads)},
            "e2e": {"value": val, "unit": "aligns/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def loop_closure_bench(rank, world, device, n_total, n_host_pairs):
    """configs[4]: GICP verification of `n_total` (scan, 41-key-frame sub-map) candidates - 4096 by default - through the
    collective C-ABI call lgs_batch_align_keyframes_dist: the candidate list is the same on every rank, the C++ host deals the
    pairs by size, each pair's last kernel stores its 96-byte record in the NCCL send buffer, one ncclAllGather returns all
    records to every rank.  STRONG scaling: n_total is fixed as N grows.  Returns pairs/s over all ranks (max-over-ranks time)."""
    import torch
    import torch.distributed as dist
    from lidar_graph_slam_b200 import api, synth
    n_az = _env_int("LGS_BENCH_LOOP_AZIMUTH", 900)
    d = synth.loop_keyframes(n_pairs=n_total, n_keyframes=41, n_azimuth=n_az, n_unique=2)
    ctx = api.Context(device)
    kf = api.KeyFrameArray(ctx)
    for c, P in zip(d["clouds"], d["poses"]):
        kf.push(c, P)
    comm = api.Comm.from_torch_distributed(device)
    # concurrent pairs per GPU, each a host thread on its own stream; never more than the host cores per rank
    n_workers = _env_int("LGS_BENCH_LOOP_WORKERS", 8 if host_threads() // max(world, 1) >= 4 else 4)
    kw = dict(search_key_frame_num=20, method=api.METHOD_GICP, n_workers=n_workers)
    kf.batch_align_dist(comm, d["scan_ids"][:4 * n_workers * world], d["center_ids"][:4 * n_workers * world], **kw)  # warm-up: every worker's device state

    def timed_call(fn):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device="cuda:%d" % device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return out, t.item()

    (recs, info), dt = timed_call(lambda: kf.batch_align_dist(comm, d["scan_ids"], d["center_ids"], **kw))
    conv = sum(1 for r in recs if r.converged)
    accepted = sum(1 for r in recs if r.converged and r.fitness <= 0.3)  # GBS:328 with score_threshold 0.3
    # algorithmic bytes of a pair (SURVEY.md section 8d "Loop pair"): sub-map assembly (32 B per point) + VoxelGrid 0.5 m
    # (16 N + 4 N + 4 N + 16 V) + k-NN covariances of both clouds (16 + 24 B per point) + every linearisation / error pass
    # (N_s (16 + 24 + 16 + 24)) + fitness (32 N_s)
    n_kf = 2 * 41
    sub_pts = float(np.mean([sum(len(d["clouds"][j]) for j in range(c - 20, c + 21) if 0 <= j < n_kf) for c in d["center_ids"][:64]]))
    scan_pts = float(np.mean([len(d["clouds"][s]) for s in d["scan_ids"][:64]]))
    one, _ = kf.assemble([j for j in range(d["center_ids"][0] - 20, d["center_ids"][0] + 21) if 0 <= j < n_kf], leaf=0.5).shape
    passes = float(np.mean([r.evaluations + r.line_search_trials for r in recs]))
    bytes_pair = 32 * sub_pts + 24 * sub_pts + 16 * one + 40 * (one + scan_pts) + passes * scan_pts * 80 + 32 * scan_pts
    peak, _ = measured_peak_hbm()
    pps = n_total / dt
    out = {"pairs_per_sec": pps, "n_pairs": n_total, "scaling": "strong", "seconds": dt, "converged": conv, "accepted_by_fitness_gate": accepted,
           "method": "FastGICP k=20, max_corr 2.0, eps 0.01, submap VoxelGrid 0.5 m (graph_based_slam.param.yaml)",
           "api": "lgs_batch_align_keyframes_dist (C-ABI; partition, verification and the ncclAllGather of the records all inside liblgs_b200.so)",
           "comm_nranks": info["world"], "nccl_version": comm.nccl_version, "pairs_rank0": info["n_local"], "verify_ms_rank0": info["verify_ms"],
           "gather_ms_rank0": info["gather_ms"], "gather_bytes": info["gather_bytes"], "workers_per_gpu": n_workers,
           "mean_scan_pts": scan_pts, "mean_submap_pts": sub_pts, "submap_pts_after_voxelgrid": int(one), "passes_per_pair": passes,
           "algorithmic_bytes_per_pair": bytes_pair, "achieved_gbs": bytes_pair * pps / 1e9, "frac_of_hbm_peak_all_gpus": bytes_pair * pps / 1e9 / (peak * world),
           "n_azimuth": n_az}
    # the same collective with the clouds of every pair coming from HOST arrays (each rank uploads only its own pairs: 17 MB of
    # sub-map per pair over PCIe) on a bounded sample
    if n_host_pairs > 0:
        try:
            scans, submaps, _ = synth.loop_pairs(n_pairs=n_host_pairs, n_keyframes=41, n_azimuth=n_az, n_unique=2)
            sizes = [(len(a), len(b)) for a, b in zip(scans, submaps)]
            mine = set(api.partition_pairs([a + b for a, b in sizes], rank, world))
            hs = [s if i in mine else None for i, s in enumerate(scans)]
            hm = [s if i in mine else None for i, s in enumerate(submaps)]
            api.batch_align_dist(comm, hs[:2 * n_workers * world], hm[:2 * n_workers * world], sizes=sizes[:2 * n_workers * world], n_workers=n_workers)
            (hrecs, hinfo), hdt = timed_call(lambda: api.batch_align_dist(comm, hs, hm, sizes=sizes, n_workers=n_workers))
            out["from_host_arrays"] = {"pairs_per_sec": n_host_pairs / hdt, "n_pairs": n_host_pairs, "converged": sum(1 for r in hrecs if r.converged),
                                       "api": "lgs_batch_align_dist", "h2d_bytes_per_pair": 16 * (sub_pts + scan_pts)}
        except Exception as e:
            out["from_host_arrays"] = {"error": repr(e)}
    comm.close()
    del kf
    import gc
    gc.collect()
    api.batch_release()
    torch.cuda.synchronize()
    return out


def gicp_odometry_bench(device, stream, ctx, n_sweeps):
    """configs[2] (the GICP half of BASELINE's metric): scan-to-scan FastGICP over `n_sweeps` (1000) consecutive 120 000-ray
    64-beam sweeps of a 1 km drive, each VoxelGrid 0.25 m + range crop (kitti.cpp:80-82), covariance reuse through
    swapSourceAndTarget (kitti.cpp:115-125).  A frame = H2D of the pinned host sweep + prefilter + setInputSource + align +
    swap; CUDA events per frame.  Also reports the accumulated trajectory's drift against the synthetic ground truth."""
    import torch
    from lidar_graph_slam_b200 import api, synth
    sweeps_dev, poses = synth.long_drive(n_sweeps, device="cuda:%d" % device)
    n_stage = min(n_sweeps, 64)  # a ring of pinned host buffers: the sweep of frame k arrives from host memory
    ring = [torch.empty((sweeps_dev.shape[1], 4), dtype=torch.float32).pin_memory() for _ in range(n_stage)]
    vg = api.VoxelGrid(ctx)
    vg.setLeafSize(0.25)
    vg.setRangeCrop(1.0)
    g = api.FastGICP(ctx)
    g.setMaxCorrespondenceDistance(1.0)

    def frame(k, host):
        vg.setInputCloud(host.cuda(device, non_blocking=True))  # host sweep -> device once; the filtered cloud stays there
        ds = vg.filter(want_membership=False)
        if k == 0:
            g.setInputTarget(ds)
            return None, ds.shape[0]
        g.setInputSource(ds)
        g.align()
        T = g.getFinalTransformation()
        g.swapSourceAndTarget()
        return T, ds.shape[0]

    import gc
    gc.collect()  # device buffers of earlier bench sections are released now, not inside a timed frame
    torch.cuda.synchronize()
    # warm-up across the drive: every staging buffer reaches its final size before the timed run (a buffer that grows inside a
    # timed frame costs a cudaFree + cudaMalloc: 2-5 ms, hundreds of ms in a process that holds the earlier sections' memory).
    # Pass 1 filters every sweep (the prefilter's buffers, and which sweep is largest after it); pass 2 runs whole frames on
    # the largest sweeps and on a sample of the drive.
    sizes = []
    for k in range(n_sweeps):
        vg.setInputCloud(sweeps_dev[k])
        sizes.append(vg.filter(want_membership=False).shape[0])
    big = [int(i) for i in np.argsort(sizes)[::-1][:3]]
    for k in [0] + big + list(range(0, n_sweeps, max(1, n_sweeps // 24))) + big[::-1] + [0, 1, 2, 3]:
        ring[k % n_stage].copy_(sweeps_dev[k])
        frame(k if k < 4 else 1, ring[k % n_stage])
    ring[0].copy_(sweeps_dev[0])
    frame(0, ring[0])
    ms, X, worst, worst_rot, n_pts, passes, host_ms = [], np.eye(4), 0.0, 0.0, [], 0, []
    for k in range(n_sweeps):
        ring[k % n_stage].copy_(sweeps_dev[k])  # D2H staging of the synthetic sweep, outside the timed region
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        h0 = time.perf_counter()
        T, npt = frame(k, ring[k % n_stage])
        h1 = time.perf_counter()
        e1.record(stream)
        torch.cuda.synchronize()
        n_pts.append(npt)
        if k:
            ms.append(e0.elapsed_time(e1))
            host_ms.append(1e3 * (h1 - h0))
            passes += g.result.evaluations + g.result.line_search_trials
            E = np.linalg.inv(np.linalg.inv(poses[k - 1]) @ poses[k]) @ T.astype(np.float64)
            worst = max(worst, float(np.linalg.norm(E[:3, 3])))
            skew = 0.5 * np.sqrt((E[2, 1] - E[1, 2]) ** 2 + (E[0, 2] - E[2, 0]) ** 2 + (E[1, 0] - E[0, 1]) ** 2)
            worst_rot = max(worst_rot, float(np.degrees(np.arctan2(skew, (np.trace(E[:3, :3]) - 1) / 2))))
            X = X @ T.astype(np.float64)
    ms = np.array(ms)
    D = np.linalg.inv(np.linalg.inv(poses[0]) @ poses[-1]) @ X
    n_mean = float(np.mean(n_pts))
    # algorithmic bytes of a frame (SURVEY.md section 8d): prefilter (16 N + 16 V) + k-NN covariances of the new cloud
    # (16 + 24 B per point) + every linearisation / error pass (N_s (16 + 24 + 16 + 24))
    n_rays = float(sweeps_dev.shape[1])
    bytes_frame = 16 * n_rays + 16 * n_mean + 40 * n_mean + (passes / max(len(ms), 1)) * n_mean * 80
    peak, _ = measured_peak_hbm()
    fps = len(ms) / (ms.sum() * 1e-3)
    slowest = [{"frame": int(i) + 1, "ms": float(ms[i]), "host_call_ms": float(host_ms[i])} for i in np.argsort(ms)[::-1][:3]]
    del sweeps_dev
    torch.cuda.empty_cache()
    return {"frames_per_sec": fps, "ms_per_frame": {"mean": float(ms.mean()), "median": float(np.median(ms)), "min": float(ms.min()), "max": float(ms.max())},
            "frames": int(len(ms)), "sweeps": n_sweeps, "slowest_frames": slowest, "p99_ms": float(np.percentile(ms, 99)), "mean_points_after_prefilter": n_mean, "passes_per_frame": passes / max(len(ms), 1),
            "max_frame_pose_error_m": worst, "max_frame_rotation_error_deg": worst_rot, "trajectory_drift_m": float(np.linalg.norm(D[:3, 3])), "distance_driven_m": float(n_sweeps - 1),
            "algorithmic_bytes_per_frame": bytes_frame, "achieved_gbs": bytes_frame * fps / 1e9, "frac_of_hbm_peak": bytes_frame * fps / 1e9 / peak,
            "method": "FastGICP k=20, max_corr 1.0; per frame: H2D of the 120000-ray pinned host sweep, VoxelGrid 0.25 m + range crop, setInputSource (device cloud), align, swapSourceAndTarget; poses[i] = poses[i-1] * T"}


def big_map_bench(device, stream, ctx, sweeps_dev, guesses, poses, reps=12):
    """configs[3]: NDT scan-to-submap against the 20 M-point rolling map at 1.0 m and 0.5 m: target build (voxelisation of all
    20 M resident points, what a key-frame change costs today) and aligns/s with the map resident, with their HBM fractions."""
    import torch
    from lidar_graph_slam_b200 import api, synth
    d = synth.rolling_map()
    tgt = torch.from_numpy(d["target"]).cuda(device)
    peak, _ = measured_peak_hbm()
    out = {"n_target": int(tgt.shape[0])}
    for res in (1.0, 0.5):
        ndt = api.NormalDistributionsTransform(ctx)
        ndt.setResolution(res)
        ndt.setStepSize(NDT_PARAMS["step"])
        ndt.setTransformationEpsilon(NDT_PARAMS["eps"])
        ndt.setMaximumIterations(NDT_PARAMS["max_iter"])
        ndt.setInputTarget(tgt)
        builds = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ndt.setInputTarget(tgt)
            e1.record(stream)
            torch.cuda.synchronize()
            builds.append(e0.elapsed_time(e1))
        gi = ndt.grid_info()
        src = torch.from_numpy(d["source"]).cuda(device)
        ndt.setInputSource(src)
        ndt.align(d["guess"])
        ndt.profile(2)
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ndt.setInputSource(src)
            ndt.align(d["guess"])
            e1.record(stream)
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        prof = ndt.profile(0)
        E = np.linalg.inv(d["T_true"]) @ ndt.getFinalTransformation().astype(np.float64)
        nl = max(prof["align_launches"], 1)
        alg = (prof["evaluations"] * prof["n_source"] * (16 + 7 * 8) + 40.0 * prof["terms"]) / nl
        kms = prof["align_ms"] / nl
        build_bytes = 16.0 * tgt.shape[0] + 48.0 * gi.n_voxels
        bms = float(np.median(builds))
        out["res_%.1f" % res] = {"target_build_ms": bms, "target_build_gbs": build_bytes / (bms * 1e-3) / 1e9, "target_build_frac_of_hbm_peak": build_bytes / (bms * 1e-3) / 1e9 / peak,
                                 "voxels": int(gi.n_voxels), "valid_voxels": int(gi.n_valid), "cell_table": "dense" if gi.dense else "hash",
                                 "aligns_per_sec": 1e3 / float(np.median(ms)), "ms_per_align_median": float(np.median(ms)), "iterations": int(ndt.result.iterations),
                                 "evaluations": int(ndt.result.evaluations + ndt.result.hessian_recomputes), "align_kernel_ms": kms,
                                 "align_kernel_gbs": alg / (kms * 1e-3) / 1e9 if kms > 0 else 0.0, "align_kernel_frac_of_hbm_peak": alg / (kms * 1e-3) / 1e9 / peak if kms > 0 else 0.0,
                                 "pose_error_m": float(np.linalg.norm(E[:3, 3]))}
        del ndt
    del tgt
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--loop-pairs", type=int, default=_env_int("LGS_BENCH_LOOP_PAIRS", 4096),
                    help="loop-closure candidates in TOTAL (BASELINE configs[4]: 4096; strong scaling over --gpus; 0 disables)")
    ap.add_argument("--loop-host-pairs", type=int, default=_env_int("LGS_BENCH_LOOP_HOST_PAIRS", 128), help="sample of pairs verified from host arrays")
    ap.add_argument("--odometry-sweeps", type=int, default=_env_int("LGS_BENCH_ODOMETRY_SWEEPS", 1000), help="configs[2]: sweeps of the GICP odometry run (0 disables)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-big-map", action="store_true", help="skip configs[3] (20 M-point map)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    rank, world, local_rank = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from lidar_graph_slam_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    W = max(args.warmup, 3)
    K = max(args.steps, 1)

    target, sweeps, guesses, poses = make_workload(rank)
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    ctx = api.Context(local_rank, stream.cuda_stream)
    ndt = api.NormalDistributionsTransform(ctx)
    ndt.setResolution(NDT_PARAMS["resolution"])
    ndt.setStepSize(NDT_PARAMS["step"])
    ndt.setTransformationEpsilon(NDT_PARAMS["eps"])
    ndt.setMaximumIterations(NDT_PARAMS["max_iter"])
    ndt.setNeighborhoodSearchMethod(api.NDT_DIRECT7)

    # target build (timed separately: setInputTarget = H2D of 1M points + voxelisation)
    tgt_pinned = torch.from_numpy(target).pin_memory()
    ndt.setInputTarget(tgt_pinned.numpy())
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    ndt.setInputTarget(tgt_pinned.numpy())
    ev1.record(stream)
    torch.cuda.synchronize()
    target_build_ms = ev0.elapsed_time(ev1)
    gi = ndt.grid_info()

    sweeps_pinned = [torch.from_numpy(s).pin_memory() for s in sweeps]
    sweeps_dev = [t.cuda(local_rank, non_blocking=True) for t in sweeps_pinned]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % local_rank)  # > 126 MB L2
    torch.cuda.synchronize()

    def step_dev(i):
        ndt.setInputSource(sweeps_dev[i % len(sweeps_dev)])
        ndt.align(guesses[i % len(guesses)])

    aligned_pinned = torch.empty((max(len(x) for x in sweeps), 4), dtype=torch.float32).pin_memory()

    def step_host(i):
        # the reference's call sequence (LSM:162-172): setInputSource(host cloud) -> align(aligned_cloud, guess) ->
        # getFinalTransformation; the aligned cloud comes back to the host like the output argument of pcl's align
        ndt.setInputSource(sweeps_pinned[i % len(sweeps_pinned)].numpy())
        ndt.align(guesses[i % len(guesses)], want_output=True, out=aligned_pinned.numpy())
        return ndt.getFinalTransformation()

    def last_step_outputs(prefix):
        r = ndt.result
        return ndt_outputs(ndt, (r.iterations, r.converged, r.evaluations, r.line_search_trials, r.hessian_recomputes), prefix)

    def timed(fn, steps, warm):
        for i in range(warm):
            fn(i)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        l0 = ctx.launch_count
        evals = 0
        for i in range(steps):
            flush.zero_()  # L2 flush, outside the event pair ...
            torch.cuda.current_stream().synchronize()  # ... and complete before the step's host-side set-up starts
            starts[i].record(stream)
            fn(i)
            stops[i].record(stream)
            evals += ndt.result.evaluations + ndt.result.hessian_recomputes
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        per = np.array([a.elapsed_time(b) for a, b in zip(starts, stops)])
        return per, ctx.launch_count - l0, evals

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # the dominant kernel is timed live in the timed region: CUDA events on the launching stream around every
    # ndt_align_kernel launch (one launch = one whole align: all its evaluations and the optimiser between them)
    ndt.profile(2)
    per_dev, launches, evals_dev = timed(step_dev, K, W)
    prof = ndt.profile(0)
    dump = rank == 0 and args.dump_outputs
    outputs = last_step_outputs("") if dump else {}
    per_host, _, evals_host = timed(step_host, K, W)
    if dump:
        outputs.update(last_step_outputs("e2e_"))
        outputs["e2e_aligned_cloud"] = aligned_pinned.numpy()[:len(sweeps[(K - 1) % len(sweeps)])].copy()
    clocks = sampler.stop() if rank == 0 else None
    if dump:
        write_outputs(args.dump_outputs, outputs)
    ms_dev, ms_host = float(per_dev.sum()), float(per_host.sum())

    # accuracy sanity of the timed workload (not a parity test: those live in tests/)
    step_dev(0)
    E = np.linalg.inv(poses[0]) @ ndt.getFinalTransformation().astype(np.float64)
    t_err = float(np.linalg.norm(E[:3, 3]))

    # roofline of the dominant kernel.  Algorithmic bytes of one evaluation (SURVEY.md section 8d): point float4 + 7 (key, slot)
    # probes per point + one 40-byte voxel record per accepted (point, voxel) term; a launch runs all evaluations of an align
    n_src = prof["n_source"]
    n_launch = max(prof["align_launches"], 1)
    alg_bytes = (prof["evaluations"] * n_src * (16 + 7 * 8) + 40.0 * prof["terms"]) / n_launch
    kern_ms = prof["align_ms"] / n_launch
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9 if kern_ms > 0 else 0.0
    hbar = prof["terms"] / max(prof["evaluations"] * n_src, 1)
    peak, peak_src = measured_peak_hbm()
    traffic, traffic_src = ncu_traffic()

    # where the align kernel's time goes (its own clock64 accounting, last align of the timed pass): the share the evaluating
    # CTAs spend in the evaluation body, and what the body alone achieves against the roofline
    step_dev(0)
    bd = ndt.align_breakdown()
    body_share = bd["raw"][0] / bd["total"] if bd["total"] > 0 else 0.0
    breakdown = {"evaluation_body_share_of_kernel": body_share,
                 "optimiser_cta": {k: bd[k] / bd["total"] for k in ("wait_grid", "add_rows", "optimiser", "publish")} if bd["total"] > 0 else None,
                 "evaluation_body_gbs": achieved / body_share if body_share > 0 else None,
                 "evaluation_body_frac_of_peak": achieved / body_share / peak if body_share > 0 else None,
                 "note": "SM cycles of CTA 0 (evaluating) in deriv_eval / all cycles of the optimiser CTA; the rest of an evaluation is the grid-wide hand-over: "
                         "waiting for the slowest CTA, adding the 147 rows, the Newton / More-Thuente step, publishing the next pose"}

    # the evaluation body alone, one launch per evaluation (the host steps the optimiser): what a single evaluation costs
    ndt.profile(1)
    for i in range(min(K, 12)):
        step_dev(i)
    prof1 = ndt.profile(0)

    # max over ranks
    t = torch.tensor([ms_dev, ms_host], dtype=torch.float64, device="cuda:%d" % local_rank)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev_max, ms_host_max = t.tolist()
    total_steps = K * world

    loop = None
    if args.loop_pairs > 0:
        try:
            loop = loop_closure_bench(rank, world, local_rank, args.loop_pairs, args.loop_host_pairs)
        except Exception as e:  # the headline line must still be printed
            loop = {"error": repr(e)}

    gicp_odo = None
    if rank == 0 and world == 1:  # reported at N = 1 only (single-scan odometry does not shard)
        try:
            gicp_odo = gicp_odometry_bench(local_rank, stream, ctx, args.odometry_sweeps) if args.odometry_sweeps > 0 else None
        except Exception as e:
            gicp_odo = {"error": repr(e)}

    big = None
    if rank == 0 and world == 1 and not args.no_big_map:
        try:
            big = big_map_bench(local_rank, stream, ctx, sweeps_dev, guesses, poses)
        except Exception as e:
            big = {"error": repr(e)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:  # reported at N = 1 only
        cpu = cpu_baseline(target, sweeps, guesses)

    if rank == 0:
        line = {
            "metric": "ndt_scan_to_map_aligns_per_sec", "value": total_steps / (ms_dev_max * 1e-3), "unit": "aligns/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_dev_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "arithmetic": "f32 terms, f64 accumulation and optimiser state", "ndt": NDT_PARAMS,
                       "sweep_pool": "%d distinct re-cast sweeps, each with its own perturbed guess" % len(sweeps), "n_source": int(n_src), "n_target": int(target.shape[0]),
                       "voxels": int(gi.n_voxels), "valid_voxels": int(gi.n_valid), "cell_table": "dense" if gi.dense else "hash",
                       "l2": "flushed between steps (256 MiB memset outside the per-step CUDA-event pairs); within an align the 1.9 MB sweep and the voxel table are re-read from L2 by design",
                       "parallelism": "1 sequence per GPU (replicas, no collective)" if world > 1 else "single GPU",
                       "evaluations_per_align": evals_dev / K, "launches_per_align": launches / K,
                       "evaluator": ("device-resident align: ONE cooperative launch of ndt_align_kernel per align - the grid evaluates, CTA 0 runs "
                                     "the Newton / More-Thuente state machine between evaluations, nothing crosses PCIe until the result record "
                                     "(LGS_NDT_DEVICE_ALIGN=0: the host steps the same machine with one launch per evaluation)"),
                       "target_build_ms": target_build_ms, "pose_error_m": t_err,
                       "ms_per_step_spread": {"min": float(per_dev.min()), "median": float(np.median(per_dev)), "max": float(per_dev.max()),
                                              "p90": float(np.percentile(per_dev, 90))},
                       "e2e_ms_per_step_spread": {"min": float(per_host.min()), "median": float(np.median(per_host)), "max": float(per_host.max())}},
            "e2e": {"value": total_steps / (ms_host_max * 1e-3), "unit": "aligns/s", "h2d_bytes_per_step": int(n_src) * 16 + 64,
                    "d2h_bytes_per_step": int(n_src) * 16 + 32 * 16,
                    "call": "setInputSource(pinned host sweep) -> align(aligned cloud to pinned host memory, guess) -> getFinalTransformation (LSM:162-172)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "ndt_align_kernel<true> (one launch = one align: %.2f derivative evaluations + the optimiser between them)" % (prof["evaluations"] / n_launch),
                         "kernel_ms": kern_ms, "launches_timed": prof["align_launches"], "timed": "live, CUDA events on the launching stream around every launch of the timed region",
                         "algorithmic_bytes": alg_bytes, "h_bar": hbar, "peak_source": peak_src, "inside_the_kernel": breakdown,
                         "single_evaluation_kernels_ms": {"ndt_derivatives_kernel<0> (score + g + H)": prof1["hess_ms"] / max(prof1["hess_launches"], 1),
                                                          "ndt_derivatives_kernel<1> (score + g)": prof1["grad_ms"] / max(prof1["grad_launches"], 1),
                                                          "ndt_derivatives_kernel<2> (f64 Hessian)": prof1["h64_ms"] / max(prof1["h64_launches"], 1),
                                                          "note": "the same evaluation body launched once per evaluation (host-stepped optimiser), separate pass"}},
            "cpu_baseline": cpu, "clocks": clocks, "loop_closure": loop, "gicp_odometry": gicp_odo, "big_map_20m": big,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
