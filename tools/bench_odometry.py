#!/usr/bin/env python
"""Offline odometry throughput (lgs_odometry_run / _dev / _dist): S sequences of 120 000-ray sweeps (synth.long_drive, 1 m
apart) with the scan-matcher YAML parameters (NDT DIRECT7, resolution 2.0, eps 0.01, 64 iterations, VoxelGrid 0.1 m,
range crop 1 m, key frames every 1 m, window 20); --method gicp / gicp_omp runs the other two scan-matcher methods.

    python tools/bench_odometry.py --sequences 2 --frames 100            # one GPU: device and host forms + per-frame split
    python tools/bench_odometry.py --scaling 1,2,4,8 --frames 100        # aggregate frames/s, weak (S = N) and strong (fixed S)

The scaling legs run this file under torch.distributed.run, one rank per GPU; a leg needing more GPUs than the box has is
reported as not run.  Prints one JSON line per measurement, with the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def drives(n_seq, n_frames, device, azimuth):
    from lidar_graph_slam_b200 import synth
    seqs, inits = [], []
    for s in range(n_seq):
        sw, poses = synth.long_drive(n_frames, device=device, n_azimuth=azimuth, seed=synth.SEED + s)
        seqs.append(sw)
        inits.append(poses[0])
    return seqs, inits


METHODS = {"ndt": 0, "gicp": 1, "gicp_omp": 3}


def single(args):
    import torch
    from lidar_graph_slam_b200 import api
    m = METHODS[args.method]
    torch.cuda.set_device(0)
    seqs, inits = drives(args.sequences, args.frames, "cuda:0", args.azimuth)
    dev = [[s[k] for k in range(s.shape[0])] for s in seqs]
    host = [[torch.empty_like(x, device="cpu").copy_(x).numpy() for x in q] for q in dev]
    n = sum(len(q) for q in dev)
    os.environ["LGS_ODOMETRY_PROFILE"] = "0"
    api.odometry([q[:6] for q in dev], method=m, initial_poses=inits)  # warm-up: modules, buffers
    out = {"card": card(), "method": args.method, "sequences": args.sequences, "frames_per_sequence": args.frames, "rays": int(dev[0][0].shape[0])}
    for form, data in (("device", dev), ("host", host)):
        best = None
        for _ in range(args.repeat):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            recs = api.odometry(data, method=m, initial_poses=inits)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        out["%s_frames_per_s" % form] = n / best
        out["%s_keyframes" % form] = int((recs["keyframe_id"] >= 0).sum())
        out["%s_dropped" % form] = int((recs["converged"] == 0).sum())
    # per-frame split from CUDA events, in a run of its own (the events synchronise every frame)
    os.environ["LGS_ODOMETRY_PROFILE"] = "1"
    api.odometry_profile()
    api.odometry(dev, method=m, initial_poses=inits)
    p = api.odometry_profile()
    out.update(profiled_frames=p["frames"], prefilter_ms_per_frame=p["prefilter_ms"] / p["frames"], align_ms_per_frame=p["align_ms"] / p["frames"],
               keyframe_ms_per_frame=p["keyframe_ms"] / p["frames"])
    print(json.dumps(out))


def rank_leg(args):
    """One rank of a scaling leg: its share of S sequences through lgs_odometry_run_dist_dev."""
    import torch
    import torch.distributed as dist
    from lidar_graph_slam_b200 import api, synth
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    S = args.sequences
    sizes = [args.frames * args.azimuth * 64] * S  # equal sequences: the partition deals them round-robin
    mine = api.partition_pairs(sizes, rank, world)
    seqs, inits, n_points = [], [], []
    for s in range(S):
        inits.append(synth.long_drive_pose(0, args.frames))
        if s in mine:
            sw, _ = synth.long_drive(args.frames, device="cuda:%d" % local, n_azimuth=args.azimuth, seed=synth.SEED + s)
            seqs.append([sw[k] for k in range(args.frames)])
            n_points.append([int(sw.shape[1])] * args.frames)
        else:
            seqs.append(None)
            n_points.append([args.azimuth * 64] * args.frames)
    ctx = api.Context(local)
    comm = api.Comm.from_torch_distributed(local)
    if mine:
        api.odometry([seqs[mine[0]][:6]], method=METHODS[args.method], initial_poses=[inits[mine[0]]], ctx=ctx)  # warm-up
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    recs, info = api.odometry_dist(comm, seqs, n_points=n_points, method=METHODS[args.method], initial_poses=inits, ctx=ctx)
    dt = time.perf_counter() - t0
    if rank == 0:
        print(json.dumps({"card": card(), "gpus": world, "sequences": S, "frames": len(recs), "wall_s": dt, "method": args.method, "frames_per_s": len(recs) / dt,
                          "gather_ms": info["gather_ms"], "scaling": args.mode}))
    comm.close()
    if world > 1:
        dist.destroy_process_group()


def scaling(args):
    import torch
    have = torch.cuda.device_count()
    for n in [int(v) for v in args.scaling.split(",")]:
        for mode, S in (("weak", n), ("strong", args.strong_sequences)):
            if n > have:
                print(json.dumps({"gpus": n, "scaling": mode, "result": "not run: the box has %d GPUs" % have}))
                continue
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                   "--master-port", str(29560 + n), os.path.abspath(__file__), "--rank-leg", "--mode", mode, "--sequences", str(S),
                   "--frames", str(args.frames), "--azimuth", str(args.azimuth), "--method", args.method]
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
            lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
            print(lines[-1] if r.returncode == 0 and lines else json.dumps({"gpus": n, "scaling": mode, "error": r.stdout[-1500:]}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sequences", type=int, default=2)
    ap.add_argument("--frames", type=int, default=100)
    ap.add_argument("--azimuth", type=int, default=1875, help="64 beams x 1875 = 120 000 rays")
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--method", default="ndt", choices=["ndt", "gicp", "gicp_omp"])
    ap.add_argument("--scaling", default="", help="GPU counts, e.g. 1,2,4,8")
    ap.add_argument("--strong-sequences", type=int, default=8)
    ap.add_argument("--rank-leg", action="store_true")
    ap.add_argument("--mode", default="weak")
    args = ap.parse_args()
    if args.rank_leg:
        rank_leg(args)
    elif args.scaling:
        scaling(args)
    else:
        single(args)


if __name__ == "__main__":
    main()
