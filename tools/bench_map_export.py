#!/usr/bin/env python
"""Map export throughput (lgs_keyframes_export_map, the save_map service of GBS:469-501): key frames of a synthetic drive
(synth.long_drive sweeps, 1 m apart, prefiltered with the prefilter node's VoxelGrid 0.1 m + 1 m range crop) at their true
poses, exported at a leaf that needs the 64-bit grid and at one the 32-bit grid takes (0.5 m), alternating.  The synthetic
world is about 5 m tall, so a 400-frame drive stays under INT32_MAX cells at 0.1 m (6.5e8 cells); 0.05 m (5e9 cells) is
the leaf that needs the 64-bit grid here.  Each leg reports whether it took the 64-bit path.

    python tools/bench_map_export.py --frames 400 --reps 7

The assembled map is far larger than the 126 MB L2, so every export reads it from HBM.  Each run is timed with CUDA
events around the call on the context's stream (the call waits for its own small results, so the events bracket all of
its work).  Reports per leaf: ms (median, min, max), points/s, and algorithmic bytes computed from N (assembled points),
V (output points) and the number of sort passes, as a fraction of the same measured HBM peak bench.py uses.  Prints one
JSON line, with the card name and power limit read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def algorithmic_bytes(n, v, cells):
    """Bytes the export has to move: assembly (float4 in + out), crop + bbox (float4 + keep flag), key kernel, radix passes
    (8 B read + 8 B written per pair per pass, plus one key read for the histograms of each sort), segment heads, centroids.
    Beyond INT32_MAX cells the key kernel also writes the 8-byte key, the high words are gathered between the two sorts,
    and the segment heads read whole keys through the sorted indices."""
    bits = max(1, int(cells - 1).bit_length())
    wide = cells > 2 ** 31 - 1
    if wide:
        passes = 4 + (max(bits - 32, 0) + 7) // 8
        key = 16 + 1 + 4 + 4 + 8
        sort = passes * 16 + (2 * 4 if bits > 32 else 4) + (16 if bits > 32 else 0)
        heads = 4 + 2 * 8
    else:
        passes = (bits + 7) // 8
        key = 16 + 1 + 4 + 4
        sort = passes * 16 + 4
        heads = 8
    per_point = 32 + 17 + key + sort + heads + 4 + 16
    return float(per_point * n + 20 * v), passes, bits


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--azimuth", type=int, default=1875)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--leaves", default="0.05,0.1,0.5")
    args = ap.parse_args()

    import torch
    from bench import measured_peak_hbm
    from lidar_graph_slam_b200 import api, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench_map_export needs a CUDA device")
    torch.cuda.set_device(0)
    stream = torch.cuda.current_stream()
    ctx = api.Context(0, stream=stream.cuda_stream)
    sweeps, poses = synth.long_drive(args.frames, device="cuda:0", n_azimuth=args.azimuth)
    vg = api.VoxelGrid(ctx)
    vg.setLeafSize(0.1)
    vg.setRangeCrop(1.0)
    kf = api.KeyFrameArray(ctx)
    for k in range(sweeps.shape[0]):
        vg.setInputCloud(sweeps[k])
        kf.push(vg.filter(False).contiguous(), poses[k])
    del sweeps
    torch.cuda.synchronize()
    L = ctx._L
    leaves = [float(x) for x in args.leaves.split(",")]
    out, n_out, info = C.c_void_p(), C.c_int64(), api.VoxelGridInfo()

    def export(leaf):
        rc = L.lgs_keyframes_export_map(kf._h, None, 0, leaf, C.byref(out), C.byref(n_out), C.byref(info))
        if rc != 0:
            raise RuntimeError(L.lgs_last_error().decode())

    c, total = C.c_int64(), C.c_int64()
    L.lgs_keyframes_size(kf._h, C.byref(c), C.byref(total))
    n = int(total.value)
    res = {}
    for leaf in leaves:  # warm-up: modules, arenas
        export(leaf)
        res[leaf] = {"ms": [], "v": int(n_out.value), "status": int(info.status), "div_b": list(info.div_b)}
    torch.cuda.synchronize()
    launches0 = ctx.launch_count
    for _ in range(args.reps):
        for leaf in leaves:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            export(leaf)
            e1.record(stream)
            e1.synchronize()
            res[leaf]["ms"].append(e0.elapsed_time(e1))
    launches = (ctx.launch_count - launches0) / args.reps
    peak, peak_src = measured_peak_hbm()
    legs = {}
    for leaf in leaves:
        r = res[leaf]
        ms = sorted(r["ms"])
        med = ms[len(ms) // 2]
        cells = 1
        for d in r["div_b"]:
            cells *= d
        nbytes, passes, bits = algorithmic_bytes(n, r["v"], cells)
        legs["leaf_%g" % leaf] = {
            "status": r["status"], "div_b": r["div_b"], "cells": cells, "key_bits": bits, "wide_path": cells > 2 ** 31 - 1, "sort_passes": passes,
            "points_in": n, "points_out": r["v"], "ms_median": med, "ms_min": ms[0], "ms_max": ms[-1], "ms_all": r["ms"],
            "points_per_s": n / (med * 1e-3), "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / (med * 1e-3) / 1e9,
            "frac_of_hbm_peak": nbytes / (med * 1e-3) / 1e9 / peak}
    print(json.dumps({"bench": "map_export", "card": card(), "frames": args.frames, "rays_per_sweep": 64 * args.azimuth, "map_points": n,
                      "map_mb": n * 16 / 1e6, "reps": args.reps, "launches_per_rep_all_leaves": launches, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
                      "legs": legs}))


if __name__ == "__main__":
    main()
