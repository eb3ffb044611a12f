"""Sequential NDT aligns against lgs_ndt_align_many on one GPU; prints one JSON line.

    python tools/bench_ndt_align_many.py [--reps 5] [--groups 2,4,8,16]

For K seeds (random guesses around the true pose) on one map it times K calls of align() and one align_guesses() call of the
same K guesses, alternately, `reps` times each, and reports aligns/s of both, launches per call and the spread (min / max) over
the repetitions.  Two workloads: BASELINE configs[0] (120 000-point sweep, 1 000 000-point map) and a loop-closure-sized
source (every fifth point of it, ~24 000 points).  --groups also times K = 16 under each LGS_NDT_MANY_MAX_GROUPS value.
Every align_guesses record is checked bitwise against its single align.  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _guesses(T, seed, count):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        d = np.eye(4)
        yaw = rng.uniform(-1, 1) * np.radians(2.0)
        d[:2, :2] = [[np.cos(yaw), -np.sin(yaw)], [np.sin(yaw), np.cos(yaw)]]
        d[:3, 3] = rng.uniform(-1, 1, 3) * np.array([0.5, 0.5, 0.05])
        out.append((d @ np.asarray(T, np.float64)).astype(np.float32))
    return out


def _key(r):
    return (np.array(r.T, np.float32).tobytes(), np.float64(r.trans_probability).tobytes(), r.iterations, r.evaluations, r.line_search_trials, r.hessian_recomputes)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ks", default="1,2,4,8,16")
    ap.add_argument("--groups", default="2,4,8,16")
    args = ap.parse_args()
    from lidar_graph_slam_b200 import api, synth

    d = synth.ndt_scan_to_map()
    workloads = {"cfg0_120k": d["source"], "loop_closure_24k": np.ascontiguousarray(d["source"][::5])}
    ctx = api.default_context()
    out = dict(gpu=subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip(),
               reps=args.reps, rows=[])
    for name, src in workloads.items():
        g = api.NormalDistributionsTransform()
        for x in (g,):
            x.setResolution(1.0)
            x.setTransformationEpsilon(0.01)
            x.setMaximumIterations(64)
            x.setInputTarget(d["target"])
            x.setInputSource(src)
        seeds = _guesses(d["guess"], 11, 16)
        g.align(seeds[0])
        g.align_guesses(seeds[:2])  # warm-up: modules, grids, scratch

        def timed(fn):
            t0 = time.perf_counter()
            l0 = ctx.launch_count
            r = fn()
            return time.perf_counter() - t0, ctx.launch_count - l0, r

        def measure(K, label, groups=None):
            if groups is not None:
                os.environ["LGS_NDT_MANY_MAX_GROUPS"] = str(groups)
            else:
                os.environ.pop("LGS_NDT_MANY_MAX_GROUPS", None)
            gs = seeds[:K]
            seq_t, many_t = [], []
            identical = True
            for _ in range(args.reps):  # alternate the two forms
                t, ls, rs = timed(lambda: [(g.align(x), g.result)[1] for x in gs])
                seq_t.append(t)
                t, lm, rm = timed(lambda: g.align_guesses(gs))
                many_t.append(t)
                identical &= [_key(a) for a in rs] == [_key(b) for b in rm]
            out["rows"].append(dict(workload=name, n_source=int(len(src)), K=K, max_groups=groups if groups is not None else "default",
                                    seq_aligns_per_s=K / float(np.median(seq_t)), many_aligns_per_s=K / float(np.median(many_t)),
                                    speedup=float(np.median(seq_t) / np.median(many_t)),
                                    seq_spread_ms=[1e3 * min(seq_t), 1e3 * max(seq_t)], many_spread_ms=[1e3 * min(many_t), 1e3 * max(many_t)],
                                    seq_launches=ls, many_launches=lm, bit_identical=bool(identical), label=label))

        for K in [int(k) for k in args.ks.split(",") if k]:
            measure(K, "ks")
        for M in [int(m) for m in args.groups.split(",") if m]:
            measure(16, "groups", M)
    os.environ.pop("LGS_NDT_MANY_MAX_GROUPS", None)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
