#!/usr/bin/env python
"""Multi-rank leg of the offline odometry tests (run under torch.distributed.run, one rank per GPU; also works as a single
process).  Every rank calls the collective lgs_odometry_run_dist with the same sequence list (clouds only for the sequences
it owns) and must receive every record; rank 0 writes them, the one-rank lgs_odometry_run records (when --solo) and the
local shares to --out for tests/test_gpu_odometry_dist.py.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
        tests/dist_odometry.py --out /tmp/odo_w2.npz
"""
import argparse
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sequences", type=int, default=9)
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--azimuth", type=int, default=450)
    ap.add_argument("--solo", type=int, default=0, help="also run lgs_odometry_run on this rank and store its records")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    import torch
    import torch.distributed as dist
    from lidar_graph_slam_b200 import api
    from odometry_reference import make_drive
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # sequences of different lengths and seeds, so that the partition has sizes to sort
    seqs, inits = [], []
    for s in range(args.sequences):
        n = args.frames + (s % 3)
        sw, poses = make_drive(n, n_azimuth=args.azimuth, spacing=0.4 + 0.05 * (s % 4), seed=100 + s, device="cuda:%d" % local)
        seqs.append([sw[k].cpu().numpy() for k in range(n)])
        inits.append(poses[0])
    sizes = [sum(len(c) for c in q) for q in seqs]
    mine = api.partition_pairs(sizes, rank, world)
    n_points = [[len(c) for c in q] for q in seqs]
    host = [q if s in mine else None for s, q in enumerate(seqs)]
    ctx = api.Context(local)
    comm = api.Comm.from_torch_distributed(local)
    recs, info = api.odometry_dist(comm, host, n_points=n_points, initial_poses=inits, ctx=ctx)
    dev = [[torch.from_numpy(c).cuda(local) for c in q] if s in mine else None for s, q in enumerate(seqs)]
    recs_dev, _ = api.odometry_dist(comm, dev, n_points=n_points, initial_poses=inits, ctx=ctx)
    assert recs.tobytes() == recs_dev.tobytes(), "host and device forms differ"
    assert info["n_local_sequences"] == len(mine) and info["n_received"] == len(recs), info
    digest = hashlib.sha256(recs.tobytes()).hexdigest()
    print("rank %d/%d: %d sequences, %d frames local, run %.1f ms, gather %.2f ms, sha256 %s" %
          (rank, world, info["n_local_sequences"], info["n_local_frames"], info["run_ms"], info["gather_ms"], digest[:16]))
    shares = [np.array(mine, np.int32)]
    if world > 1:
        got = [None] * world
        dist.all_gather_object(got, (digest, mine))
        assert all(g[0] == digest for g in got), "ranks received different records"
        shares = [np.array(g[1], np.int32) for g in got]
    solo = api.odometry(seqs, initial_poses=inits, ctx=ctx) if args.solo else np.zeros(0, api.ODOMETRY_FRAME)
    if rank == 0 and args.out:
        np.savez(args.out, records=recs, solo=solo, sizes=np.array(sizes, np.int64), **{"share%d" % r: s for r, s in enumerate(shares)})
    comm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
