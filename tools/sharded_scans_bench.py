#!/usr/bin/env python
"""A whole sequence through parallel.ShardedScans, plain or under ``torchrun --nproc-per-node N``:

  evaluate   ShardedScans.evaluate on bench.py's config-2 workload: 8-scan batches of 65 536-point os1-64 scans
             (x, y, z, label, pinned host memory, built as tools/predict_radius_bench.py builds them) against the
             config-2 base map, radius submaps, forward and metric partials on the GPU
  replay     ShardedScans.replay on the config-3 workload in the sensor frame (tools/filter_scans_bench.py's 32 hdl-32
             scans and poses, device-resident), 8-scan batches, eps at the median score of the first batch

Every rank builds the same sequence (``--scans`` scans, the distinct scans cycled) and runs its own batches (batch k on
rank k mod N).  Reported per call: scans/s of the whole sequence (best of ``--rounds``, the slowest rank's time), and
the gather's own time: from the end of the last call to the reassembled results on rank 0 (the CUDA events of
ShardedScans.gather_events).  Also: the card's name and power limit, read with nvidia-smi in the same run.  Prints one
JSON line on rank 0.  Needs a GPU; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

EPS = 0.84          # bench.py's metric threshold


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=256, help="scans per sequence")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--lanes", type=int, default=3)
    args = ap.parse_args()

    import torch
    import bench
    from filter_scans_bench import pose_matrix
    from prune_batch_bench import gpu_card
    from sps_b200 import synth
    from sps_b200.datasets import RadiusSubmap
    from sps_b200.engine import MapHash
    from sps_b200.parallel import ShardedScans

    d = bench.Dist()
    # config 2: the scans of bench.make_batches' first two batches (rank 0's seeds on every rank: one sequence)
    world = synth.World(0)
    map2 = synth.base_map(world, bench.SENSOR, n_poses=12, seed=0, voxel=bench.VOXEL).astype(np.float32)
    pool2 = []
    for b in bench.make_batches(0):
        scan = b[b[:, 4] == 1]
        for j in range(bench.BATCH):
            pool2.append(np.ascontiguousarray(scan[scan[:, 0] == j][:, [1, 2, 3, 5]]))
    eval_scans = [torch.as_tensor(pool2[i % len(pool2)]).pin_memory() for i in range(args.scans)]
    # config 3 in the sensor frame
    traj = synth.loop_trajectory(radius=35.0, n=400)
    map3 = synth.base_map(world, "hdl-32", n_poses=400, seed=0, voxel=bench.VOXEL, trajectory=traj,
                          target_voxels=1_000_000)
    poses3 = np.stack([pose_matrix(traj(7 * i)) for i in range(32)])
    rng = np.random.default_rng(0)
    pool3 = []
    for i in range(32):
        xyz = synth.scan(world, "hdl-32", traj(7 * i), seed=i).astype(np.float64)
        h = np.hstack([xyz, np.ones((len(xyz), 1))]) @ np.linalg.inv(poses3[i]).T
        pool3.append(torch.as_tensor(np.hstack([h[:, :3] / h[:, 3:], rng.random((len(xyz), 1))]).astype(np.float32)).cuda())
    replay_scans = [pool3[i % 32] for i in range(args.scans)]
    replay_poses = torch.as_tensor(np.stack([poses3[i % 32] for i in range(args.scans)])).cuda()

    n_max = max(len(s) for s in eval_scans) * bench.BATCH * 6
    model, _, _, _ = bench.setup_model(argparse.Namespace(lanes=args.lanes, no_graphs=False, backend=0), n_max, d.local,
                                       bench.random_state_dict())
    sub = RadiusSubmap(torch.as_tensor(map2).cuda(), bench.VOXEL)
    mh = MapHash(torch.as_tensor(map3).cuda(), bench.VOXEL)
    eps3 = float(model.filter_scans_async(replay_scans[:args.batch], replay_poses[:args.batch], mh, 0.84)
                 .result().scan_scores.median())
    runs = {"evaluate": (ShardedScans(model, EPS, args.batch), lambda ss: ss.evaluate(eval_scans, sub)),
            "replay": (ShardedScans(model, eps3, args.batch), lambda ss: ss.replay(replay_scans, replay_poses, mh))}
    report = {}
    for name, (ss, fn) in runs.items():
        fn(ss)                                   # warm-up: lanes, contexts, NCCL communicators
        ms, gather_ms = [], []
        for _ in range(args.rounds):
            ms.append(d.timed(lambda k: fn(ss), 1))
            start, end = ss.gather_events
            gather_ms.append(d.max_ms(start.elapsed_time(end)))
        best = int(np.argmin(ms))
        res = fn(ss)
        report[name] = {"scans_per_s": round(args.scans / (ms[best] * 1e-3), 1), "ms_sequence": round(ms[best], 3),
                        "ms_sequence_rounds": [round(m, 3) for m in ms], "gather_ms": round(gather_ms[best], 4),
                        "metrics": res.metrics}
        if name == "replay":
            report[name]["kept_fraction"] = None if res.kept is None else len(res.kept) / len(res.scan_scores)
    result = {"metric": "scans/s", "n_gpus": d.world, "scans": args.scans, "batch": args.batch, "lanes": args.lanes,
              "gpu": gpu_card(d.local), "eps_replay": eps3,
              "workload": {"evaluate": bench.WORKLOAD + ", pinned host scans",
                           "replay": "config3 in the sensor frame: hdl-32 scans with their poses against a 1M-voxel "
                                     "base map, device-resident, eps at the median score"},
              **report}
    d.close()
    if d.rank == 0:
        print(json.dumps(result))


if __name__ == "__main__":
    main()
