#!/usr/bin/env python
"""Replay of sensor-frame deployment scans through the ROS node's whole callback, one at a time against batched, on
bench.py's config-3 workload.

  node      per scan on the device: util.transform_point_cloud -> ScanStreamer.infer -> util.filter_scan
  batch B   SPSModel.filter_scans_async on B scans at once (B = 4, 8, 16): pose transform, voxel-prune submaps,
            collation, one forward, the node's metric partials and the published rows in one library call, pipelined
            over the model's lanes

Same world, base map (1 M voxels) and 32 hdl-32 scans as tools/prune_batch_bench.py, moved into the sensor frame by the
inverse of their trajectory poses (sensor 1.8 m above the ground), with a seeded intensity column; 0.1 m crop lattice
and voxels; eps is the median score of the first scan under the benchmark's random weights, so that about half the
points are published (with those weights every score lies below the node's 0.84).  Each path runs on device-resident
scans and on pinned host scans (host: the node path copies each scan in and its published rows back; the batched path
returns every result, the whole published-row buffer included, to pinned host memory).  The paths alternate in one process, window by window; the best of the windows is
reported.  Also reported: the largest per-scan score difference between the two paths in the same run (the batched
forward shape-sorts its rows from 400 000 rows on, the per-scan one never, so the last bits may differ), whether the
published row counts of every scan agree (a score within that difference of eps can flip), the published fraction, and
the card's name, power limit and maximum SM clock, read with nvidia-smi
in the same call.  Prints one JSON line.  Needs a GPU; writes nothing.
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

SENSOR_HEIGHT = 1.8      # synth.scan's default


def pose_matrix(pose):
    """synth.loop_trajectory's (x, y, yaw) at the sensor height -> the 4x4 float64 sensor -> map matrix."""
    x, y, a = pose
    T = np.eye(4)
    T[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    T[:3, 3] = (x, y, SENSOR_HEIGHT)
    return T


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=256, help="scans per timed window (a multiple of 16)")
    ap.add_argument("--rounds", type=int, default=3, help="alternating windows per path")
    ap.add_argument("--lanes", type=int, default=3)
    ap.add_argument("--batches", default="4,8,16")
    args = ap.parse_args()

    import torch
    import bench
    from prune_batch_bench import gpu_card
    from sps_b200 import engine as E, synth, util

    d = bench.Dist()
    world = synth.World(0)
    traj = synth.loop_trajectory(radius=35.0, n=400)
    base = synth.base_map(world, "hdl-32", n_poses=400, seed=0, voxel=bench.VOXEL, trajectory=traj,
                          target_voxels=1_000_000)
    poses = np.stack([pose_matrix(traj(7 * i)) for i in range(32)])
    rng = np.random.default_rng(0)
    pool = []
    for i in range(32):
        xyz = synth.scan(world, "hdl-32", traj(7 * i), seed=i).astype(np.float64)
        h = np.hstack([xyz, np.ones((len(xyz), 1))]) @ np.linalg.inv(poses[i]).T
        pool.append(np.hstack([h[:, :3] / h[:, 3:], rng.random((len(xyz), 1))]).astype(np.float32))
    n = len(pool[0])
    host = [torch.as_tensor(s).pin_memory() for s in pool]
    dev = [h.cuda() for h in host]
    dev_poses = torch.as_tensor(poses).cuda()
    mh = E.MapHash(torch.as_tensor(base).cuda(), bench.VOXEL)
    sd = bench.random_state_dict()
    batches = [int(b) for b in args.batches.split(",")]
    model, _, net, _ = bench.setup_model(argparse.Namespace(lanes=args.lanes, no_graphs=False, backend=0),
                                         2 * n * max(batches), d.local, sd)
    eng = E.Engine(2 * n)
    streamer = E.ScanStreamer(mh, eng, net, n, bench.VOXEL)
    d_in = [torch.empty((n, 4), dtype=torch.float32, device="cuda") for _ in range(2)]
    h_kept = [torch.empty((n, 4), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_count = [torch.empty(1, dtype=torch.int32).pin_memory() for _ in range(2)]
    # concatenated scans + offsets per batch start (a batch = scans k*B .. k*B+B-1 of the pool, cycled); device poses
    # for device scans, host poses for host scans
    cat = {}
    for B in batches:
        for src, name in ((dev, "dev"), (host, "host")):
            for k in range(32 // B):
                t = torch.cat(src[k * B:(k + 1) * B])
                p = dev_poses[k * B:(k + 1) * B] if name == "dev" else torch.as_tensor(poses[k * B:(k + 1) * B])
                cat[name, B, k] = (t.pin_memory() if name == "host" else t, [i * n for i in range(B + 1)], p)

    # eps: the median score of scan 0 on the node path
    eps = float(streamer.infer(util.transform_point_cloud(dev[0], poses[0])).median())
    node_scores, node_kept = {}, {}

    def node_window(on_device):
        def step(k):
            j = k % 32
            scan = dev[j]
            if not on_device:
                d_in[k & 1].copy_(host[j], non_blocking=True)
                scan = d_in[k & 1]
            scores = streamer.infer(util.transform_point_cloud(scan, poses[j]))
            kept, count = util.filter_scan(scan, scores, eps)
            if not on_device:
                h_kept[k & 1].copy_(kept, non_blocking=True)
                h_count[k & 1].copy_(count, non_blocking=True)
            return scores, count
        for k in range(32):                 # warm-up, and the per-scan results of the comparison
            scores, count = step(k)
            if on_device:
                node_scores[k] = scores.clone()
                node_kept[k] = int(count.item())
        return d.timed(step, args.scans)

    batch_out = {}

    def batch_window(B, on_device):
        name = "dev" if on_device else "host"
        pending, keep = [], [True]

        def finish_one():
            k, p = pending.pop(0)
            out = p.result()
            if keep[0] and on_device:
                batch_out[B, k % (32 // B)] = (out.scan_scores.clone(), out.kept_offsets.cpu().numpy())

        def step(k):
            t, offs, p = cat[name, B, k % (32 // B)]
            pending.append((k, model.filter_scans_async(t, p, mh, eps, offsets=offs)))
            if len(pending) >= model.lanes:
                finish_one()

        def drain():
            while pending:
                finish_one()
        for k in range(max(model.lanes, 32 // B)):
            step(k)
        drain()
        keep[0] = False
        return d.timed(step, args.scans // B, finish=drain)

    paths = [("node", None, True), ("node", None, False)] + [("batch", B, od) for B in batches for od in (True, False)]
    ms = {p: [] for p in paths}
    for _ in range(args.rounds):
        for p in paths:
            ms[p].append(node_window(p[2]) if p[0] == "node" else batch_window(p[1], p[2]))
    eng.status()
    model.check()
    card = gpu_card(d.local)

    # per-scan agreement of the two paths in this run
    max_diff, kept_agree = 0.0, True
    for B in batches:
        for k in range(32 // B):
            scores, koff = batch_out[B, k]
            for j in range(B):
                max_diff = max(max_diff, float((scores[j * n:(j + 1) * n] - node_scores[k * B + j]).abs().max()))
                kept_agree &= int(koff[j + 1] - koff[j]) == node_kept[k * B + j]

    def report(p):
        calls = args.scans if p[0] == "node" else args.scans // p[1]
        best = min(ms[p])
        return {"scans_per_s": args.scans / (best * 1e-3), "ms_per_call": round(best / calls, 4),
                "ms_per_call_windows": [round(m / calls, 4) for m in ms[p]]}
    result = {
        "metric": "scans/s", "gpu": card, "points_per_scan": n, "map_voxels": int(len(base)), "scans_per_window": args.scans,
        "rounds": args.rounds, "lanes": args.lanes, "eps": eps,
        "workload": "config3 in the sensor frame: 32 hdl-32 scans along a loop trajectory with their poses against a "
                    "1M-voxel base map, 0.1 m crop and voxels",
        "node_device": report(("node", None, True)), "node_pinned_host": report(("node", None, False)),
        "batched": {str(B): {"device": report(("batch", B, True)), "pinned_host": report(("batch", B, False))}
                    for B in batches},
        "kept_fraction": sum(node_kept.values()) / (32 * n),
        "max_abs_score_diff_batched_vs_node": max_diff, "kept_counts_agree": bool(kept_agree),
    }
    d.close()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
