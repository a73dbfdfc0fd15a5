#!/usr/bin/env python
"""Replay of deployment scans, one at a time against batched, on bench.py's config-3 workload.

  stream    ScanStreamer.infer per scan (bench.py --config 3): prune + assemble + forward as one CUDA graph per scan
  batch B   SPSModel.infer_scans_async on B scans at once (B = 4, 8, 16): voxel-prune submaps, collation and one forward
            per batch in one library call, pipelined over the model's lanes

Each path runs on device-resident scans and on pinned host scans (host: the scores come back to pinned host memory).
Same world, base map (1 M voxels) and 32 hdl-32 scans as bench.py::run_config3, 0.1 m crop lattice and voxels.  The
paths alternate in one process, window by window; the best window of each is reported.  Also reported: the largest
per-scan score difference between the two paths in the same run (the batched forward shape-sorts its rows from
400 000 rows on, the per-scan one never, so the last bits of fp16 activations may differ) and the card's name, power
limit and maximum SM clock, read with nvidia-smi in the same call.  Prints one JSON line.  Needs a GPU; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_card(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception:
        return {"name": None, "power_limit": None, "clocks_max_sm": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=256, help="scans per timed window (a multiple of 16)")
    ap.add_argument("--rounds", type=int, default=3, help="alternating windows per path")
    ap.add_argument("--lanes", type=int, default=3)
    ap.add_argument("--batches", default="4,8,16")
    args = ap.parse_args()

    import torch
    import bench
    from sps_b200 import engine as E, synth

    d = bench.Dist()
    world = synth.World(0)
    traj = synth.loop_trajectory(radius=35.0, n=400)
    base = synth.base_map(world, "hdl-32", n_poses=400, seed=0, voxel=bench.VOXEL, trajectory=traj,
                          target_voxels=1_000_000)
    pool = [synth.scan(world, "hdl-32", traj(7 * i), seed=i) for i in range(32)]
    n = len(pool[0])
    host = [torch.as_tensor(s).pin_memory() for s in pool]
    dev = [h.cuda() for h in host]
    mh = E.MapHash(torch.as_tensor(base).cuda(), bench.VOXEL)
    sd = bench.random_state_dict()
    batches = [int(b) for b in args.batches.split(",")]
    model, _, net, _ = bench.setup_model(argparse.Namespace(lanes=args.lanes, no_graphs=False, backend=0),
                                         2 * n * max(batches), d.local, sd)
    eng = E.Engine(2 * n)
    streamer = E.ScanStreamer(mh, eng, net, n, bench.VOXEL)
    h_out = [torch.empty(n, dtype=torch.float32).pin_memory() for _ in range(2)]
    # concatenated scans + offsets per batch start (a batch = scans k*B .. k*B+B-1 of the pool, cycled)
    cat = {}
    for B in batches:
        for src, name in ((dev, "dev"), (host, "host")):
            for k in range(32 // B):
                t = torch.cat(src[k * B:(k + 1) * B])
                cat[name, B, k] = (t.pin_memory() if name == "host" else t, [i * n for i in range(B + 1)])

    stream_scores = {}

    def stream_window(on_device):
        src = dev if on_device else host

        def step(k):
            streamer.infer(src[k % 32])
            if not on_device:
                h_out[k & 1].copy_(streamer.scores, non_blocking=True)
        for k in range(32):                 # warm-up, and the per-scan scores of the comparison
            step(k)
            if on_device:
                stream_scores[k] = streamer.scores.clone()
        return d.timed(step, args.scans)

    batch_scores = {}

    def batch_window(B, on_device):
        name = "dev" if on_device else "host"
        pending, keep = [], [True]

        def finish_one():
            k, p = pending.pop(0)
            out = p.result()
            if keep[0] and on_device:
                batch_scores[B, k % (32 // B)] = out[0].clone()

        def step(k):
            t, offs = cat[name, B, k % (32 // B)]
            pending.append((k, model.infer_scans_async(t, mh, offsets=offs)))
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

    paths = [("stream", None, True), ("stream", None, False)] + [("batch", B, od) for B in batches for od in (True, False)]
    ms = {p: [] for p in paths}
    for _ in range(args.rounds):
        for p in paths:
            ms[p].append(stream_window(p[2]) if p[0] == "stream" else batch_window(p[1], p[2]))
    eng.status()
    model.check()
    card = gpu_card(d.local)

    # per-scan agreement of the two paths in this run
    max_diff = 0.0
    for B in batches:
        for k in range(32 // B):
            got = batch_scores[B, k]
            for j in range(B):
                max_diff = max(max_diff, float((got[j * n:(j + 1) * n] - stream_scores[k * B + j]).abs().max()))

    def report(p):
        best = min(ms[p])
        per_call = best / (args.scans if p[0] == "stream" else args.scans // p[1])
        return {"scans_per_s": args.scans / (best * 1e-3), "ms_per_call": round(per_call, 4),
                "ms_per_call_windows": [round(m / (args.scans if p[0] == "stream" else args.scans // p[1]), 4)
                                        for m in ms[p]]}
    result = {
        "metric": "scans/s", "gpu": card, "points_per_scan": n, "map_voxels": int(len(base)), "scans_per_window": args.scans,
        "rounds": args.rounds, "lanes": args.lanes,
        "workload": "config3: 32 hdl-32 scans along a loop trajectory against a 1M-voxel base map, 0.1 m crop and voxels",
        "stream_device": report(("stream", None, True)), "stream_pinned_host": report(("stream", None, False)),
        "batched": {str(B): {"device": report(("batch", B, True)), "pinned_host": report(("batch", B, False))}
                    for B in batches},
        "max_abs_score_diff_batched_vs_stream": max_diff, "scores_agree_2e-3": max_diff <= 2e-3,
    }
    d.close()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
