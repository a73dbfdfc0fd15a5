#!/usr/bin/env python
"""Offline evaluation from scans alone against today's host-prepared rows, on bench.py's config-2 workload.

  A  forward_async on pinned host rows [N, 5] prepared with scipy (bench.py --config 2 "e2e"; the submap selection is
     not in the timed step)
  B  predict_radius_async on pinned host scans [sum n_b, 4] (x, y, z, label): radius submaps, collation, forward and
     per-scan metric partials on the GPU

Same world, base map and seeds as bench.py::make_batches (8 x 65 536 os1-64 scans per step, 0.1 m radius and voxels);
under ``torchrun --nproc-per-node N`` every rank takes its own scans and the partials are gathered at the end
(parallel.gather_partials).  The two paths alternate in one process, window by window.  Prints one JSON line with the
card's name and power limit.  Needs a GPU; writes nothing.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

EPS = 0.84          # bench.py's metric threshold


def gpu_card(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception:
        return {"name": None, "power_limit": None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3, help="alternating A/B windows per path")
    ap.add_argument("--lanes", type=int, default=3)
    args = ap.parse_args()

    import torch
    import bench
    from sps_b200 import parallel, synth
    from sps_b200.datasets import RadiusSubmap

    d = bench.Dist()
    batches = bench.make_batches(d.rank)
    world = synth.World(0)
    map_xyz = synth.base_map(world, bench.SENSOR, n_poses=12, seed=0, voxel=bench.VOXEL).astype(np.float32)
    rows_host = [torch.as_tensor(np.ascontiguousarray(b[:, :5])).pin_memory() for b in batches]
    scans_host, offsets = [], []
    for b in batches:
        scan = b[b[:, 4] == 1]
        scans_host.append(torch.as_tensor(np.ascontiguousarray(scan[:, [1, 2, 3, 5]])).pin_memory())
        sizes = np.bincount(scan[:, 0].astype(np.int64), minlength=bench.BATCH)
        offsets.append(np.concatenate([[0], np.cumsum(sizes)]).tolist())
    n_max = max(len(h) for h in rows_host)
    model, engine, net, _ = bench.setup_model(argparse.Namespace(lanes=args.lanes, no_graphs=False, backend=0), n_max, d.local)
    sub = RadiusSubmap(torch.as_tensor(map_xyz).cuda(), bench.VOXEL)

    def run_a(k):
        return model.forward_async(rows_host[k % len(rows_host)])

    def run_b(k):
        j = k % len(scans_host)
        return model.predict_radius_async(scans_host[j], sub, EPS, offsets=offsets[j])

    last = {}      # (path, batch) -> results of a warm-up step (copies: a lane's buffers are reused `lanes` calls later)

    def window(fn, steps, key):
        pending, keep = [], [True]

        def finish_one():
            kk, p = pending.pop(0)
            out = p.result()
            if keep[0]:
                last[key, kk % len(batches)] = tuple(t.clone() for t in out) if isinstance(out, tuple) else out.clone()

        def step(k):
            pending.append((k, fn(k)))
            if len(pending) >= model.lanes:
                finish_one()

        def drain():
            while pending:
                finish_one()
        for k in range(max(args.warmup, model.lanes * len(batches))):
            step(k)
        drain()
        keep[0] = False
        return d.timed(step, steps, finish=drain)

    ms = {"A": [], "B": []}
    for _ in range(args.rounds):
        ms["A"].append(window(run_a, args.steps, "A"))
        ms["B"].append(window(run_b, args.steps, "B"))

    # the batching kernels alone (sps_radius_batch on device-resident scans), CUDA events
    lib = engine.lib
    dev_scans = [s.cuda() for s in scans_host]
    nb = lib.sps_radius_batch_scratch_bytes(max(len(s) for s in dev_scans), bench.BATCH)
    scratch = torch.empty(nb, dtype=torch.uint8, device="cuda")
    rows_dev = torch.empty((engine.max_points, 6), dtype=torch.float32, device="cuda")
    roff = torch.empty(bench.BATCH + 1, dtype=torch.int32, device="cuda")
    n_rows = torch.empty(1, dtype=torch.int32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def batch_kernels(j):
        h_off = (C.c_int64 * (bench.BATCH + 1))(*offsets[j])
        rc = lib.sps_radius_batch(sub.handle, C.c_void_p(dev_scans[j].data_ptr()), 4, h_off, bench.BATCH,
                                  C.c_void_p(rows_dev.data_ptr()), rows_dev.shape[0], C.c_void_p(roff.data_ptr()),
                                  C.c_void_p(n_rows.data_ptr()), C.c_void_p(scratch.data_ptr()), nb, st)
        assert rc == 0, rc
    for j in range(4):
        batch_kernels(j % len(dev_scans))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record()
    for j in range(reps):
        batch_kernels(j % len(dev_scans))
    e1.record()
    torch.cuda.synchronize()
    batching_ms = e0.elapsed_time(e1) / reps

    # B's scan scores == SPSModel.forward on make_batch rows, bit for bit; its rows == the scipy-prepared multiset
    exact = True
    for j in range(len(batches)):
        rows = sub.make_batch(dev_scans[j], offsets[j])
        ref = model(rows[:, :5])
        model.check()
        exact &= bool(torch.equal(last["B", j][0].cuda(), ref[rows[:, 4] == 1]))
        exact &= len(rows) == len(batches[j])

    # partials of every distinct batch on this rank -> all ranks (scan ids r::world), predict.py's metrics
    counts = torch.cat([last["B", j][1] for j in range(len(batches))]).cuda()
    sums = torch.cat([last["B", j][2] for j in range(len(batches))]).cuda()
    all_counts, all_sums = parallel.gather_partials(counts, sums, d.world * len(counts))
    metrics = parallel.metrics_from_partials(all_counts, all_sums)

    scans_per_window = d.world * bench.BATCH * args.steps
    n_scan = int(np.mean([len(s) for s in scans_host]))
    n_rows_mean = int(np.mean([len(h) for h in rows_host]))

    def path(key, h2d, d2h, batching):
        best = min(ms[key])
        return {"scans_per_s": scans_per_window / (best * 1e-3), "ms_per_step": best / args.steps,
                "ms_per_step_windows": [round(m / args.steps, 4) for m in ms[key]],
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "batching": batching}
    result = {
        "metric": "scans/s", "n_gpus": d.world, "steps_per_window": args.steps, "rounds": args.rounds,
        "lanes": args.lanes, "gpu": gpu_card(d.local), "workload": bench.WORKLOAD,
        "A_forward_async_host_rows": path("A", n_rows_mean * 5 * 4, n_rows_mean * 4,
                                          "scipy on the host, before the timed steps"),
        "B_predict_radius_async_host_scans": path("B", n_scan * 4 * 4,
                                                  n_scan * 4 + bench.BATCH * (4 * 8 + 5 * 8) + 4,
                                                  {"kernel_ms_per_step": round(batching_ms, 4),
                                                   "what": "sps_radius_batch (count + scan, write), CUDA events, "
                                                           "device-resident scans"}),
        "scores_bit_identical_to_forward_on_make_batch_rows": exact,
        "metrics": metrics, "scans_in_metrics": int((all_sums[:, 0] > 0).sum()),
    }
    d.close()
    if d.rank == 0:
        print(json.dumps(result))


if __name__ == "__main__":
    main()
