#!/usr/bin/env python
"""Benchmark of the SPS inference hot path on B200 (contract: see the task's bench.py section).

Default (``--config 2``, the headline): a *step* = one collated batch (BASELINE.json configs[1]: OS1-64-like
65 536-point scans, batch 8, kd-tree-style radius-0.1 m submaps with duplicates, 0.1 m voxels, random-init weights)
through ``SPSModel.forward``: voxelise -> kernel maps -> 4-D MinkUNet -> devoxelise + sigmoid.

  value  scans/s, whole job, inputs resident in HBM when the timed region starts
  e2e    the same through the reference-facing call with HOST (pinned) buffers: H2D of the rows,
         forward, D2H of the scores, inside the timed region
  --impl reference   the CPU restatement of MinkowskiEngine's algorithm (oracle/me_cpu.c; the
         reference itself cannot run: ME is not vendored/installable, DESIGN.md) on all host cores

Other workloads of BASELINE.json (one JSON line each, same keys):
  --config 3   streamed ROS path: HDL-32 scans against a 1 M-voxel base map, crop + assemble + forward per scan
               as one CUDA graph (a step = one scan)
  --config 4   sequence-sharded inference: 10 000 scans split r::W over the ranks, NCCL gather of the scan scores
               AND of the per-scan metric partials, metrics aggregated as scripts/predict.py:70-83
  --config 5   stress shape (0.05 m voxels, 524 288-point scan + 30 m map crop): kernel-map + convolution sweep
               across layer widths with a per-layer roofline table
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SENSOR, BATCH, VOXEL, N_DISTINCT = "os1-64", 8, 0.1, 2
PTS_PER_SCAN = 65536
WORKLOAD = "config2: os1-64 (65536 pts/scan) x batch 8 + radius-0.1m submap (duplicates kept), 0.1 m voxels"
DTYPE = {0: "f16", 1: "f32", 2: "tf32", 3: "f16"}
ARITH = {0: "fp16 operands and stored activations, fp32 accumulate and epilogue (tcgen05); 8-output-channel layers with "
            "split hi+lo fp16 weights, level-0 tail (conv0 out, convtr7p2s2 out, block8) stored as fp16 hi|lo pairs",
         1: "fp32 CUDA cores", 2: "TF32 operands on fp32 rows (tcgen05), fp32 accumulate", 3: "as 0"}


def make_batches(rank: int, n_distinct=N_DISTINCT, batch=BATCH):
    """Seeded synthetic batches, rows [N,6] = (b,x,y,z,t,label); different scans per rank."""
    from sps_b200 import synth
    world = synth.World(0)
    map_xyz = synth.base_map(world, SENSOR, n_poses=12, seed=0, voxel=VOXEL)
    return [synth.make_batch(sensor=SENSOR, batch=batch, seed=100 * rank + i + 1, voxel=VOXEL, submap="radius",
                             world=world, map_xyz=map_xyz) for i in range(n_distinct)]


def random_state_dict():
    """Random-init weights with the reference's distributions (resnet.py:87-94 + ME defaults), made by the PRODUCT's
    own parameter module -- the GPU arm does not touch ``oracle/``."""
    import torch
    from sps_b200.models import CustomMinkUNet
    torch.manual_seed(0)
    return {k: v.detach().cpu().numpy() for k, v in CustomMinkUNet(1, 1, D=4).state_dict().items()}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed regions."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, enabled=True):
        self.index, self.lines, self.proc, self.enabled = index, [], None, enabled

    def start(self):
        if not self.enabled:      # only the rank that prints the line samples (eight pollers contend for the driver's locks)
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm": p["hbm_gbs"], "tensor": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "tensor_burst": p["bf16_tflops"], "src": "measured"}
    return {"hbm": 6650.0, "tensor": 1400.0, "tensor_burst": 1590.0, "src": "fallback"}


# layers of CustomMinkUNet in execution order: (stage name, kind, cin, cout, level of the OUTPUT rows)
PLANES = (8, 16, 32, 64, 64, 32, 16, 8)


def conv_layers(planes=PLANES, init_dim=8):
    P = planes
    out, c = [], init_dim
    for i in range(4):
        L = i + 1
        out.append((["conv1p1s2", "conv2p2s2", "conv3p4s2", "conv4p8s2"][i], "down", c, c, L, 0))
        out.append((f"block{L}.conv1", "k3", c, P[i], L, 0))
        out.append((f"block{L}.conv2", "k3", P[i], P[i], L, c if c != P[i] else 0))
        c = P[i]
    skip = (P[2], P[1], P[0], init_dim)
    for i in range(4):
        L = 3 - i
        co = P[4 + i]
        out.append((["convtr4p16s2", "convtr5p8s2", "convtr6p4s2", "convtr7p2s2"][i], "up", c, co, L, 0))
        cin = co + skip[i]
        out.append((f"block{5 + i}.conv1", "k3", cin, co, L, 0))
        out.append((f"block{5 + i}.conv2" + ("+final" if i == 3 else ""), "k3", co, co, L, cin))
        c = co
    return out


def stage_accounting(V, P3, P5, n_points, half_rows=True, planes=PLANES):
    """Algorithmic bytes / FLOPs per stage of ONE forward (SURVEY.md §8d formulas).

    Convolutions: FLOPs = 2 * pairs * Cin * Cout (+ the fused 1x1 term); minimum bytes = activations in + out +
    weights + 4 bytes of index per (in, out) PAIR (the kernels read present-only slices, not a dense K x V table).
    Activation element size: 2 bytes on fp16 rows, 4 on the fp32 rows of the level-0 tail / of the fp32 modes.
    Kernel maps: V * 20 (coordinates) + 8 * pairs (the pair-list form of §8d: what a present-only table holds)."""
    acc = {}
    cap = 1024
    while 2 * cap < 3 * n_points:      # csrc/common.cuh table_capacity: power of two >= 1.5 n
        cap *= 2
    acc["vox.clear"] = {"bytes": cap * 16}                       # the open-addressing table, 16-byte slots
    acc["vox.insert"] = {"bytes": n_points * 20 + n_points * 4}   # rows in, slot index out
    acc["vox.rank"] = {"bytes": n_points * 4 + n_points * 4}      # slot index in, block-local rank out
    acc["vox.assign"] = {"bytes": n_points * 4 + n_points * 4 + V[0] * 8}   # slot index in, inverse map + voxel keys out
    for L in range(5):
        acc[f"blocks.L{L}"] = {"bytes": V[L] * 8 + V[L] * 4}
        acc[f"kmap3.L{L}"] = {"bytes": V[L] * 20 + 8 * P3[L]}
    acc["kmap5.L0"] = {"bytes": V[0] * 20 + 8 * P5}
    for L in range(1, 5):
        acc[f"stride.L{L}"] = {"bytes": V[L - 1] * 20 + V[L] * 20 + V[L - 1] * 4}
    acc["devox_sigmoid"] = {"bytes": n_points * 4 + V[0] * 4 + n_points * 4}
    acc["conv0+kmap5"] = {"bytes": V[0] * 20 + 4 * V[0] + 8 * 4 * V[0], "flops": 2 * P5 * 8}
    for L in range(4):   # shape sort (key + row index in, row index out) and per-tile slices (present entries x 4 B, read + write)
        acc[f"sort.L{L}"] = {"bytes": V[L] * 12 + V[L] * 4}
        acc[f"slices.L{L}"] = {"bytes": 2 * 4 * P3[L] + V[L] * 16}
    acc["up_order"] = {"bytes": sum(V[L] * 8 for L in range(4))}       # parent word in, row index out (class order of the transposed convs)
    acc["blocks"] = {"bytes": sum(V[L] * 12 for L in range(5))}
    acc["kmap3"] = {"bytes": sum(V[L] * 20 + 8 * P3[L] for L in range(5))}
    acc["sort"] = {"bytes": sum(V[L] * 16 for L in range(4))}
    acc["slices"] = {"bytes": sum(2 * 4 * P3[L] + V[L] * 16 for L in range(4))}
    eb = 2 if half_rows else 4

    def esize(name):   # level-0 tail tensors: fp16 hi|lo pairs (4 bytes per value) in the fp16 forward, fp32 otherwise
        return 4 if name in ("conv1p1s2:in", "convtr7p2s2:out", "block8.conv1:in", "block8.conv1:out",
                             "block8.conv2+final:in", "block8.conv2+final:in2") else eb
    for name, kind, cin, cout, L, cin2 in conv_layers(planes):
        if kind == "down":
            vin, vout, K, pairs = V[L - 1], V[L], 8, V[L - 1]
        elif kind == "up":
            vin, vout, K, pairs = V[L + 1], V[L], 8, V[L]
        else:
            vin, vout, K, pairs = V[L], V[L], 81, P3[L]
        out_ch = 0 if name.endswith("+final") else cout
        b = vin * cin * esize(name + ":in") + vout * out_ch * esize(name + ":out") + K * cin * cout * eb + 4 * pairs
        f = 2 * pairs * cin * cout
        if cin2:
            b += vout * cin2 * esize(name + ":in2") + cin2 * cout * eb
            f += 2 * vout * cin2 * cout
        if name.endswith("+final"):
            b += vout * 4
            f += 2 * vout * cout
        acc[name] = {"bytes": b, "flops": f, "tensor_core": True}
    return acc


def measure_sizes(engine, points):
    """Voxel and pair counts of one batch (explicit, un-fused map build so that every table can be counted)."""
    from sps_b200.engine import _stream
    lib, h = engine.lib, engine.handle
    engine.voxelize(points, VOXEL)
    engine.build_maps()

    def pairs(level, kind):
        out = C.c_int64()
        lib.sps_ctx_pair_count(h, level, kind, C.byref(out), _stream())
        return out.value
    V = [engine.count(L) for L in range(5)]
    return V, [pairs(L, 3) for L in range(5)], pairs(0, 5)


# shared-memory fill rate of the LDGSTS path on one B200 (tools/gather4_probe.cu 64 0: rows resident in L1, so neither L2 nor
# DRAM limits it): 8.77 TB/s with two 256-thread producer groups per SM, 4.95 TB/s with one
LDGSTS_FILL_PEAK_GBS = 8770.0


def tile_walk(engine, V):
    """Present kernel offsets of every 128-row tile of the 3x3x3x3 maps, per level, in the order the convolution walks them
    (sps_ctx_level.tile_mask: the shape-sorted order where the level was sorted).  Call after measure_sizes."""
    out = []
    for L in range(5):
        v = engine.level(L)
        nt = (V[L] + 127) // 128
        if not v.tile_mask or nt == 0:
            out.append(np.zeros(0, np.int64))
            continue
        m = engine._read(v.tile_mask, nt * 4, np.uint32).reshape(nt, 4)[:, :3]
        out.append(np.array([bin(int(a)).count("1") + bin(int(b)).count("1") + bin(int(c)).count("1") for a, b, c in m], np.int64))
    return out


def staging_accounting(nact, planes=PLANES):
    """Shared-memory staging work of the 81-offset layers of the fp16 forward -- the resource the kernel is actually
    bound by.  Every stage is a 128-row x 128-byte A slab (16 KB: 32 warp-wide 16-byte cp.async instructions) plus an N-row
    weight slab; the stage count per tile mirrors csrc/conv_umma.cu (offsets per stage by channel count, two-segment walk of
    block5.conv1, hi|lo rows of the level-0 tail, fused 1x1 term).  LDGSTS retires one warp instruction per 8 cycles and SM
    (B300_MICROARCH.md, `LDGSTS rt`): 64 bytes per cycle and SM is the roof."""
    def gp(groups):
        return 1 if groups <= 1 else 2 if groups <= 2 else 4 if groups <= 4 else (groups + 7) // 8 * 8
    out = {}
    for name, kind, cin, cout, L, cin2 in conv_layers(planes):
        if kind != "k3" or len(nact[L]) == 0:
            continue
        na = nact[L]
        split_in = L == 0                       # level-0 tail: hi|lo rows, doubled channels
        g = (cin * (2 if split_in and name.startswith("block8.conv1") else 1)) // 8
        g2 = (cin2 * (2 if split_in else 1)) // 8
        packed2 = gp(g) < 8 and 0 < g2 <= 8     # the 1x1 term rides as extra offset slots of the last stage
        n2 = -(-g2 // gp(g)) if packed2 else 0
        if name == "block5.conv1" and cin == 96:
            st = na + (na + 1) // 2              # 64 channels per offset, then 32-channel halves two offsets per stage
        elif gp(g) < 8:
            eps = 8 // gp(g)
            st = (na + n2 + eps - 1) // eps
        else:
            st = na * (gp(g) // 8)
        if cin2 and not packed2:
            st = st + (g2 + 7) // 8
        stages = int(st.sum())
        weights_tma = gp(g) >= 8
        winstr = 0 if weights_tma else max(cout if cout > 8 else 16, 16) // 4      # N rows x 8 chunks / 32 lanes
        out[name] = {"stages": stages, "staged_bytes": stages * 128 * 128, "ldgsts_warp_instr": stages * (32 + winstr)}
    return out


def profile_pass(engine, net, d_batches, steps, voxel=VOXEL):
    """Per-stage CUDA-event durations (events recorded by the library on its launch stream)."""
    import torch
    engine.profile(True)
    sums, n = {}, 0
    for k in range(steps):
        engine.forward(net, d_batches[k % len(d_batches)], voxel)
        torch.cuda.synchronize()
        for nm, ms in engine.profile_read().items():
            sums[nm] = sums.get(nm, 0.0) + ms
        n += 1
    engine.profile(False)
    return {k: v / n for k, v in sums.items()}


def roofline_from(stage_ms, acc, peaks):
    """Per-stage achieved rates, and the roofline object of the DOMINANT KERNEL FAMILY: the tcgen05 implicit-GEMM
    convolution kernel (all its launches of one forward together), against both of its roofs."""
    rows = {}
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath))
    for name, t in stage_ms.items():
        a = acc.get(name)
        if not a or t <= 0:
            continue
        gbs = a["bytes"] / (t * 1e-3) / 1e9
        row = {"ms": round(t, 4), "GB/s": round(gbs, 1), "hbm_frac": round(gbs / peaks["hbm"], 4)}
        if "flops" in a:
            tf = a["flops"] / (t * 1e-3) / 1e12
            row.update({"TFLOP/s": round(tf, 3), "tensor_frac": round(tf / peaks["tensor"], 5)})
        if isinstance(traffic.get(name), (int, float)):
            row["traffic_over_algorithmic"] = round(traffic[name] / a["bytes"], 2)
        rows[name] = row
    fam = [n for n in rows if acc[n].get("tensor_core")]
    other = [n for n in rows if n not in fam]
    t_fam = sum(rows[n]["ms"] for n in fam)
    if not fam or t_fam <= 0:
        return None, rows
    fam_bytes = sum(acc[n]["bytes"] for n in fam)
    fam_flops = sum(acc[n]["flops"] for n in fam)
    n_launch = len(fam)
    gbs = fam_bytes / (t_fam * 1e-3) / 1e9
    tf = fam_flops / (t_fam * 1e-3) / 1e12
    hbm_frac, tensor_frac = gbs / peaks["hbm"], tf / peaks["tensor"]
    fam_traffic = [traffic[n] for n in fam if isinstance(traffic.get(n), (int, float))]
    roof = {"kernel": "k_conv_umma (tcgen05 implicit-GEMM sparse convolution)", "launches_per_step": n_launch,
            "kernel_ms_per_launch": round(t_fam / n_launch, 5), "family_ms_per_step": round(t_fam, 4),
            "share_of_step": round(t_fam / sum(r["ms"] for r in rows.values()), 3),
            "bound": "hbm" if hbm_frac >= tensor_frac else "tensor",
            "achieved": round(gbs, 1) if hbm_frac >= tensor_frac else round(tf, 2),
            "peak": peaks["hbm"] if hbm_frac >= tensor_frac else peaks["tensor"],
            "unit": "GB/s" if hbm_frac >= tensor_frac else "TFLOP/s",
            "frac": round(max(hbm_frac, tensor_frac), 4),
            "hbm": {"achieved_GBs": round(gbs, 1), "peak_GBs": peaks["hbm"], "frac": round(hbm_frac, 4),
                    "algorithmic_bytes_per_launch": int(fam_bytes / n_launch)},
            "tensor": {"achieved_TFLOPs": round(tf, 2), "peak_TFLOPs": peaks["tensor"], "frac": round(tensor_frac, 4),
                       "peak_kind": "bf16 dense, sustained (MEASURED_PEAKS.json)",
                       "algorithmic_flops_per_launch": int(fam_flops / n_launch)},
            "traffic": int(sum(fam_traffic) / len(fam_traffic)) if len(fam_traffic) == n_launch else None,
            "peak_source": peaks["src"],
            "other_stages_ms": round(sum(rows[n]["ms"] for n in other), 4)}
    return roof, rows


def cpu_baseline(rows, sd, steps=3, warmup=1):
    """oracle/me_cpu.c on ONE scan of the batch (bounded sample), all host threads."""
    from oracle import me_cpu
    nthreads = host_threads()
    blob = me_cpu.pack_weights(sd)
    one = np.ascontiguousarray(rows[rows[:, 0] == 0][:, :5])
    for _ in range(warmup):
        me_cpu.forward(one, VOXEL, blob, nthreads)
    t0 = time.perf_counter()
    for _ in range(steps):
        me_cpu.forward(one, VOXEL, blob, nthreads)
    dt = (time.perf_counter() - t0) / steps
    return {"value": 1.0 / dt, "unit": "scans/s", "cores": nthreads, "kind": "port",
            "sample": f"1 scan of the batch ({len(one)} rows: {PTS_PER_SCAN} scan pts + submap), {steps} timed forwards, "
                      f"{dt * 1e3:.0f} ms each; C/OpenMP restatement of ME's CPU algorithm (ME itself not installable)",
            "host_cpus": os.cpu_count()}


def run_reference(args):
    """The reference arm: ME's CPU algorithm (oracle/me_cpu.c) on all host threads.  The thread count is set
    explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import me_cpu
    nthreads = host_threads()
    if args.config == 3:
        from sps_b200 import synth
        world = synth.World(0)
        traj = synth.loop_trajectory(radius=35.0, n=400)
        base = synth.base_map(world, "hdl-32", n_poses=48, seed=0, voxel=VOXEL, trajectory=traj)
        scan = synth.scan(world, "hdl-32", traj(7), seed=1)
        one = np.ascontiguousarray(synth.assemble(scan, synth.submap_voxel_overlap(base, scan, VOXEL))[:, :5])
        workload = WORKLOAD3
    else:
        rows = make_batches(0, n_distinct=1, batch=1)[0]
        one = np.ascontiguousarray(rows[:, :5])
        workload = WORKLOAD if args.config == 2 else WORKLOAD4
    blob = me_cpu.pack_weights(random_state_dict())
    for _ in range(args.warmup):
        me_cpu.forward(one, VOXEL, blob, nthreads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        me_cpu.forward(one, VOXEL, blob, nthreads)
    dt = time.perf_counter() - t0
    value = args.steps / dt
    sample = (f"each step = 1 scan of the workload ({len(one)} rows incl. submap), {nthreads} host threads "
              f"(omp_set_num_threads, {os.cpu_count()} CPUs on the box); C/OpenMP restatement of MinkowskiEngine's CPU "
              "algorithm (the reference itself is not installable offline)")
    print(json.dumps({
        "impl": "reference", "metric": "scans/s", "value": value, "unit": "scans/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "scans/s", "cores": nthreads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


WORKLOAD3 = ("config3: hdl-32 scans (57600 pts) streamed against a 1M-voxel base map: prune crop + assemble + forward "
             "per scan as one CUDA graph, 0.1 m voxels")
WORKLOAD4 = ("config4: 10000 os1-64 scans (batches of 8) sharded r::W over the ranks, replicated weights, NCCL gather of "
             "the scan scores and of the per-scan metric partials")


def bind_to_gpu_numa(local_rank):
    """Multi-rank runs: pin this process to the CPUs NVML names as local to its GPU, so that the pinned staging buffers of
    the end-to-end path are allocated on the GPU's NUMA node and the H2D copies of eight ranks do not all cross one socket
    (round 1: e2e scaling 5.9x at 8 GPUs against 7.6x device-resident).  Best effort: returns the CPU count bound to, or
    None when NVML or the affinity call is not available (e.g. a container with a restricted CPU set)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        ideal = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = ideal & allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
        return len(cpus) if cpus else None
    except Exception:
        return None


class Dist:
    """torch.distributed plumbing of one rank (NCCL over NVLink); no-ops at world size 1."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
        torch.cuda.set_device(self.local)
        self.numa = None
        if self.world > 1:
            self.numa = bind_to_gpu_numa(self.local)    # before any pinned allocation: first touch decides the node
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.comm = torch.cuda.Stream()   # collectives run here: the compute lanes never wait for them

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ms(self, ms):
        t = self.torch.tensor([ms], device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, finish=None):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            fn(k)
        if finish:
            finish()
        torch.cuda.current_stream().wait_stream(self.comm)
        e1.record()
        torch.cuda.synchronize()
        self.barrier()
        return self.max_ms(e0.elapsed_time(e1))

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


class ScoreGather:
    """The only collective of the path (north star): all ranks' SCAN-row scores -- fp32 [batch x points per scan] per step,
    not the padded scores of every input row -- gathered with one all_gather_into_tensor on the comm stream, behind the
    lane's completion.  `every` steps share one collective (SURVEY 8e: "at the end, or every B scans"): a collective per
    step couples the ranks step by step -- every rank's NCCL kernel spins on SMs until the slowest rank arrives, which cost
    0.1 ms per 2.5 ms step at 2..8 GPUs.  Optionally the per-scan metric partials travel with it (config 4)."""

    def __init__(self, d: Dist, scan_rows, n_scan_total, with_partials=False, every=1):
        torch = d.torch
        self.d = d
        self.scan_rows = scan_rows                     # per distinct batch: int32 device positions of the t == 1 rows
        self.n, self.every, self.keys = n_scan_total, max(1, every), []
        self.buf = torch.empty(self.every * n_scan_total, dtype=torch.float32, device="cuda")
        self.all = torch.empty(d.world * self.every * n_scan_total, dtype=torch.float32, device="cuda") if d.world > 1 else None
        self.events = []
        self.with_partials = with_partials
        if with_partials:
            self.counts = torch.zeros((self.every, BATCH, 4), dtype=torch.int64, device="cuda")
            self.sums = torch.zeros((self.every, BATCH, 5), dtype=torch.float64, device="cuda")
            self.all_counts = torch.zeros((d.world, self.every, BATCH, 4), dtype=torch.int64, device="cuda")
            self.all_sums = torch.zeros((d.world, self.every, BATCH, 5), dtype=torch.float64, device="cuda")
        from sps_b200 import _cabi
        self.lib = _cabi.load()

    def publish(self, scores_dev, k, rows_dev=None, eps=0.84, sink=None):
        """Enqueue on the comm stream: compact the scan rows of ``scores_dev`` (the step's device scores) into this
        step's slot; the collective goes out when `every` slots are filled (or at flush())."""
        torch, d = self.d.torch, self.d
        if d.world == 1 and not self.with_partials:
            return
        idx = self.scan_rows[k % len(self.scan_rows)]
        slot = len(self.keys)
        with torch.cuda.stream(d.comm):
            st = C.c_void_p(d.comm.cuda_stream)
            self.lib.sps_gather_rows(C.c_void_p(scores_dev.data_ptr()), 1, 1, C.c_void_p(idx.data_ptr()), idx.numel(),
                                     C.c_void_p(self.buf.data_ptr() + 4 * slot * self.n), st)
            if self.with_partials:
                for b in range(BATCH):   # SPSNet.predict_step partials per scan (models.py:84-104)
                    self.lib.sps_confusion_counts(C.c_void_p(scores_dev.data_ptr()), C.c_void_p(rows_dev.data_ptr()),
                                                  rows_dev.stride(0), rows_dev.shape[0], float(b), float(eps),
                                                  C.c_void_p(self.counts[slot, b].data_ptr()),
                                                  C.c_void_p(self.sums[slot, b].data_ptr()), st)
        self.keys.append(k)
        if len(self.keys) >= self.every:
            self.flush(sink)

    def flush(self, sink=None):
        """The collective over the filled slots (always the whole buffer: unused slots carry stale bytes)."""
        torch, d = self.d.torch, self.d
        if not self.keys:
            return
        with torch.cuda.stream(d.comm):
            if d.world > 1:
                d.dist.all_gather_into_tensor(self.all, self.buf)
                if self.with_partials:
                    d.dist.all_gather_into_tensor(self.all_counts, self.counts)
                    d.dist.all_gather_into_tensor(self.all_sums, self.sums)
            elif self.with_partials:
                self.all_counts[0].copy_(self.counts)
                self.all_sums[0].copy_(self.sums)
            if sink is not None:
                sink(self, list(self.keys))
            ev = torch.cuda.Event()
            ev.record(d.comm)
        self.keys = []
        self.events.append(ev)
        if len(self.events) > 1:          # the slot buffer is rewritten by the next round: never overtake the collective
            self.events.pop(0).synchronize()


def setup_model(args, n_max, local, sd=None):
    import torch
    from sps_b200.models import SPSModel
    sd = sd or random_state_dict()
    model = SPSModel(VOXEL, max_points=n_max)
    model.MinkUNet.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
    model = model.cuda().eval()
    model.lanes = args.lanes
    model.use_graphs = model.use_graphs and not args.no_graphs
    model.set_conv_backend(args.backend)
    engine, net = model._prepare(n_max, torch.device("cuda", local))
    return model, engine, net, sd


def dump_outputs(out_dir, arrays):
    """Writes each array as ``out_dir/<name>.npy``: the inputs are seeded, so two builds can be compared array by array."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64) and a.nbytes <= 64 << 20, (name, a.dtype, a.nbytes)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_config2(args):
    import torch
    d = Dist()
    batches = make_batches(d.rank)
    host = [torch.as_tensor(np.ascontiguousarray(b[:, :5])).pin_memory() for b in batches]
    dev = [h.cuda() for h in host]
    scan_rows = [torch.as_tensor(np.nonzero(b[:, 4] == 1)[0].astype(np.int32)).cuda() for b in batches]
    n_max = max(len(h) for h in host)
    model, engine, net, sd = setup_model(args, n_max, d.local)
    gather = ScoreGather(d, scan_rows, BATCH * PTS_PER_SCAN, every=args.gather_every)
    pending = []
    last = [None]      # handle of the most recent finished step

    def finish_one():
        kk, p = pending.pop(0)
        p.result()
        gather.publish(p.device_scores, kk)
        last[0] = p

    def step(inputs):
        def fn(k):
            # consecutive steps alternate between the model's lanes (engine context + stream each); every step's scores
            # are waited for inside the timed region, then the scan rows go to every rank on the comm stream
            pending.append((k, model.forward_async(inputs[k % len(inputs)])))
            if len(pending) >= model.lanes:
                finish_one()
        return fn

    def drain():
        while pending:
            finish_one()
        gather.flush()

    def measure(inputs, steps):
        fn = step(inputs)
        # warm-up: every (lane, batch) pair is seen twice before it replays as a CUDA graph (eager, then capture)
        nwarm = max(args.warmup, 3, (3 * model.lanes * len(inputs)) if model.use_graphs else 0)
        for k in range(nwarm):
            fn(k)
        drain()
        return d.timed(fn, steps, finish=drain)

    sampler = ClockSampler(d.local, enabled=d.rank == 0)
    sampler.start()
    ms_dev = measure(dev, args.steps)       # inputs resident in HBM
    # the last timed step's scores, copied before the next window reuses the lane's buffer
    outputs = {"scores": last[0].device_scores.cpu().numpy()} if args.dump_outputs and d.rank == 0 else None
    ms_host = measure(host, args.steps)     # public host-side API: pinned H2D of step k+1 overlaps the kernels of step k
    clocks = sampler.stop()
    engine.status()
    launches = engine.launch_count() * args.steps
    alt = None
    if d.world == 1 and args.backend in (0, 3) and not args.no_alt:
        # the same step with TF32 operands on fp32 rows (backend 2), printed beside the headline
        model.set_conv_backend(2)
        ms_alt = measure(dev, min(args.steps, 10))
        alt = {"backend": 2, "dtype": "tf32", "ms_per_step": ms_alt / min(args.steps, 10), "arithmetic": ARITH[2]}
        model.set_conv_backend(args.backend)

    scans = d.world * BATCH * args.steps
    value, e2e = scans / (ms_dev * 1e-3), scans / (ms_host * 1e-3)
    result = {
        "metric": "scans/s", "value": value, "unit": "scans/s", "n_gpus": d.world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[args.backend], "data": "synthetic",
        "config": {"workload": WORKLOAD, "arithmetic": ARITH[args.backend],
                   "rows_per_step": int(np.mean([len(h) for h in host])),
                   "scans_per_step_per_gpu": BATCH, "weights": "random-init (seed 0), BN eval fresh stats",
                   "l2": f"per-step working set (kernel maps + features, several GB) exceeds the 126 MB L2; "
                         f"{len(host)} distinct batches rotate",
                   "conv_backend": args.backend, "lanes": args.lanes, "cuda_graphs": bool(model.use_graphs), "tma_weight_stages": bool(engine.lib.sps_tma_weights_available()),
                   "sharding": f"scan-sharded, replicated weights; every {args.gather_every} steps one NCCL all_gather_into_tensor of the "
                               f"scan-row scores (fp32 [{BATCH} x {PTS_PER_SCAN}] per rank and step) on a dedicated stream",
                   "cpus_bound_to_gpu_numa": d.numa},
        "mpoints_per_s": value * PTS_PER_SCAN / 1e6,
        "e2e": {"value": e2e, "unit": "scans/s", "ms_per_step": ms_host / args.steps,
                "h2d_bytes_per_step": int(np.mean([h.numel() * 4 for h in host])),
                "d2h_bytes_per_step": int(np.mean([len(h) * 4 for h in host]))},
        "gpu_launches": launches, "clocks": clocks,
    }
    if alt:
        result["alt"] = alt
    if d.rank == 0:
        peaks = load_peaks()
        nprof = min(args.steps, 5)
        stage_ms = profile_pass(engine, net, dev, nprof)
        V, P3, P5 = measure_sizes(engine, dev[(nprof - 1) % len(dev)])
        acc = stage_accounting(V, P3, P5, len(dev[(nprof - 1) % len(dev)]), half_rows=args.backend in (0, 3))
        roof, rows = roofline_from(stage_ms, acc, peaks)
        if args.backend in (0, 3) and roof:
            # the resource the kernel is bound by: 16-byte cp.async copies into the shared-memory stages
            nact = tile_walk(engine, V)
            stg = staging_accounting(nact)
            sm_hz = (clocks.get("sm_mhz") or 1920) * 1e6
            t_lsu = 0.0
            for nm, a in stg.items():
                if nm in rows:
                    bound_ms = a["ldgsts_warp_instr"] * 8 / 148 / sm_hz * 1e3
                    rows[nm].update({"stages": a["stages"], "staged_GB/s": round(a["staged_bytes"] / (rows[nm]["ms"] * 1e-3) / 1e9, 1),
                                     "ldgsts_bound_ms": round(bound_ms, 4), "ldgsts_frac": round(bound_ms / rows[nm]["ms"], 3)})
                    t_lsu += bound_ms
            t_k3 = sum(rows[nm]["ms"] for nm in stg if nm in rows)
            staged = sum(a["staged_bytes"] for nm, a in stg.items() if nm in rows)
            roof["staging"] = {"what": "81-offset layers: bytes written into the shared-memory A stages by 16-byte cp.async (LDGSTS) copies, "
                                       "absent and padded slots included -- the resource that bounds the gather",
                               "layers": len(stg), "layers_ms": round(t_k3, 4),
                               "staged_GBs": round(staged / (t_k3 * 1e-3) / 1e9, 1) if t_k3 else None,
                               "peak_GBs": LDGSTS_FILL_PEAK_GBS,
                               "frac": round(staged / (t_k3 * 1e-3) / 1e9 / LDGSTS_FILL_PEAK_GBS, 3) if t_k3 else None,
                               "peak_source": "measured: tools/gather4_probe.cu (256 producer threads, L1-resident rows, 2 CTAs per SM), "
                                              "profiles/r2_gather_probe.md",
                               "issue_bound_ms": round(t_lsu, 4),
                               "tile_fill": {f"L{L}": round(P3[L] / max(int(nact[L].sum()) * 128, 1), 3) for L in range(4)}}
        result["roofline"] = roof
        result["stages"] = rows
        result["stage_sum_ms"] = round(sum(stage_ms.values()), 4)
        result["sizes"] = {"voxels_per_level": V, "pairs3": P3, "pairs5": P5,
                           "flops_per_step": int(sum(a.get("flops", 0) for a in acc.values()))}
        if d.world == 1 and not args.no_cpu_baseline:
            result["cpu_baseline"] = cpu_baseline(batches[0], sd)
        if outputs:
            dump_outputs(args.dump_outputs, outputs)
    d.close()
    if d.rank == 0:
        print(json.dumps(result))


def run_config3(args):
    """Streamed ROS path (c_ws/src/sps_filter/scripts/sps_node.py:111-120), one scan per step."""
    import torch
    from sps_b200 import synth, engine as E
    d = Dist()
    steps = args.steps if args.steps_given else 1000
    world = synth.World(0)
    traj = synth.loop_trajectory(radius=35.0, n=400)
    base = synth.base_map(world, "hdl-32", n_poses=400, seed=0, voxel=VOXEL, trajectory=traj, target_voxels=1_000_000)
    pool = [synth.scan(world, "hdl-32", traj(7 * i + 3 * d.rank), seed=i + 100 * d.rank) for i in range(32)]
    n = len(pool[0])
    host = [torch.as_tensor(s).pin_memory() for s in pool]
    dev = [h.cuda() for h in host]
    mh = E.MapHash(torch.as_tensor(base).cuda(), VOXEL)
    sd = random_state_dict()
    net = E.Net(sd)
    eng = E.Engine(2 * n)
    eng.set_conv_backend(args.backend)
    streamer = E.ScanStreamer(mh, eng, net, n, VOXEL)
    h_out = [torch.empty(n, dtype=torch.float32).pin_memory() for _ in range(2)]

    def step_dev(k):
        streamer.infer(dev[k % 32])

    def step_host(k):     # host xyz in (pinned), scores back to pinned host memory, every scan
        streamer.infer(host[k % 32])
        h_out[k & 1].copy_(streamer.scores, non_blocking=True)

    for k in range(max(args.warmup, 3)):
        step_dev(k)
    sampler = ClockSampler(d.local, enabled=d.rank == 0)
    sampler.start()
    ms_dev = d.timed(step_dev, steps)
    for k in range(3):
        step_host(k)
    ms_host = d.timed(step_host, steps)
    clocks = sampler.stop()
    eng.status()
    scans = d.world * steps
    value, e2e = scans / (ms_dev * 1e-3), scans / (ms_host * 1e-3)
    result = {
        "metric": "scans/s", "value": value, "unit": "scans/s", "n_gpus": d.world, "steps": steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": DTYPE[args.backend], "data": "synthetic",
        "config": {"workload": WORKLOAD3, "map_voxels": int(len(base)), "points_per_scan": n, "arithmetic": ARITH[args.backend],
                   "scans": "32 distinct scans along a loop trajectory, cycled",
                   "l2": "per-scan working set (~200 MB of maps + features) exceeds the 126 MB L2 together with the 1M-voxel map hash",
                   "conv_backend": args.backend},
        "mpoints_per_s": value * n / 1e6,
        "e2e": {"value": e2e, "unit": "scans/s", "ms_per_step": ms_host / steps, "h2d_bytes_per_step": n * 12,
                "d2h_bytes_per_step": n * 4},
        "gpu_launches": (eng.launch_count() + 7) * steps, "clocks": clocks,
    }
    if d.rank == 0:
        peaks = load_peaks()
        counts = torch.zeros(2, dtype=torch.int32, device="cuda")
        eng.profile(True)
        mh.infer_scan(eng, net, dev[5], VOXEL, counts=counts)
        torch.cuda.synchronize()
        stage_ms = eng.profile_read()
        eng.profile(False)
        sub = mh.crop_voxel(dev[5])[0]
        rows5 = torch.as_tensor(synth.assemble(pool[5], sub.cpu().numpy())[:, :5]).cuda()
        V, P3, P5 = measure_sizes(eng, rows5)
        acc = stage_accounting(V, P3, P5, len(rows5), half_rows=args.backend in (0, 3))
        roof, rows = roofline_from(stage_ms, acc, peaks)
        result["roofline"] = roof
        result["stages"] = rows
        result["sizes"] = {"voxels_per_level": V, "pairs3": P3, "submap_voxels": int(len(sub))}
        if d.world == 1 and not args.no_cpu_baseline:
            from oracle import me_cpu
            one = np.ascontiguousarray(rows5.cpu().numpy())
            blob = me_cpu.pack_weights(sd)
            nt = host_threads()
            me_cpu.forward(one, VOXEL, blob, nt)
            t0 = time.perf_counter()
            for _ in range(5):
                me_cpu.forward(one, VOXEL, blob, nt)
            dt = (time.perf_counter() - t0) / 5
            result["cpu_baseline"] = {"value": 1.0 / dt, "unit": "scans/s", "cores": nt, "kind": "port",
                                      "sample": f"1 scan + its submap ({len(one)} rows), forward only (no crop), 5 timed runs, {dt * 1e3:.0f} ms each"}
    d.close()
    if d.rank == 0:
        print(json.dumps(result))


def run_config4(args):
    """10 000 scans split r::W (scripts/predict.py:70-83 over the whole sequence): every step a rank runs one batch of
    8 of ITS scans, computes the per-scan metric partials on the device and all-gathers scores + partials."""
    import torch
    from sps_b200.parallel import metrics_from_partials
    d = Dist()
    n_scans = 10000
    steps = args.steps if args.steps_given else n_scans // (BATCH * d.world)
    batches = make_batches(d.rank)
    rows_dev = [torch.as_tensor(np.ascontiguousarray(b)).cuda() for b in batches]       # [N,6] with labels
    dev = [r[:, :5].contiguous() for r in rows_dev]
    scan_rows = [torch.as_tensor(np.nonzero(b[:, 4] == 1)[0].astype(np.int32)).cuda() for b in batches]
    n_max = max(len(x) for x in dev)
    model, engine, net, sd = setup_model(args, n_max, d.local)
    gather = ScoreGather(d, scan_rows, BATCH * PTS_PER_SCAN, with_partials=True, every=args.gather_every)
    tot_counts = torch.zeros((steps, d.world, BATCH, 4), dtype=torch.int64, device="cuda")
    tot_sums = torch.zeros((steps, d.world, BATCH, 5), dtype=torch.float64, device="cuda")
    pending = []

    def sink(g, keys):      # the gathered partials of the steps of one collective -> their rows of the totals
        for slot, kk in enumerate(keys):
            if kk < steps:
                tot_counts[kk].copy_(g.all_counts[:, slot])
                tot_sums[kk].copy_(g.all_sums[:, slot])

    def finish_one():
        kk, p = pending.pop(0)
        p.result()

        gather.publish(p.device_scores, kk, rows_dev=rows_dev[kk % len(rows_dev)], sink=sink)

    def fn(k):
        pending.append((k, model.forward_async(dev[k % len(dev)])))
        if len(pending) >= model.lanes:
            finish_one()

    def drain():
        while pending:
            finish_one()
        gather.flush(sink)

    for k in range(max(args.warmup, 3, (3 * model.lanes * len(dev)) if model.use_graphs else 0)):
        fn(k)
    drain()
    sampler = ClockSampler(d.local, enabled=d.rank == 0)
    sampler.start()
    ms = d.timed(fn, steps, finish=drain)
    clocks = sampler.stop()
    engine.status()
    scans = d.world * BATCH * steps
    value = scans / (ms * 1e-3)
    result = {
        "metric": "scans/s", "value": value, "unit": "scans/s", "n_gpus": d.world, "steps": steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": DTYPE[args.backend], "data": "synthetic",
        "config": {"workload": WORKLOAD4, "scans_total": scans, "arithmetic": ARITH[args.backend],
                   "scans": f"{len(dev)} distinct batches of 8 per rank, cycled (generating 10 000 distinct scans on the host "
                            "would take longer than the run)",
                   "collective": f"per step: all_gather_into_tensor of fp32 [{BATCH} x {PTS_PER_SCAN}] scan scores, int64 "
                                 f"[{BATCH} x 4] confusion counts and fp64 [{BATCH} x 5] sums per rank, comm stream",
                   "conv_backend": args.backend, "lanes": args.lanes},
        "mpoints_per_s": value * PTS_PER_SCAN / 1e6,
        "e2e": {"value": value, "unit": "scans/s", "ms_per_step": ms / steps, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": "device-resident inputs; the host-side end-to-end number of this workload is config 2's e2e"},
        "gpu_launches": (engine.launch_count() + 1 + BATCH) * steps, "clocks": clocks,
    }
    if d.rank == 0:
        c = tot_counts.reshape(-1, 4).cpu()
        s = tot_sums.reshape(-1, 5).cpu()
        result["metrics"] = metrics_from_partials(c, s)      # mean of per-scan values (predict.py:70-83)
        result["metrics"]["scans_with_partials"] = int((s[:, 0] > 0).sum())
    d.close()
    if d.rank == 0:
        print(json.dumps(result))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--backend", type=int, default=0,
                    help="0 auto (tcgen05 on fp16 rows + fp32 FMA on the 8-channel layers), 1 fp32 CUDA-core, "
                         "2 tcgen05 TF32 on fp32 rows, 3 = 0")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the backend-2 (TF32) comparison line")
    ap.add_argument("--no-graphs", action="store_true", help="enqueue every forward kernel by kernel instead of replaying CUDA graphs")
    ap.add_argument("--gather-every", type=int, default=4,
                    help="multi-GPU: steps whose scan-row scores (and metric partials) share one NCCL all-gather")
    ap.add_argument("--lanes", type=int, default=3, help="engine contexts/streams forward_async alternates between")
    ap.add_argument("--widths", default="1,2,4,8", help="config 5: PLANES multipliers of the sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="config 2: write the fp32 scores of the last device-resident timed step to DIR/scores.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config != 2):
        ap.error("--dump-outputs is implemented for --config 2 of --impl ours")
    args.steps_given = args.steps is not None
    if args.steps is None:
        args.steps = 20
    if args.impl == "reference":
        return run_reference(args)
    if args.config == 3:
        return run_config3(args)
    if args.config == 4:
        return run_config4(args)
    if args.config == 5:
        from tools import width_sweep
        return width_sweep.run(args)
    return run_config2(args)


if __name__ == "__main__":
    main()
