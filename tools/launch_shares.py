"""ncu launch list of a bench run vs the live CUDA-event stage times of the bench line: kernel shares of the step.
usage: launch_shares.py gpurun_out/r2_launches.csv profiles/r2_bench_n1.json > profiles/r2_launches_summary.md"""
import csv, json, sys, collections
rows = list(csv.reader(open(sys.argv[1])))
for i, r in enumerate(rows):
    if r and r[0] == "ID":
        hdr, start = r, i + 1
        break
ki, vi, ui = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
seq = []
for r in rows[start:]:
    if len(r) > vi:
        v = float(r[vi].replace(",", "")) * {"ns": 1e-3, "nsecond": 1e-3, "us": 1.0, "usecond": 1.0, "ms": 1e3}.get(r[ui], 1.0)
        seq.append((r[ki].replace("void ", "").split("(")[0], v))
bench = json.loads(open(sys.argv[2]).read().strip().splitlines()[-1])
st = {k: v["ms"] * 1e3 for k, v in bench["stages"].items()}
n = len(seq) // 2                                   # two forwards were captured
fwd = seq[n:]
groups = [("`k_conv_umma6<*>` (all instantiations)", lambda k: k.startswith("k_conv_umma6"),
           [k for k in st if k.startswith(("conv1", "conv2", "conv3", "conv4", "convtr", "block")) and k != "blocks"]),
          ("`k_kernel_map_blk3`", lambda k: k.startswith("k_kernel_map_blk3"), ["kmap3"]),
          ("shape sort (4 x `k_onesweep_pass`; the keys come out of the kernel-map pass)", lambda k: k.startswith("k_onesweep"), ["sort"]),
          ("`k_tile_masks_perm`", lambda k: k.startswith("k_tile_masks_perm"), ["slices"]),
          ("`k_conv0_const`", lambda k: k.startswith("k_conv0"), ["conv0+kmap5"]),
          ("strided levels (`k_level_begin`, `k_insert_coarse`, `k_first_rank`, `k_assign_coarse` x 4)", None,
           ["stride.L1", "stride.L2", "stride.L3", "stride.L4"]),
          ("voxelisation (`k_level_begin`, `k_insert_points`, `k_first_rank`, `k_assign_points`)", None,
           ["vox.clear", "vox.insert", "vox.rank", "vox.assign"]),
          ("block tables (`k_blocks_begin`, `k_block_insert`, `k_cells_fill`)", lambda k: k.startswith(("k_blocks_begin", "k_block_insert", "k_cells_fill")), ["blocks"]),
          ("`k_up_order`", lambda k: k.startswith("k_up_order"), ["up_order"]),
          ("`k_devox_sigmoid`", lambda k: k.startswith("k_devox"), ["devox_sigmoid"])]
tot_ncu = sum(v for _, v in fwd)
tot_b = sum(st.values())
# the first four launches are the voxelisation, the next sixteen the strided levels (launch order of the forward)
by_pos = {"voxelisation": fwd[:4], "strided": fwd[4:20]}
print(f"Launch list `profiles/r2_launches.csv` (`ncu --metrics gpu__time_duration.sum --clock-control none` over `python bench.py --steps 2 "
      f"--warmup 3 --lanes 1`, the two timed forwards): second forward ({n} launches), per kernel group.  ncu serialises launches and runs "
      f"them with cold caches, so absolute times are larger than inside the pipelined step; the SHARES are what must agree with the live "
      f"CUDA-event stage times of `profiles/r2_bench_n1.json` (stage sum {tot_b / 1e3:.2f} ms single lane).\n")
print("| kernel group | launches | ncu us | ncu share | bench stages us | bench share |")
print("|---|---:|---:|---:|---:|---:|")
for name, pred, stages in groups:
    if pred is None:
        sel = by_pos["voxelisation" if name.startswith("voxel") else "strided"]
    else:
        sel = [(k, v) for k, v in fwd[20:] if pred(k)] if not name.startswith("`k_conv_umma6") else [(k, v) for k, v in fwd if pred(k)]
    t = sum(v for _, v in sel)
    b = sum(st.get(s, 0.0) for s in stages)
    print(f"| {name} | {len(sel)} | {t:.1f} | {100 * t / tot_ncu:.1f}% | {b:.1f} | {100 * b / tot_b:.1f}% |")
print(f"| total | {len(fwd)} | {tot_ncu:.1f} | 100% | {tot_b:.1f} | 100% |")
