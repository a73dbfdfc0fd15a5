"""Build an experimental variant of libsps_b200.so (extra nvcc flags) next to the product library:
    python tools/build_variant.py NAME -Xptxas -maxrregcount=64 ...   ->  sps_b200/variants/libsps_NAME.so
Select it at run time with SPS_B200_LIB=sps_b200/variants/libsps_NAME.so (A/B measurements only)."""
import os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sps_b200 import build as b
name, flags = sys.argv[1], sys.argv[2:]
out_dir = os.path.join(ROOT, "sps_b200", "variants")
os.makedirs(out_dir, exist_ok=True)
out = os.path.join(out_dir, f"libsps_{name}.so")
srcs = [os.path.join(b.CSRC, f) for f in b.SOURCES]
cmd = ["/usr/local/cuda/bin/nvcc"] + [f for f in b.NVCC_FLAGS if f not in ("-Xptxas", "-v")] + flags + ["-o", out] + srcs
res = subprocess.run(cmd, capture_output=True, text=True)
sys.stderr.write(res.stderr[-2000:])
print(out if res.returncode == 0 else "FAILED")
sys.exit(res.returncode)
