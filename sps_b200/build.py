"""In-tree build of the C-ABI CUDA library (nvcc, sm_100a only; no torch headers involved)."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsps_b200.so")
STAMP = os.path.join(HERE, ".libsps_b200.stamp")
SOURCES = ["api.cu", "maps.cu", "ballquery.cu", "rosio.cu", "shard.cu", "conv_simt.cu", "conv_umma.cu", "net.cu"]
HEADERS = ["common.cuh", "ctx.h", "scan.cuh", "partials.cuh", "rosio.cuh", "umma_common.cuh", "profile.h",
           os.path.join("..", "..", "include", "sps_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v"]


def _digest() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        path = os.path.join(CSRC, f)
        if os.path.exists(path):
            with open(path, "rb") as fh:
                h.update(fh.read())
    h.update((" ".join(NVCC_FLAGS) + os.environ.get("SPS_NVCC_EXTRA", "")).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libsps_b200.so next to this file unless it is already up to date."""
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read() == digest:
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    srcs = [os.path.join(CSRC, f) for f in SOURCES if os.path.exists(os.path.join(CSRC, f))]
    extra = os.environ.get("SPS_NVCC_EXTRA", "").split()
    cmd = [nvcc] + NVCC_FLAGS + extra + ["-o", LIB] + srcs
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libsps_b200.so")
    with open(os.path.join(HERE, "ptxas_info.txt"), "w") as fh:
        fh.write(res.stderr)
    with open(STAMP, "w") as fh:
        fh.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
