"""Build pearl_b200/libpearlb200.so in-tree with nvcc for sm_100a (no JIT cache:
the built .so travels to the GPU box with the repo snapshot)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = [os.path.join(HERE, "csrc", f) for f in ("replay_buffer.cu", "dqn.cu", "dqn_tc.cu", "ppo.cu", "per.cu", "sac.cu", "dsac.cu", "td3.cu", "gemm_tc.cu", "umma_test.cu")]
HDR = [os.path.join(HERE, "csrc", "common.cuh"), os.path.join(HERE, "csrc", "sampler.cuh"), os.path.join(HERE, "csrc", "umma.cuh"), os.path.join(HERE, "csrc", "dqn_common.cuh"), os.path.join(HERE, "csrc", "gemm.cuh"), os.path.join(os.path.dirname(HERE), "include", "pearl_b200.h")]
OUT = os.path.join(HERE, "libpearlb200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
]


def build(force: bool = False, verbose: bool = False) -> str:
    newest = max(os.path.getmtime(p) for p in SRC + HDR + [os.path.abspath(__file__)])
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= newest:
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-o", OUT] + SRC
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libpearlb200.so")
    with open(os.path.join(HERE, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force=True, verbose=True))
