"""Builds tests/emu/libk16_emu.so: the packed kernel's row sweep compiled as HOST code (nvcc)."""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
CSRC = ROOT / "genomicsbench_b200/csrc"
DEPS = [CSRC / "bsw_kernel16.cuh", CSRC / "bsw_kernels.cuh", CSRC / "bsw_warp16.cuh", CSRC / "bsw_global2.cuh",
        CSRC / "bsw_global_plan.h", CSRC / "bsw_global.cuh", CSRC / "bsw_long32.cuh"]


def build(force: bool = False, name: str = "k16") -> Path:
    """name = "k16" (thread-per-pair sweep), "w16" (warp-per-pair register sweep, the lanes as coroutines), "l32" (the
    int32 ring sweep of bsw_extend32, lanes as coroutines) or "g2" (bsw_global's second kernel with its chunk planner)."""
    so, src = HERE / f"lib{name}_emu.so", HERE / f"{name}_emu.cu"
    if not force and so.exists() and all(so.stat().st_mtime >= d.stat().st_mtime for d in DEPS + [src]):
        return so
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-shared",
           "-Xcompiler", "-fPIC,-fopenmp,-pthread", "-I", str(ROOT / "include"), "-o", str(so), str(src), "-lgomp", "-lpthread"]
    env = dict(os.environ)
    env["PATH"] = "/usr/bin:" + env.get("PATH", "")
    subprocess.run(cmd, check=True, env=env)
    return so


if __name__ == "__main__":
    print(build(force=True))
    print(build(force=True, name="w16"))
    print(build(force=True, name="g2"))
