"""Builds libtwisterl_b200.so (hand-written sm_100a CUDA + the C ABI) in-tree with nvcc.

    python -m twisterl_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "lib" / "libtwisterl_b200.so"
SOURCES = ["twr_engine.cu", "twr_kernels.cu", "twr_forward_fp32.cu", "twr_forward_tc2.cu", "twr_forward_generic.cu", "twr_mcts.cu", "twr_comm.cu", "twr_safetensors.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: the twisterl_b200 CUDA library cannot be built")


def is_stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.cpp")) + [PKG.parent / "include" / "twisterl_b200.h"]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not is_stale():
        return LIB
    nvcc = _nvcc()
    obj_dir = PKG / "lib" / "obj"
    obj_dir.mkdir(parents=True, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = obj_dir / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out)
        objs.append(str(obj))
    cmd = [nvcc, "-shared", "-o", str(LIB), *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-lcuda", "-ldl", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}{r.stderr}")
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
