"""Builds tepose_b200/libtepose_b200.so (the C-ABI library of include/tepose_b200.h) with nvcc for
sm_100a.  In-tree, so the built library travels with the repo snapshot to the GPU box."""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libtepose_b200.so")
OBJ = os.path.join(HERE, "build")
SOURCES = ["api.cu", "geometry.cu", "pack.cu", "gemm_f32.cu", "gemm_tc.cu", "skinny.cu", "gru.cu", "regressor.cu", "smpl.cu", "metrics.cu", "train.cu", "loss.cu", "conv.cu", "crop.cu", "slots.cu", "render.cu", "smooth.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _stale(target: str, deps) -> bool:
    if not os.path.isfile(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, variant: str = "") -> str:
    """variant="fence": the same sources with -DTP_BARRIER_ACQUIRE_FENCE (every grid barrier executes the formal acquire fence after
    its relaxed polls) -> libtepose_b200_fence.so; tests/test_gpu_e2e.py checks that its outputs are bit-identical to the default
    build's (the default relies on every post-barrier read of other CTAs' data being an L2-coherent access)."""
    nvcc = _nvcc()
    flags = list(NVCC_FLAGS)
    obj_dir, lib_path = OBJ, LIB
    if variant == "fence":
        flags.append("-DTP_BARRIER_ACQUIRE_FENCE")
        obj_dir, lib_path = os.path.join(HERE, "build_fence"), os.path.join(HERE, "libtepose_b200_fence.so")
    elif variant:
        raise ValueError(f"unknown build variant {variant!r}")
    os.makedirs(obj_dir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".inl"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "tepose_b200.h"))

    def compile_one(src):
        s = os.path.join(CSRC, src)
        o = os.path.join(obj_dir, src[:-3] + ".o")
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + flags + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
        return o

    with concurrent.futures.ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(lib_path, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_path] + objs
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib_path


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True, variant="fence" if "--fence" in sys.argv else ""))
