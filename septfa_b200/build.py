"""In-tree build of libseptfa.so (nvcc, sm_100a only). ``python -m septfa_b200.build``."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libseptfa.so")
SOURCES = ["frontend.cu", "tcn.cu", "gemm_tc.cu", "gemm_conv1_persist.cu", "gemm_conv1_tma.cu", "gemm_conv1_pair.cu", "dconv_mma2.cu", "resid_fused.cu", "backend.cu", "preproc.cu", "online.cu", "live.cu", "resample.cu", "septfa_abi.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link libseptfa.so next to the package."""
    nvcc = _nvcc()
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")] + os.environ.get("SEPTFA_NVCC_FLAGS", "").split()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "septfa.h"))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
            if verbose:
                sys.stderr.write(r.stderr)
        return o

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
