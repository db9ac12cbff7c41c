"""Builds libmeshanything_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels to the GPU box)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
# MA_B200_NO_FHFMA=1 selects the convert + FFMA variant of the canonical dot products (own file names, so both builds
# travel to the GPU box side by side); the default uses the mixed-precision FMA (SASS FHFMA), see canon.cuh
VARIANT = "_nofhfma" if os.environ.get("MA_B200_NO_FHFMA") == "1" else ""
LIB = os.path.join(LIB_DIR, f"libmeshanything_b200{VARIANT}.so")
SOURCES = ["gemm_canon.cu", "attention.cu", "attention_stream.cu", "elementwise.cu", "decode_fast.cu", "decode_mega.cu", "api.cu", "glue.cu", "gemm_tc.cu", "gemm_ws.cu", "attention_tc.cu", "api_encoder.cu", "surface.cu", "watertight.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
if VARIANT:
    NVCC_FLAGS.append("-DMA_NO_FHFMA")


def _nvcc() -> str:
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def have_nvcc() -> bool:
    return bool(shutil.which("nvcc")) or os.path.exists("/usr/local/cuda/bin/nvcc")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(HERE, "..", "include", f) for f in os.listdir(os.path.join(HERE, "..", "include"))]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = _nvcc()
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    objs = []

    def compile_one(src: str) -> str:
        obj = os.path.join(LIB_DIR, src.replace(".cu", f"{VARIANT}.o"))
        cmd = [nvcc, *NVCC_FLAGS, "-ccbin", "g++", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True, env=env)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-ccbin", "g++", "-o", LIB, *objs, "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
