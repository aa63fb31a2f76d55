"""Build libclengine.so (hand-written sm_100a kernels + C-ABI) in-tree with nvcc.

    python -m crowdllama_b200.build            # incremental
    python -m crowdllama_b200.build --force

Output: crowdllama_b200/lib/libclengine.so (git-ignored, travels to the GPU box with gpurun).
nvcc cross-compiles for sm_100a without a GPU.  cudart is linked statically so the library
carries no dependency on torch's bundled runtime.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

HERE = Path(__file__).resolve().parent
CSRC = HERE / "csrc"
OBJ = HERE / "lib" / "obj"
LIB = HERE / "lib" / "libclengine.so"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
HOSTCXX = "/usr/bin/g++"

SOURCES = ["decode_kernels.cu", "decode_mega.cu", "decode_mega_batch.cu", "attn_decode_tc.cu", "batch_kernels.cu", "engine.cu", "ops_api.cu", "prefill.cu", "gemm_tcgen05.cu", "prefill_kernels.cu", "attn_prefill_tc.cu", "sample_kernels.cu",
           "host_util.cpp", "tokenizer.cpp", "weights_io.cpp", "scheduler.cpp", "capi.cpp"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-ccbin", HOSTCXX,
         "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function,-fvisibility=default", "--expt-relaxed-constexpr",
         "-I", str(HERE.parent / "include")]


def _newest_header() -> float:
    hs = list(CSRC.glob("*.h")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.inc")) + [HERE.parent / "include" / "clengine.h"]
    return max(h.stat().st_mtime for h in hs)


def _compile(src: Path, force: bool) -> Path:
    obj = OBJ / (src.name + ".o")
    if not force and obj.exists() and obj.stat().st_mtime > max(src.stat().st_mtime, _newest_header()):
        return obj
    cmd = [NVCC, *FLAGS, "-x", "cu", "-c", str(src), "-o", str(obj)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        raise RuntimeError(f"nvcc failed for {src.name}:\n{r.stdout}\n{r.stderr}")
    return obj


def build(force: bool = False, verbose: bool = False) -> Path:
    OBJ.mkdir(parents=True, exist_ok=True)
    srcs = [CSRC / s for s in SOURCES if (CSRC / s).exists()]
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(lambda s: _compile(s, force), srcs))
    if force or not LIB.exists() or any(o.stat().st_mtime > LIB.stat().st_mtime for o in objs):
        cmd = [NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", HOSTCXX, "-cudart", "static",
               "-o", str(LIB), *map(str, objs), "-lpthread", "-ldl", "-lrt"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print(f"built {LIB} ({LIB.stat().st_size >> 10} KiB)")
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
