"""Builds libdvd_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m dvd_b200.build [--force] [--verbose]

Objects are cached under dvd_b200/csrc/build/ keyed by a hash of the source, its headers and the
flags, so incremental rebuilds only recompile what changed.  The .so is git-ignored but travels to
the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libdvd_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr", "-Xptxas", "-v"]
EXTRA = os.environ.get("DVD_NVCC_EXTRA", "").split()        # e.g. -DDVD_GEMM_TRACE for tools/gemm_trace.py (instrumented build)
if EXTRA:                                                   # instrumented builds never replace the product library
    FLAGS += EXTRA
    BUILD = os.path.join(CSRC, "build_trace")
    LIB = os.path.join(HERE, "libdvd_b200_trace.so")
SOURCES = ["api.cu", "unwarp.cu", "gemm_simt.cu", "misc.cu", "gemm_tc.cu", "gemm_pair.cu", "attn_tc.cu", "attn_pair.cu", "denoiser.cu", "prep.cu"]


def _headers():
    hs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(os.path.dirname(HERE), "include", "dvd_b200.h"))
    return hs


def _digest(src):
    h = hashlib.sha256()
    for p in [src] + _headers():
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()[:16]


def _compile(name, force, verbose):
    src = os.path.join(CSRC, name)
    obj = os.path.join(BUILD, name.replace(".cu", ".o"))
    stamp = obj + ".hash"
    dig = _digest(src)
    if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == dig:
        return obj, ""
    cmd = [NVCC] + FLAGS + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {name}:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(dig)
    with open(obj + ".ptxas.log", "w") as f:
        f.write(r.stderr)
    return obj, r.stderr if verbose else ""


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(BUILD, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        res = list(ex.map(lambda s: _compile(s, force, verbose), srcs))
    objs = [o for o, _ in res]
    for _, log in res:
        if log:
            print(log)
    newest = max(os.path.getmtime(o) for o in objs)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < newest:
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
