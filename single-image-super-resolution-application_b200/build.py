"""In-tree nvcc build of libhitsir_b200.so (sm_100a only).

    python single-image-super-resolution-application_b200/build.py [--force]

The shared object is written next to this file so that it travels with the repo snapshot
(`*.so` is git-ignored but not gpurun-ignored).  No JIT cache, no torch extension machinery:
the library is a plain C-ABI object (include/hitsir_b200.h) loaded with ctypes.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libhitsir_b200.so")
SOURCES = ["engine.cu", "umma_gemm.cu", "umma_gemm_tma.cu", "proj_fc1.cu", "conv3_c64.cu", "ffn_tail.cu", "scc_umma.cu", "scc_dense.cu", "glue.cu", "pack.cu",
           "ensemble.cu", "metrics.cu", "resize.cu"]
HEADERS = ["common.cuh", "gemm.cuh", "kernels.cuh", "ycbcr.cuh", os.path.join("..", "..", "include", "hitsir_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-DNDEBUG"]


def _digest() -> str:
    h = hashlib.sha256()
    for name in SOURCES + HEADERS:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode())
            h.update(f.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def _run(cmd):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("command failed: %s\n%s" % (" ".join(cmd), r.stdout))
    return r.stdout


def build(force: bool = False, verbose: bool = False, defines=(), lib: str = None) -> str:
    """Compile every CUDA source for sm_100a and link the shared library.  Returns its path.
    `defines` adds -D flags to a variant build written to `lib` (kernel experiments: several variants travel to the GPU box in one
    snapshot)."""
    variant = bool(defines or lib)
    tag = os.path.splitext(os.path.basename(lib))[0] if lib else "var"
    bdir = os.path.join(BUILD, tag) if variant else BUILD
    out_lib = lib or LIB
    os.makedirs(bdir, exist_ok=True)
    stamp = os.path.join(bdir, "stamp.txt")
    extra = ["-D" + d for d in defines]
    digest = _digest() + " " + " ".join(extra)
    if not force and os.path.exists(out_lib) and os.path.exists(stamp) and open(stamp).read().strip() == digest:
        return out_lib
    objs = [os.path.join(bdir, s.replace(".cu", ".o")) for s in SOURCES]

    def compile_one(pair):
        src, obj = pair
        out = _run([NVCC] + FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj])
        if verbose and out.strip():
            print(out)

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        list(ex.map(compile_one, zip(SOURCES, objs)))
    _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-o", out_lib] + objs)
    with open(stamp, "w") as f:
        f.write(digest)
    return out_lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
