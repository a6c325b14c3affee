"""In-tree build of the CUDA shared library (sm_100a only).

Every .cu is compiled to an object (in parallel) and linked into _lib/libdfd_b200.so; objects are cached under
_lib/obj/ keyed by the compile flags, so tuning sweeps (DFD_NVCC_DEFS="-DDFD_TILE_K=4 ...", DFD_LIB_TAG=k4)
only rebuild what the defines touch."""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
OBJ_DIR = os.environ.get("DFD_OBJ_DIR", os.path.join(OUT_DIR, "obj"))  # per checkout, so builds by different users never share it

SOURCES = ["dfd_api.cu", "dfd_exec.cu", "dfd_exchange.cu", "dfd_reduce.cu", "dfd_scatter_twopass_local.cu", "dfd_scatter_twopass_peer.cu",
           "dfd_scatter_onepass_local.cu", "dfd_scatter_onepass_peer.cu", "dfd_scatter_follow_local.cu", "dfd_scatter_follow_peer.cu"]
TUNABLE = {s for s in SOURCES if s.startswith("dfd_scatter_") or s == "dfd_api.cu"}  # sources that see the tile-geometry macros
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def out_path(tag: str = "") -> str:
    return os.path.join(OUT_DIR, f"libdfd_b200{('_' + tag) if tag else ''}.so")


OUT = out_path(os.environ.get("DFD_LIB_TAG", ""))


def object_path(src: str) -> str:
    """Where build() caches the object of a source compiled with the default flags (used by the CPU host-logic harness of the
    test-suite, which links the product's own dfd_exec object against a host stand-in of the CUDA runtime)."""
    key = hashlib.sha1(" ".join(NVCC_FLAGS).encode()).hexdigest()[:10]
    return os.path.join(OBJ_DIR, f"{os.path.splitext(src)[0]}.{key}.o")


def _newest_source() -> float:
    t = 0.0
    for d in (CSRC, os.path.join(ROOT, "include")):
        for f in os.listdir(d):
            t = max(t, os.path.getmtime(os.path.join(d, f)))
    return t


def build(force: bool = False, verbose: bool = False, defs: str | None = None, tag: str | None = None) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(OUT_DIR, exist_ok=True)
    tag = os.environ.get("DFD_LIB_TAG", "") if tag is None else tag
    out = out_path(tag)
    newest = _newest_source()
    if not force and os.path.exists(out) and os.path.getmtime(out) >= newest:
        return out
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = (os.environ.get("DFD_NVCC_DEFS", "") if defs is None else defs).split()  # e.g. "-DDFD_TILE_K=4" for tuning sweeps
    extra_onepass = os.environ.get("DFD_NVCC_DEFS_ONEPASS", "").split()  # e.g. "-DDFD_ONEPASS_NB=4": single-pass kernels only
    inc = ["-I", os.path.join(ROOT, "include"), "-I", CSRC]

    def compile_one(src: str) -> str:
        flags = NVCC_FLAGS + (extra if src in TUNABLE else []) + (extra_onepass if ("onepass" in src or "follow" in src or src == "dfd_api.cu") else []) + (["-Xptxas", "-v"] if verbose else [])
        key = hashlib.sha1(" ".join(flags).encode()).hexdigest()[:10]
        obj = os.path.join(OBJ_DIR, f"{os.path.splitext(src)[0]}.{key}.o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < newest:
            subprocess.check_call([nvcc] + flags + inc + ["-c", os.path.join(CSRC, src), "-o", obj])
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC"] + objs + ["-o", out, "-ldl"])
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
