#!/usr/bin/env python3
"""Build libtcs.so (sm_100a only) in-tree with nvcc.  No torch headers are involved: the library
is a plain C-ABI shared object that the Python shim loads with ctypes.

    python vae-diffusion-toy-crystals_b200/build.py [--force]
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "toycrystals_b200")
LIB = os.path.join(OUT_DIR, "libtcs.so")
OBJ_DIR = os.path.join(HERE, "build")
SOURCES = ["tcs_api.cu", "conv_tc.cu", "kernels_simt.cu", "kernels_split.cu", "kernels_embed.cu", "kernels_step.cu",
           "prior_api.cu", "linear_tc.cu", "kernels_prior.cu", "attn_tc.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def source_hash() -> str:
    """SHA-256 over every source and header that goes into libtcs.so (and this recipe); compiled into the library
    (tcs_build_info() ends in TCS_SRC_HASH=<hex>) so that a stale prebuilt .so is detected, whatever its mtime."""
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    files += [os.path.join(HERE, "..", "include", "tcs.h"), os.path.join(HERE, "..", "include", "tcs_prior.h"),
              os.path.abspath(__file__)]
    h = hashlib.sha256()
    for f in files:
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def lib_hash(path: str = LIB):
    """The TCS_SRC_HASH compiled into an existing libtcs.so (read from the file, no dlopen), or None."""
    if not os.path.exists(path):
        return None
    blob = open(path, "rb").read()
    k = blob.find(b"TCS_SRC_HASH=")
    return blob[k + 13:k + 29].decode(errors="replace") if k >= 0 else None


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(d) <= t for d in deps)


def build_lib(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "tcs.h"))
    headers.append(os.path.join(HERE, "..", "include", "tcs_prior.h"))
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    want = source_hash()
    if not force and lib_hash() == want:
        return LIB

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
        is_api = os.path.basename(src) == "tcs_api.cu"       # carries the hash: rebuilt whenever anything changed
        if not force and not is_api and _newer(obj, [src] + headers):
            return obj, ""
        extra = [f'-DTCS_SRC_HASH="{want}"'] if is_api else []
        r = subprocess.run([NVCC, *FLAGS, *extra, "-c", src, "-o", obj], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        res = list(ex.map(compile_one, srcs))
    with open(os.path.join(OBJ_DIR, "ptxas.log"), "a") as f:
        for _, log in res:
            f.write(log)
            if verbose:
                sys.stderr.write(log)
    objs = [o for o, _ in res]
    r = subprocess.run([NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    if lib_hash() != want:
        raise RuntimeError("libtcs.so does not carry the source hash it was just built with")
    return LIB


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
