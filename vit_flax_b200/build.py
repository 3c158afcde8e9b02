"""Build ``libvitb200.so`` in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m vit_flax_b200.build [--force] [--verbose]

The shared object lands next to this file so it travels with the repo snapshot
to the GPU box; it is git-ignored.  cudart is linked statically and the driver
API is reached through ``cudaGetDriverEntryPoint``, so the library loads (and
its symbols can be checked) on a machine with no GPU and no libcuda.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OUT = PKG / "libvitb200.so"
OBJ_DIR = PKG / "build"
SOURCES = ["runtime.cu", "gemm_tc.cu", "attention.cu", "attention_tc5.cu", "attention_tc5m.cu", "simt.cu", "patch_tc.cu", "backward.cu", "attention_bwd_tc5.cu", "attention_probs_tc5.cu", "optim.cu", "api.cu"]
HEADERS = [CSRC / "common.h", CSRC / "ptx.cuh", PKG.parent / "include" / "vitb200.h"]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
] + (["-DVITB200_TRACE"] if os.environ.get("VITB200_TRACE") else [])   # debug timelines (profiles/trace_attention.py)


def _digest() -> str:
    h = hashlib.sha256()
    for p in [CSRC / s for s in SOURCES] + HEADERS + [Path(__file__)]:
        h.update(p.read_bytes())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def _compile(src: str, verbose: bool) -> str:
    obj = OBJ_DIR / (src.replace(".cu", ".o"))
    cmd = [NVCC, *FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
    if verbose:
        sys.stderr.write(r.stderr)
    (OBJ_DIR / (src + ".ptxas.log")).write_text(r.stderr)
    return str(obj)


def build(force: bool = False, verbose: bool = False) -> Path:
    OBJ_DIR.mkdir(exist_ok=True)
    stamp = OBJ_DIR / "digest.txt"
    digest = _digest()
    if not force and OUT.exists() and stamp.exists() and stamp.read_text() == digest:
        return OUT
    with cf.ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    cmd = [NVCC, "-shared", "-o", str(OUT), *objs, "-gencode", "arch=compute_100a,code=sm_100a",
           "-Xlinker", "--no-undefined"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp.write_text(digest)
    return OUT


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(p)
