"""In-tree nvcc build of libccvpe_b200.so (sm_100a only; the .so travels to the GPU box with the repo snapshot).

Every .cu is compiled to its own object (in parallel, cached by mtime under ccvpe_b200/build/) and the objects are linked
into one shared library; nothing here needs a GPU (nvcc cross-compiles)."""
from __future__ import annotations

import concurrent.futures
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ_DIR = os.path.join(PKG_DIR, "build")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
LIB_PATH = os.path.join(PKG_DIR, "libccvpe_b200.so")
SOURCES = ["runtime.cu", "descriptors.cu", "match.cu", "pointwise.cu", "hypotheses.cu", "igemm_simt.cu", "igemm_tcgen05.cu",
           "conv_ring_tcgen05.cu", "match_tcgen05.cu", "project_tcgen05.cu", "stem_tcgen05.cu", "encoder_ops.cu", "ingest.cu", "resize.cu", "affine.cu", "track.cu", "train_ops.cu", "wgrad_tcgen05.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libccvpe_b200.so cannot be built")


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
           [os.path.join(INCLUDE, "ccvpe_b200.h")]


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in _sources()] + _headers()
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_one(nvcc: str, src: str, obj: str, verbose: bool):
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas=-v"] if verbose else []) + ["-c", "-o", obj, src]
    res = subprocess.run(cmd, capture_output=True, text=True)
    return src, res.returncode, res.stdout + res.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdr_time = max(os.path.getmtime(h) for h in _headers())
    jobs, objs = [], []
    for s in _sources():
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ_DIR, s[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_time):
            jobs.append((src, obj))
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as pool:
        for src, rc, log in pool.map(lambda j: _compile_one(nvcc, j[0], j[1], verbose), jobs):
            if rc != 0:
                raise RuntimeError("nvcc failed on %s:\n%s" % (src, log))
            if verbose:
                print(log, file=sys.stderr)
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH + ".tmp"] + objs
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    os.replace(LIB_PATH + ".tmp", LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
