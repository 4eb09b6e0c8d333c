"""Builds libsc_b200.so (sm_100a only) in-tree with nvcc.  No JIT cache, no torch extension:
the product boundary is a plain C ABI (include/scb.h) loaded through ctypes."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsc_b200.so")
SOURCES = ["api.cu", "mesh_ops.cu", "nbody.cu", "assemble.cu", "getrf.cu", "getrs.cu", "spmv.cu", "diag.cu", "delaunay.cu",
           "vortex.cu", "interp.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xptxas=-v",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


STAMP = LIB + ".stamp"
ABI_VERSION = 205  # must equal scb_version() of the sources (csrc/api.cu)


def source_digest() -> str:
    """Content hash of everything the library is built from (sources, header, flags).  Content, not
    mtimes: the tree is copied to the GPU box and checkouts reset timestamps."""
    import hashlib

    h = hashlib.blake2b(digest_size=16)
    deps = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    deps.append(os.path.join(os.path.dirname(HERE), "include", "scb.h"))
    for d in deps:
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build() -> bool:
    """True when libsc_b200.so is missing or was built from other sources than the ones in the tree."""
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    try:
        with open(STAMP) as f:
            return f.read().strip() != source_digest()
    except OSError:
        return True


def build(force: bool = False, verbose: bool = False) -> str:
    """Builds the library if needed.  Safe to call from several processes at once (torchrun ranks):
    an exclusive file lock serialises the builders and the late-comers find an up-to-date library."""
    if not force and not needs_build():
        return LIB
    import fcntl

    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    with open(os.path.join(HERE, "build", ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    nvcc = _nvcc()
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    with open(os.path.join(HERE, "build", "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    tmp = LIB + f".tmp{os.getpid()}"
    cmd = [nvcc, "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    os.replace(tmp, LIB)  # atomic: a concurrent loader never maps a half-written file
    with open(STAMP, "w") as f:
        f.write(source_digest())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
