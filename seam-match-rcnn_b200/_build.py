"""Build the CUDA library in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

The resulting ``libseam_b200.so`` sits next to this file, is git-ignored and travels to the
GPU box with the source snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libseam_b200.so")
INFO_PATH = os.path.join(HERE, "libseam_b200.buildinfo")
SOURCES = ["seam_b200.cu"]
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh"))   # every header goes into the content hash
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; cannot build libseam_b200.so")


def source_hash() -> str:
    """Content hash of everything that goes into the library (mtimes do not survive the
    snapshot copy to the GPU box, contents do)."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "seam_b200.h"))
    for d in deps:
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH) or not os.path.exists(INFO_PATH):
        return True
    with open(INFO_PATH) as f:
        return f.read().strip() != source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ -> libseam_b200.so (only when sources are newer). Returns the path.

    Safe under several processes (one rank per GPU starting at once): the build is serialised by a lock file, the
    library is written under a temporary name and renamed into place, so nobody ever maps a half-written file."""
    if not force and not is_stale():
        return LIB_PATH
    import fcntl
    with open(LIB_PATH + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not is_stale():             # another process built it while this one waited
                return LIB_PATH
            tmp = f"{LIB_PATH}.tmp{os.getpid()}"
            cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", tmp] + \
                  [os.path.join(CSRC, s) for s in SOURCES]
            proc = subprocess.run(cmd, capture_output=True, text=True)
            if proc.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
            if verbose:
                print(proc.stderr)
            os.replace(tmp, LIB_PATH)
            with open(INFO_PATH + ".tmp", "w") as f:
                f.write(source_hash())
            os.replace(INFO_PATH + ".tmp", INFO_PATH)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH
