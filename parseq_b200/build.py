"""Builds libparseq_b200.so in-tree with nvcc for sm_100a (no torch involved in the build)."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libparseq_b200.so")
SOURCES = ["engine.cu"]
HEADERS = ["ptx.cuh", "gemm.cuh", "kernels.cuh", "dec_ar.cuh", "dec_ar2.cuh", "attn_tc.cuh", "gemm_ln.cuh", "gemm_ln2.cuh", "mlp_ln.cuh", "resize.cuh", os.path.join("..", "..", "include", "parseq_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    import fcntl
    os.makedirs(LIB_DIR, exist_ok=True)
    # one builder at a time (several ranks may import concurrently); the library appears atomically
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not needs_build():        # another process built it while we waited
            return LIB_PATH
        tmp = LIB_PATH + f".tmp{os.getpid()}"
        cmd = [_nvcc()] + NVCC_FLAGS + ["-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            if os.path.exists(tmp):
                os.remove(tmp)
            raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
        os.replace(tmp, LIB_PATH)
        if verbose:
            print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force=True, verbose=True))
