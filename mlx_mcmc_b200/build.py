"""Build libb200mcmc.so in-tree with nvcc for sm_100a (no GPU needed: nvcc cross-compiles).

    python -m mlx_mcmc_b200.build [--force]

The shared library is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(CSRC, "libb200mcmc.so")
STAMP = os.path.join(CSRC, ".build_stamp")

SOURCES = ["capi.cu", "pointwise.cu", "nuts_pointwise.cu", "glm.cu", "glm_samplers.cu", "glm_tc.cu", "comm.cu", "diag.cu", "sample.cu", "jit.cu", "loglik.cu"]
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-I", INCLUDE,
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _fingerprint() -> str:
    # location independent: the snapshot on the GPU box lives under another root, and a library built here must count
    # as current there (it is the binary the parity claims refer to)
    h = hashlib.sha256(" ".join(f for f in NVCC_FLAGS if f != INCLUDE).encode())
    names = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    for n in names + ["../../include/b200mcmc.h"]:
        with open(os.path.join(CSRC, n), "rb") as f:
            h.update(n.encode())
            h.update(f.read())
    return h.hexdigest()


def is_current() -> bool:
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _fingerprint()


def build_debug() -> str:
    """The same sources with -DB2M_DEBUG_ASSERTS (index / invariant asserts inside the kernels) into
    csrc/_debug/libb200mcmc.so; selected for a process with B2M_LIB=<path> (tools/debug_asserts_smoke.py)."""
    nvcc = _nvcc()
    out_dir = os.path.join(CSRC, "_debug")
    os.makedirs(out_dir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(out_dir, src.replace(".cu", ".o"))
        r = subprocess.run([nvcc, *NVCC_FLAGS, "-DB2M_DEBUG_ASSERTS", "-c", os.path.join(CSRC, src), "-o", obj],
                           capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return obj

    with cf.ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(compile_one, _sources()))
    lib = os.path.join(out_dir, "libb200mcmc.so")
    r = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib, *objs, "-lcudart", "-ldl"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a and link libb200mcmc.so.  Returns the library path."""
    if not force and is_current():
        return LIB
    # one builder at a time: ranks of a torchrun job that all find the library stale must not compile into the same
    # object files concurrently; the ones that waited find it current
    import fcntl
    with open(os.path.join(CSRC, ".build_lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and is_current():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    nvcc = _nvcc()
    objs = []

    def compile_one(src):
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(compile_one, _sources()))
    r = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-lcudart", "-ldl"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(STAMP, "w") as f:
        f.write(_fingerprint())
    return LIB


if __name__ == "__main__":
    print(build_debug() if "--debug" in sys.argv else build(force="--force" in sys.argv, verbose="-v" in sys.argv))
