"""In-tree build of libsalp_b200.so (the C-ABI library of include/salp_b200.h) with nvcc.

sm_100a only, -lineinfo so ncu's source page maps to the .cu/.cuh files.  nvcc cross-compiles
without a GPU, so this also runs in the GPU-less build container.  The .so is git-ignored but
travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsalp_b200.so")
OBJ_DIR = os.path.join(HERE, "_obj")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
          "-Xptxas", "-v"]
# translation unit -> extra flags
UNITS = {
    "salp_kernels.cu": [],
    "salp_step_f64.cu": ["-fmad=false"],   # reference mode: no FMA contraction
    "salp_capi.cu": [],
    "salp_policy.cu": [],
    "salp_lstm.cu": [],                    # tcgen05 / TMA LSTM cell (needs the sm_100a target)
    "salp_lstm_train.cu": [],              # element-wise halves of the learner's LSTM step
    "salp_sac.cu": [],                     # SAC actor: SIMT layer 1, tcgen05 layer 2, fused heads
}


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")
    return exe


def _sources():
    out = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    out.append(os.path.join(HERE, "..", "include", "salp_b200.h"))
    out.append(os.path.abspath(__file__))
    return out


def _digest() -> str:
    import hashlib
    h = hashlib.sha256()
    for s in _sources():
        with open(s, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


HASH_FILE = os.path.join(HERE, "libsalp_b200.so.hash")


def is_stale() -> bool:
    """Content hash, not mtime: the gpurun snapshot does not preserve mtimes."""
    if not os.path.exists(LIB) or not os.path.exists(HASH_FILE):
        return True
    with open(HASH_FILE) as f:
        return f.read().strip() != _digest()


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    os.makedirs(OBJ_DIR, exist_ok=True)
    # ranks of one torchrun job may find the library stale together: one builds, the rest wait
    import fcntl
    with open(os.path.join(OBJ_DIR, "build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not is_stale():
            return LIB
        return _build_locked(verbose)


def _build_locked(verbose: bool) -> str:
    objs = []
    log = []
    for unit, extra in UNITS.items():
        obj = os.path.join(OBJ_DIR, unit.replace(".cu", ".o"))
        cmd = [nvcc(), *ARCH, *COMMON, *extra, "-c", os.path.join(CSRC, unit), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError(f"nvcc failed on {unit}")
        objs.append(obj)
    cmd = [nvcc(), *ARCH, "-shared", "-o", LIB + ".tmp", *objs, "-Xlinker", "--exclude-libs,ALL"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        sys.stderr.write(log[-1])
        raise RuntimeError("link of libsalp_b200.so failed")
    os.replace(LIB + ".tmp", LIB)
    with open(os.path.join(OBJ_DIR, "build.log"), "w") as f:
        f.write("\n".join(log))
    with open(HASH_FILE, "w") as f:
        f.write(_digest())
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
