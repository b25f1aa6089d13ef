"""CPU: the wide form of the pipeline kernel starts each producer warp's fp64 shape track at the first
substep of its chunk (two updates of a track that carries nothing) instead of carrying it from substep 1.
The host build of shape_front (tests/emu/shape_seed_check.cu) checks that the seeded track gives the
carried track's bits at every chunk start and on both sides of the phase edges (k_T0, k_jet) and of the
end of the updates, and that every later ShapeFront is identical."""
import ctypes as C
import fcntl
import os
import shutil
import subprocess

import numpy as np
import pytest

from grasp_lab_salp_b200 import PRECISION_MIXED, default_params
from parity import asymmetric_params

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
SRC = os.path.join(HERE, "shape_seed_check.cu")
OUT = os.path.join(HERE, "_build")


def _lib():
    os.makedirs(OUT, exist_ok=True)
    lib = os.path.join(OUT, "libshape_seed_check.so")
    with open(lib + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "-shared",
                        "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-mfma", "-o", lib + ".tmp", SRC],
                       check=True, capture_output=True, text=True)
        os.replace(lib + ".tmp", lib)
    L = C.CDLL(lib)
    L.salp_seed_check.restype = C.c_int
    L.salp_seed_check.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_int, C.POINTER(C.c_int)]
    return L


@pytest.fixture(scope="module")
def lib():
    return _lib()


def _actions(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.random((n, 3), dtype=np.float32)
    a[:, 2] = a[:, 2] * 2 - 1
    edge = np.array([[1, 1, 0], [1, 0, 0], [0.05, 0, 0.3], [0.5, 0.2, -1], [0, 1, 1]], dtype=np.float32)
    return np.concatenate([edge, a])


@pytest.mark.parametrize("params", ["default", "asymmetric"])
def test_seeded_shape_track_matches_carried_track(lib, params):
    p = default_params() if params == "default" else asymmetric_params(PRECISION_MIXED)
    seeds = fronts = 0
    for a in _actions(60, 7):
        for last in (-1, 10_000):               # the lane's own end of shape motion, or every substep to K
            out = (C.c_int * 6)()
            bad = lib.salp_seed_check(C.byref(p), float(a[0]), float(a[1]), float(a[2]), last, out)
            assert bad == 0, f"action {a}: {bad} mismatches (K {out[0]}, k_T0 {out[1]}, k_jet {out[2]}, kA {out[3]})"
            seeds += out[4]
            fronts += out[5]
    assert seeds > 1000 and fronts > 100_000
