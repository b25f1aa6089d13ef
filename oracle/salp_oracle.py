"""TEST INFRASTRUCTURE ONLY -- ctypes wrapper of oracle/salp_oracle.c (the CPU restatement).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product (grasp_lab_salp_b200/) never does.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from grasp_lab_salp_b200.params import (NUM_EPISODE_METRICS, SalpParams, default_params,
                                        field_dtype, field_id)

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libsalp_oracle.so")
_HASH_PATH = _LIB_PATH + ".hash"
_lib = None
_built = None


def _digest() -> str:
    h = hashlib.sha256()
    for f in (os.path.join(_HERE, "salp_oracle.c"), os.path.join(_HERE, "..", "include", "salp_b200.h"),
              os.path.join(_HERE, "Makefile")):
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force: bool = False) -> str:
    """Path of the oracle library, compiled first if missing or built from other sources (content
    hash: a copied tree does not keep mtimes).  A read-only tree gets it in a temporary directory."""
    global _built
    if _built is not None and not force:
        return _built
    d = _digest()
    if not force and os.path.exists(_LIB_PATH) and os.path.exists(_HASH_PATH):
        with open(_HASH_PATH) as fh:
            if fh.read() == d:
                _built = _LIB_PATH
                return _built
    out = os.path.dirname(_LIB_PATH)
    in_tree = os.access(out if os.path.isdir(out) else _HERE, os.W_OK)
    if not in_tree:
        out = tempfile.mkdtemp(prefix="salp_oracle_")
    subprocess.run(["make", "-s", "-B", "-C", _HERE, f"OUT={out}"], check=True, stdout=subprocess.DEVNULL)
    if in_tree:
        with open(_HASH_PATH, "w") as fh:
            fh.write(d)
    _built = os.path.join(out, "libsalp_oracle.so")
    return _built


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.orc_create.restype = C.c_void_p
        L.orc_create.argtypes = [C.POINTER(SalpParams), C.c_int64, C.c_uint64, C.c_int64]
        L.orc_destroy.argtypes = [C.c_void_p]
        L.orc_set_scene_pool.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
        L.orc_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        L.orc_step.argtypes = [C.c_void_p] + [C.c_void_p] * 9 + [C.c_int, C.c_int64, C.c_int64]
        L.orc_get_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.orc_get_state.restype = C.c_int
        L.orc_set_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.orc_set_state.restype = C.c_int
        L.orc_get_cycle_plan.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_np_sincosf.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def np_sincosf(x: np.ndarray):
    x = np.ascontiguousarray(x, dtype=np.float32)
    s = np.empty_like(x)
    c = np.empty_like(x)
    lib().orc_np_sincosf(_ptr(x), _ptr(s), _ptr(c), x.size)
    return s, c


class OracleVecEnv:
    """N independent scalar float64 environments; optional thread pool over env ranges."""

    def __init__(self, num_envs: int, params: SalpParams | None = None, seed: int = 0,
                 env_id_offset: int = 0, threads: int = 1):
        self.params = (params or default_params()).copy()
        self.num_envs = int(num_envs)
        self.obs_dim = self.params.obs_dim
        self._h = C.c_void_p(lib().orc_create(C.byref(self.params), self.num_envs, seed, env_id_offset))
        self.threads = max(1, int(threads))
        self._pool = ThreadPoolExecutor(self.threads) if self.threads > 1 else None
        n, d = self.num_envs, self.obs_dim
        self.obs = np.zeros((n, d), np.float32)
        self.terminal_obs = np.zeros((n, d), np.float32)
        self.reward = np.zeros(n, np.float64)
        self.terminated = np.zeros(n, np.uint8)
        self.truncated = np.zeros(n, np.uint8)
        self.terms = np.zeros((n, 8), np.float64)
        self.substeps = np.zeros(n, np.int32)
        self.metrics = np.zeros((n, NUM_EPISODE_METRICS), np.float64)

    def close(self):
        if self._h:
            lib().orc_destroy(self._h)
            self._h = None
        if self._pool:
            self._pool.shutdown()
            self._pool = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ranges(self):
        n, t = self.num_envs, self.threads
        # small interleaved chunks: K varies a lot between envs
        chunk = max(1, n // (t * 8))
        return [(a, min(chunk, n - a)) for a in range(0, n, chunk)]

    def _run(self, fn):
        if self._pool is None:
            fn(0, self.num_envs)
        else:
            list(self._pool.map(lambda r: fn(*r), self._ranges()))

    def set_scene_pool(self, targets, obstacles):
        if targets is None:
            lib().orc_set_scene_pool(self._h, None, None, 0)
            return
        targets = np.ascontiguousarray(targets, np.float32)
        obstacles = np.ascontiguousarray(obstacles, np.float32)
        P = targets.shape[1]
        assert targets.shape == (self.num_envs, P, 2)
        assert obstacles.shape == (self.num_envs, P, self.params.num_obstacles, 2)
        lib().orc_set_scene_pool(self._h, _ptr(targets), _ptr(obstacles), P)

    def reset(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self._run(lambda a, c: lib().orc_reset(self._h, _ptr(m), _ptr(self.obs), a, c))
        return self.obs

    def step(self, actions, auto_reset: bool = False):
        actions = np.ascontiguousarray(actions, np.float32)
        assert actions.shape == (self.num_envs, 3)
        self._run(lambda a, c: lib().orc_step(
            self._h, _ptr(actions), _ptr(self.obs), _ptr(self.reward), _ptr(self.terminated),
            _ptr(self.truncated), _ptr(self.terminal_obs), _ptr(self.terms), _ptr(self.substeps),
            _ptr(self.metrics), int(auto_reset), a, c))
        return self.obs, self.reward, self.terminated, self.truncated

    def get_state(self, name: str) -> np.ndarray:
        out = np.zeros(self.num_envs, field_dtype(name))
        rc = lib().orc_get_state(self._h, field_id(name), _ptr(out))
        if rc != 0:
            raise KeyError(name)
        return out

    def set_state(self, name: str, values):
        v = np.ascontiguousarray(np.broadcast_to(values, (self.num_envs,)), field_dtype(name))
        if lib().orc_set_state(self._h, field_id(name), _ptr(v)) != 0:
            raise KeyError(name)

    def cycle_plan(self) -> np.ndarray:
        """[N,5]: refill_time, jet_time, turn_time, total, total_is_float32 of the last step."""
        out = np.zeros((self.num_envs, 5), np.float64)
        lib().orc_get_cycle_plan(self._h, _ptr(out))
        return out
