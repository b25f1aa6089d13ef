"""ctypes binding of libsalp_b200.so -- exactly the entry points of include/salp_b200.h.

This is the binding a maintainer of the reference would add (INTEGRATION.md shows the same
stub).  There is NO CPU fallback: if the CUDA library is missing and cannot be built, or no
sm_100 GPU is present, the calls fail loudly (ImportError / SalpError).
"""
from __future__ import annotations

import ctypes as C
import os

from .params import SalpParams

OK = 0
ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_RANGE, ERR_ALLOC, ERR_HANDOFF = -1, -2, -3, -4, -5, -6
_ERR_NAMES = {ERR_INVALID: "SALP_ERR_INVALID", ERR_CUDA: "SALP_ERR_CUDA", ERR_NO_DEVICE: "SALP_ERR_NO_DEVICE",
              ERR_RANGE: "SALP_ERR_RANGE", ERR_ALLOC: "SALP_ERR_ALLOC", ERR_HANDOFF: "SALP_ERR_HANDOFF"}


class SalpError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{_ERR_NAMES.get(code, code)}: {message}")
        self.code = code


class SalpStepIO(C.Structure):
    """struct SalpStepIO (include/salp_b200.h); raw device or host addresses."""
    _fields_ = [("actions", C.c_void_p), ("obs", C.c_void_p), ("reward", C.c_void_p),
                ("terminated", C.c_void_p), ("truncated", C.c_void_p), ("terminal_obs", C.c_void_p),
                ("reward_terms", C.c_void_p), ("substeps", C.c_void_p), ("episode_metrics", C.c_void_p)]


# every symbol include/salp_b200.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "salp_default_params": (C.c_int, [C.POINTER(SalpParams)]),
    "salp_create": (C.c_int, [C.POINTER(SalpParams), C.c_int64, C.c_int, C.c_uint64, C.c_int64,
                              C.POINTER(C.c_void_p)]),
    "salp_destroy": (C.c_int, [C.c_void_p]),
    "salp_num_envs": (C.c_int64, [C.c_void_p]),
    "salp_obs_dim": (C.c_int32, [C.c_void_p]),
    "salp_last_error": (C.c_char_p, [C.c_void_p]),
    "salp_build_info": (C.c_char_p, []),
    "salp_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "salp_step": (C.c_int, [C.c_void_p, C.POINTER(SalpStepIO), C.c_uint32, C.c_void_p]),
    "salp_reset_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "salp_step_host": (C.c_int, [C.c_void_p, C.POINTER(SalpStepIO), C.c_uint32]),
    "salp_set_scene_pool": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "salp_get_state": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64]),
    "salp_set_state": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64]),
    "salp_state_ptr": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "salp_trace_cycle": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]),
    "salp_check": (C.c_int, [C.c_void_p]),
    "salp_launch_count": (C.c_int64, [C.c_void_p]),
    "salp_last_step_kernel": (C.c_char_p, [C.c_void_p]),
    "salp_abi_version": (C.c_int32, []),
    "salp_sizeof_params": (C.c_int64, []),
    "salp_sizeof_step_io": (C.c_int64, []),
    "salp_probe_fp32_peak": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "salp_debug_p4_stamps": (C.c_int, [C.POINTER(C.c_longlong)]),
    "salp_mlp_packed_size": (C.c_int64, [C.c_int32]),
    "salp_mlp_act": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_float),
                               C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "salp_lstm_weight_bytes": (C.c_int64, []),
    "salp_lstm_scratch_bytes": (C.c_int64, [C.c_int64]),
    "salp_lstm_pack_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                         C.c_void_p, C.c_void_p, C.c_void_p]),
    "salp_lstm_cell": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "salp_lstm_check": (C.c_int, []),
    "salp_sac_weight_bytes": (C.c_int64, [C.c_int32]),
    "salp_sac_pack_weights": (C.c_int, [C.c_void_p] * 8 + [C.c_int32, C.c_void_p, C.c_void_p]),
    "salp_sac_act": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_float),
                               C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_void_p]),
    "salp_sac_pack_weights_grouped": (C.c_int, [C.c_void_p] * 8 + [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "salp_sac_act_grouped": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                       C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_void_p]),
    "salp_sac_check": (C.c_int, []),
    "salp_lstm_pointwise_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "salp_lstm_pointwise_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
}

ABI_VERSION = 1        # SALP_ABI_VERSION of include/salp_b200.h this binding mirrors

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libsalp_b200.so")
_cdll = None


def bind(cdll, names=None):
    """Attach prototypes to a loaded library (also used by tests/emu with its host build)."""
    for name, (res, args) in PROTOTYPES.items():
        if names is not None and name not in names:
            continue
        fn = getattr(cdll, name)
        fn.restype = res
        fn.argtypes = args
    return cdll


def check_layout(cdll):
    """A library whose struct layouts differ from the ctypes mirrors would be driven through the
    wrong offsets: refuse it (stale prebuilt .so, or a header edited without its mirror)."""
    got = (cdll.salp_abi_version(), cdll.salp_sizeof_params(), cdll.salp_sizeof_step_io())
    want = (ABI_VERSION, C.sizeof(SalpParams), C.sizeof(SalpStepIO))
    if got != want:
        raise ImportError(f"libsalp_b200.so does not match this binding: (abi, sizeof SalpParams, sizeof SalpStepIO) "
                          f"= {got}, expected {want}; rebuild with `python -m grasp_lab_salp_b200.build --force`")


def load():
    """Load (building in-tree first if the sources changed and nvcc is available)."""
    global _cdll
    if _cdll is not None:
        return _cdll
    from . import build
    try:
        build.build_library()
    except Exception as e:
        # no nvcc on this box: the prebuilt .so that travelled with the repo is used -- but only if it
        # was built from exactly these sources (content hash), never a stale one
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"libsalp_b200.so is missing and could not be built ({e}); "
                              "the SALP simulator has no CPU fallback") from e
        if build.is_stale():
            raise ImportError(f"libsalp_b200.so is stale (sources changed since it was built) and the rebuild "
                              f"failed: {e}") from e
    cdll = bind(C.CDLL(LIB_PATH))
    check_layout(cdll)
    _cdll = cdll
    return _cdll
