"""GPU: the 8-warp form of the pipeline kernel (one block per SM, <= #SMs x 32 envs), whose producer
warps hand the dyn warp whole coefficient sets (salp_pipe4_kernel.cuh), against the 4-warp form of the
same kernel (SALP_PIPE_WIDE=0) and the fused kernel: bit for bit on every output and on every state
column.  Each test asserts the kernel it reached and, through the stamp block of
salp_debug_p4_stamps, which form ran."""
import ctypes as C
import os

import numpy as np
import pytest

from grasp_lab_salp_b200 import PRECISION_MIXED, SalpBatch, _lib
from grasp_lab_salp_b200.params import FIELDS
from parity import asymmetric_params, golden_params, load_golden

pytestmark = pytest.mark.gpu

PIPE = "salp_step_kernel_pipe4"
STAMPS = 0x20000000          # salp_pipe4_kernel.cuh: SALP_P4_FLAG_STAMPS


def default_params_(num_obstacles=2):
    return golden_params(load_golden("ref_random.npz"), precision=PRECISION_MIXED, num_obstacles=num_obstacles)


def threads_of_pipeline_block(n, params, wide):
    """Block size of the pipeline kernel at n envs (stamp 10): 256 for the 8-warp form, 128 for the 4-warp one."""
    import torch
    b = SalpBatch(n, params, seed=0)
    b.reset_device()
    env = {} if wide else {"SALP_PIPE_WIDE": "0"}
    with _env(env):
        b.step_device(torch.full((n, 3), 0.5, device="cuda"), extra_flags=STAMPS)
    assert b.last_step_kernel == PIPE
    out = (C.c_longlong * 16)()
    assert _lib.load().salp_debug_p4_stamps(out) == 0
    b.check()
    b.close()
    return out[10]


class _env:
    def __init__(self, kv):
        self.kv, self.old = kv, {}

    def __enter__(self):
        for k, v in self.kv.items():
            self.old[k] = os.environ.get(k)
            os.environ[k] = v

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v


def compare_forms(n, params, acts, check_handoff=False):
    """Step wide / 4-warp / fused batches through acts [T, n, 3] with auto-reset; every output and every
    state column must agree bit for bit."""
    assert "SALP_PIPE_WIDE" not in os.environ
    wide, four, fused = (SalpBatch(n, params, seed=5) for _ in range(3))
    r0 = [x.reset() for x in (wide, four, fused)]
    np.testing.assert_array_equal(r0[0], r0[1])
    for t in range(len(acts)):
        rw = wide.step(acts[t], auto_reset=True, check_handoff=check_handoff)
        assert wide.last_step_kernel == PIPE
        with _env({"SALP_PIPE_WIDE": "0"}):
            r4 = four.step(acts[t], auto_reset=True)
        assert four.last_step_kernel == PIPE
        rf = fused.step(acts[t], auto_reset=True, pipeline=False)
        assert fused.last_step_kernel != PIPE
        for x, y, z in zip(rw, r4, rf):
            np.testing.assert_array_equal(x, y)
            np.testing.assert_array_equal(x, z)
        np.testing.assert_array_equal(wide.substeps, fused.substeps)
    for b in (wide, four, fused):
        b.check()                               # (checked mode: no SALP_ERR_HANDOFF)
    for col in FIELDS:
        a = wide.get_state(col)
        np.testing.assert_array_equal(a, four.get_state(col), err_msg=col)
        np.testing.assert_array_equal(a, fused.get_state(col), err_msg=col)
    for b in (wide, four, fused):
        b.close()


def uniform(rng, T, n):
    a = rng.random((T, n, 3), dtype=np.float32)
    a[..., 2] = a[..., 2] * 2 - 1
    return a


def clipped_gaussian(rng, T, n):
    a = rng.normal(0.4, 0.35, (T, n, 3)).astype(np.float32)
    a[..., :2] = np.clip(a[..., :2], 0, 1)
    a[..., 2] = np.clip(a[..., 2] * 2 - 0.8, -1, 1)
    return a


@pytest.mark.parametrize("dist", ["uniform", "clipped_gaussian"])
def test_wide_form_matches_four_warp_form_and_fused_kernel(dist):
    n, T = 4096, 32
    p = default_params_()
    assert threads_of_pipeline_block(n, p, wide=True) == 256
    assert threads_of_pipeline_block(n, p, wide=False) == 128
    rng = np.random.default_rng(11)
    compare_forms(n, p, (uniform if dist == "uniform" else clipped_gaussian)(rng, T, n))


@pytest.mark.parametrize("n", [1, 31, 33, 4095, 4736])
def test_wide_form_ragged_sizes(n):
    p = default_params_()
    assert threads_of_pipeline_block(n, p, wide=True) == 256
    acts = uniform(np.random.default_rng(n), 10, n)
    acts[1, : min(n, 64)] = 0.0                 # warps where every lane has K = 0
    acts[2, :, 1] *= 0.02                       # short cycles: the shape moves almost all the time
    compare_forms(n, p, acts)


def test_wide_form_short_cycles_and_chunk_edges():
    """Cycles of K = 0, 1, 2, ... substeps (W at every position of the 8-substep chunks, inside chunk 0,
    Kw < 8), alone and behind long, tiny and no contractions (test_gpu_configurations.short_cycle_actions)."""
    ks = np.concatenate([np.arange(0, 42), [63, 64, 65, 66, 95, 96, 97, 127, 128, 129]])
    m = len(ks)
    a = np.zeros((4 * m, 3), np.float32)
    coast = 0.125 + (np.tile(ks, 4) - 0.5) * 0.01
    a[:, 1] = np.where(np.tile(ks, 4) > 0, coast / 10.0, 0.0)
    a[m:2 * m, 0] = 0.3
    a[2 * m:3 * m, 0] = 0.05
    a[3 * m:, 2] = 0.7
    # every warp of 32 lanes alone, too: lane i's cycle is K = ks[i], so each warp ends inside its first chunks
    acts = np.repeat(a[None], 3, axis=0)
    p = default_params_()
    assert threads_of_pipeline_block(len(a), p, wide=True) == 256
    compare_forms(len(a), p, acts)


@pytest.mark.parametrize("coefs,num_obstacles", [("asymmetric", 2), ("default", 0), ("default", 1), ("default", 8)])
def test_wide_form_configurations(coefs, num_obstacles):
    """asymmetric_params() takes the general form (seven-quad rows of ring C); 0, 1 and 8 obstacles
    change the observation tile of the epilogue."""
    p = asymmetric_params(PRECISION_MIXED, num_obstacles) if coefs == "asymmetric" else default_params_(num_obstacles)
    n = 2048
    assert threads_of_pipeline_block(n, p, wide=True) == 256
    compare_forms(n, p, uniform(np.random.default_rng(num_obstacles + 3), 12, n))


def test_wide_form_checked_handoff_at_full_size():
    """SALP_STEP_CHECK_HANDOFF: every ring C row carries its substep tag, checked by the dyn warp; the
    checked wide kernel gives the bits of the unchecked one (and of the 4-warp form and the fused kernel)."""
    n, T = 4096, 60
    acts = uniform(np.random.default_rng(31), T, n)
    acts[1, :64] = 0.0
    acts[2, :, 1] *= 0.02
    compare_forms(n, default_params_(), acts, check_handoff=True)
