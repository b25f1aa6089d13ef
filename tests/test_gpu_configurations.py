"""GPU (B200): the step kernels off make_env()'s configuration.

make_env()'s coefficients are axisymmetric (body axes 1 and 2 carry the same added mass and drag),
so with them every kernel runs the AXI form of the substep loop, and the general form's extra terms
(roll terms w1 w2 JdI0 / v1 v2 AdI0, separate axis-2 entries, quads 2-3 of the pipeline kernel's
rotational ring row) are either zero or equal to their axis-1 twins.  Here every production step
kernel runs coefficient sets that take the general form (parity.asymmetric_params, parity.one_break),
and observation widths other than 10 (0, 1 and 8 obstacles), against:

  * the float64 C oracle, one env-step at a time from identical state (per-step tolerance), also
    from a tumbling state (parity.tumbling), where the general form's roll / pitch terms are not
    below fp32 noise;
  * each other, bit for bit (the pipeline and the fused kernel round every operation identically);
  * the host build of the same body, for the randomised kernel (the oracle has no robustness switches).

Every test asserts the kernel it reached (SalpBatch.last_step_kernel), so that a routing change
cannot silently move a case onto another kernel."""
import numpy as np
import pytest

from grasp_lab_salp_b200 import PRECISION_F64, PRECISION_MIXED, SalpBatch
from grasp_lab_salp_b200.params import (FIELDS, RAND_ACTION, RAND_DISTURBANCE, RAND_DYNAMICS, RAND_LATENCY,
                                        RAND_OBSERVATION)
from oracle.salp_oracle import OracleVecEnv
from parity import (ASYM_FLOORS, AXISYM_CONDITIONS, MIXED_FLOORS, PER_STEP_CHANNELS, TOL_MIXED, TUMBLING_FLOORS,
                    ASYM_REWARD_FLOOR,
                    asymmetric_params, axisym_broken, golden_params, load_golden, lockstep_compare, obs_errors,
                    one_break, rel_err, sample_scene_pool, SMALL_CHANNELS, tumbling)

pytestmark = pytest.mark.gpu

PIPE = "salp_step_kernel_pipe4"
FUSED = "salp_step_kernel_lat<MIXED>"
F64 = "salp_step_kernel<F64>"
RANDOMIZED = "salp_step_kernel_lat<MIXED_RANDOMIZED>"

# route -> (envs, step() flags, the kernel it must reach)
ROUTES = {
    "pipe": (1000, {}, PIPE),                                  # one pipeline block per SM
    "pipe_2_blocks_per_sm": (6001, {}, PIPE),                  # 4737-9472 envs on 148 SMs
    "fused": (1000, dict(pipeline=False), FUSED),
    "fused_sorted": (2048, dict(pipeline=False, sort_by_k=True), FUSED),
    "f64": (1000, {}, F64),
}


def params_for(coefs, precision=PRECISION_MIXED, num_obstacles=2):
    if coefs == "asymmetric":
        return asymmetric_params(precision, num_obstacles)
    p = golden_params(load_golden("ref_random.npz"), precision=precision, num_obstacles=num_obstacles)
    assert axisym_broken(p) == set()          # make_env()'s defaults take the AXI form
    return p


def short_cycle_actions():
    """test_gpu_parity.test_pipeline_kernel_short_cycles_and_chunk_boundaries: cycles of K = 0, 1, 2, ...
    substeps (end of cycle on every position of the 8-substep hand-off chunks and the 32-substep flush),
    alone, behind a long and a tiny contraction, and with a nozzle turn.  [208, 3]"""
    ks = np.concatenate([np.arange(0, 42), [63, 64, 65, 66, 95, 96, 97, 127, 128, 129]])
    m = len(ks)
    acts = np.zeros((4 * m, 3), np.float32)
    coast = 0.125 + (np.tile(ks, 4) - 0.5) * 0.01
    acts[:, 1] = np.where(np.tile(ks, 4) > 0, coast / 10.0, 0.0)
    acts[m:2 * m, 0] = 0.3
    acts[2 * m:3 * m, 0] = 0.05
    acts[3 * m:, 2] = 0.7
    return acts


# Contractions next to the integrator's stability limit (a0 ~ 0.0885-0.094, DESIGN.md 3.3) amplify any
# rounding difference by orders of magnitude (states of 1e9 and more): fp32 and fp64 part there for good
# reason, and check_blowup_golden (test_gpu_parity.py) covers that neighbourhood.  The per-step
# comparisons keep their contractions out of this band (with room for the +-10 % action randomisation).
STABILITY_BAND = (0.075, 0.11)
# the blow-up neighbourhood itself, for the bit-identity tests (test_pipeline_kernel_matches_fused_kernel)
BLOWUP_ROWS = [[0, 0, 0], [1, 1, 1], [1, 0, -1], [0.088, 0, 0.5], [0.5, 0.5, 1e-4], [0.09, 0, 0], [0, 1, 1], [1, 1, 0]]


def edge_actions(seed, T, n):
    """Uniform-random actions with a whole warp and scattered rows of K = 0 cycles (step 1), short cycles
    (step 2: the shape moves almost all the time) and the crafted short-cycle set (step 3); no contraction
    in STABILITY_BAND."""
    acts = np.random.default_rng(seed).uniform([0, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
    a0 = acts[..., 0]
    lo, hi = STABILITY_BAND
    band = (a0 > lo) & (a0 < hi)
    a0[band] += hi - lo
    acts[1, 32:64] = 0.0
    acts[1, ::97] = 0.0
    acts[2, :, 1] *= 0.02
    if T > 3:
        sc = short_cycle_actions()
        acts[3, : min(n, len(sc))] = sc[:n]
    return acts


class Routed:
    """A SalpBatch whose step() always passes the same flags and records the kernel of every step."""

    def __init__(self, env, **flags):
        self.env, self.flags, self.kernels = env, flags, set()

    def step(self, actions, auto_reset=False):
        out = self.env.step(actions, auto_reset=auto_reset, **self.flags)
        self.kernels.add(self.env.last_step_kernel)
        return out

    def __getattr__(self, name):
        return getattr(self.env, name)


def oracle_lockstep(params, route, *, T=8, seed=3, floors=ASYM_FLOORS, reward_floor=ASYM_REWARD_FLOOR, num_obstacles=2,
                    n=None, tumble=False):
    """lockstep_compare(resync=True) of the kernel `route` reaches against the float64 oracle, with a
    scene pool, auto-reset and edge_actions(); tumble: a tumbling body before every step (parity.tumbling,
    TUMBLING_FLOORS).  Returns (product, oracle) for further checks."""
    n_route, flags, kernel = ROUTES[route]
    n = n or n_route
    assert (params.precision == PRECISION_F64) == (kernel == F64)
    prod = Routed(SalpBatch(n, params, seed=seed), **flags)
    orc = OracleVecEnv(n, params, seed=seed, threads=8)
    t, o = sample_scene_pool(np.random.default_rng(seed), n, 6, num_obstacles)
    prod.set_scene_pool(t, o)
    orc.set_scene_pool(t, o)
    acts = edge_actions(seed + 8, T, n)
    inject = tumbling(n) if tumble else None
    report = {}
    if kernel == F64:
        # smoke()'s bar for this kernel (the device libm differs from glibc's in the last bits), and for the
        # near-zero out-of-plane channels 1e-10 absolute, TOL_F64's (small_rtol x small_floor).  Measured
        # worst: 5.6e-9 (roll angle at the defaults, rounding noise), 1.8e-11 rad/s absolute on the driven
        # roll rate of asymmetric_params()
        lockstep_compare(prod, orc, acts, resync=True, rtol=1e-8, floor=1e-3, small_floor=1e-2,
                         num_obstacles=num_obstacles, report=report, inject=inject)
    else:
        lockstep_compare(prod, orc, acts, resync=True, rtol=TOL_MIXED["rtol"], floor=TOL_MIXED["floor"],
                         floors=TUMBLING_FLOORS if tumble else floors, num_obstacles=num_obstacles, report=report,
                         inject=inject, reward_floor=reward_floor)
    print(f"{route} n={n} D={prod.obs_dim}{' tumbling' if tumble else ''}: worst per-step errors",
          {k: f"{v:.2e}" for k, v in report.items()})
    assert prod.kernels == {kernel}, prod.kernels
    prod.check()
    return prod, orc


# ---------------------------------------------------------------------------------------------
# 1. every kernel against the float64 oracle, per step, on asymmetric coefficients
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tumble", [False, True], ids=["free", "tumbling"])
@pytest.mark.parametrize("route", list(ROUTES))
def test_asymmetric_coefficients_vs_oracle(route, tumble):
    precision = PRECISION_F64 if route == "f64" else PRECISION_MIXED
    prod, orc = oracle_lockstep(asymmetric_params(precision), route, tumble=tumble)
    assert orc.get_state("episode_index").max() > 0          # episodes ended and auto-reset on the way
    assert np.abs(orc.get_state("angvel_x")).max() > 1e-4     # roll is driven, not rounding noise


@pytest.mark.parametrize("tumble", [False, True], ids=["free", "tumbling"])
@pytest.mark.parametrize("name", AXISYM_CONDITIONS)
@pytest.mark.parametrize("route", ["pipe", "fused"])
def test_one_broken_axisymmetry_condition_vs_oracle(route, name, tumble):
    oracle_lockstep(one_break(name), route, T=4, tumble=tumble)


# ---------------------------------------------------------------------------------------------
# 2. bit identity across kernels on asymmetric coefficients
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1000, 6001])
def test_asymmetric_pipeline_kernel_matches_fused_kernels(n):
    """Every operation of the mixed loop is explicitly rounded, so the pipeline kernel (rotational
    coefficient half handed over in four quads per ring row in the general form) and the fused kernel,
    natural and K-sorted order, agree bit for bit: 12 free-running steps with K = 0 warps, short cycles
    and auto-resets; hand-off tags checked on alternate steps."""
    T = 12
    p = asymmetric_params(PRECISION_MIXED)
    acts = edge_actions(21, T, n)
    acts[0, :8] = BLOWUP_ROWS                               # incl. cycles that blow up and are cut
    acts[6] = acts[3]                                       # the short-cycle set once more, later in the episodes
    pipe, fused, fsort = (SalpBatch(n, p, seed=4) for _ in range(3))
    o = pipe.reset()
    np.testing.assert_array_equal(o, fused.reset())
    np.testing.assert_array_equal(o, fsort.reset())
    ended = 0
    for t in range(T):
        r1 = pipe.step(acts[t], auto_reset=True, check_handoff=(t % 2 == 0))
        assert pipe.last_step_kernel == PIPE
        r2 = fused.step(acts[t], auto_reset=True, pipeline=False)
        assert fused.last_step_kernel == FUSED
        r3 = fsort.step(acts[t], auto_reset=True, pipeline=False, sort_by_k=True)
        assert fsort.last_step_kernel == FUSED
        for other in (fused, fsort):
            for x, y in zip(r1, (other.obs, other.reward, other.terminated, other.truncated)):
                np.testing.assert_array_equal(x, y, err_msg=f"step {t}")
            for name in ("terminal_obs", "terms", "substeps"):
                np.testing.assert_array_equal(getattr(pipe, name), getattr(other, name), err_msg=f"{name} step {t}")
            done = (r1[2] | r1[3]).astype(bool)                 # (metric rows are defined where an episode ended)
            np.testing.assert_array_equal(pipe.metrics[done], other.metrics[done], err_msg=f"metrics step {t}")
        ended += int((r1[2] | r1[3]).sum())
    assert ended > 0
    for env in (pipe, fused, fsort):
        env.check()                                         # no SALP_ERR_HANDOFF
    for col in FIELDS:
        a = pipe.get_state(col)
        np.testing.assert_array_equal(a, fused.get_state(col), err_msg=col)
        np.testing.assert_array_equal(a, fsort.get_state(col), err_msg=col)


def test_asymmetric_pipeline_kernel_is_deterministic_at_full_size():
    """BASELINE's 4096 envs x 40 free-running steps, general form: two handles give the same bits."""
    n, T = 4096, 40
    p = asymmetric_params(PRECISION_MIXED)
    acts = np.random.default_rng(77).uniform([0, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
    a, b = SalpBatch(n, p, seed=5), SalpBatch(n, p, seed=5)
    np.testing.assert_array_equal(a.reset(), b.reset())
    for t in range(T):
        ra = a.step(acts[t], auto_reset=True)
        rb = b.step(acts[t], auto_reset=True)
        assert a.last_step_kernel == PIPE and b.last_step_kernel == PIPE
        for x, y in zip(ra, rb):
            np.testing.assert_array_equal(x, y)
        np.testing.assert_array_equal(a.substeps, b.substeps)
    for col in FIELDS:
        np.testing.assert_array_equal(a.get_state(col), b.get_state(col), err_msg=col)
    a.check()
    b.check()


# ---------------------------------------------------------------------------------------------
# 3. obstacle counts 0, 1, 8 (observation widths 6, 8, 22) through every kernel and I/O face
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("coefs", ["default", "asymmetric"])
@pytest.mark.parametrize("num_obstacles", [0, 1, 8])
@pytest.mark.parametrize("route", ["pipe", "fused", "f64"])
def test_obstacle_counts_vs_oracle(route, num_obstacles, coefs):
    """Per step against the oracle, then a masked reset on the device face against the oracle's."""
    import torch
    precision = PRECISION_F64 if route == "f64" else PRECISION_MIXED
    p = params_for(coefs, precision, num_obstacles)
    floors, reward_floor = (ASYM_FLOORS, ASYM_REWARD_FLOOR) if coefs == "asymmetric" else (MIXED_FLOORS, 10.0)
    prod, orc = oracle_lockstep(p, route, T=5, floors=floors, reward_floor=reward_floor, num_obstacles=num_obstacles)
    assert prod.obs_dim == 6 + 2 * num_obstacles
    n = prod.num_envs
    mask = np.zeros(n, np.uint8)
    mask[::7] = 1
    mask[-1] = 1                                            # the ragged last warp too
    obs_o = orc.reset(mask).copy()
    prod.dev["obs"].copy_(torch.from_numpy(prod.obs).cuda())
    obs_d = prod.reset_device(torch.from_numpy(mask).cuda())
    torch.cuda.synchronize()
    sel = mask == 1
    np.testing.assert_allclose(obs_d.cpu().numpy()[sel], obs_o[sel], rtol=1e-6, atol=1e-6)
    np.testing.assert_array_equal(obs_d.cpu().numpy()[~sel], prod.obs[~sel])
    for col in ("episode_index", "cycle", "ep_length", "target_x", "target_y"):
        np.testing.assert_array_equal(prod.get_state(col), orc.get_state(col), err_msg=col)


@pytest.mark.parametrize("coefs", ["default", "asymmetric"])
@pytest.mark.parametrize("num_obstacles", [0, 1, 8])
@pytest.mark.parametrize("route", ["pipe", "fused", "f64"])
def test_obstacle_counts_io_faces_bit_identical(route, num_obstacles, coefs):
    """The three I/O faces on the same steps, same bits: staged host (pageable numpy, through device
    buffers), zero-copy host (page-locked buffers written through mapped memory) and device
    (step_device(extras=True)).  n = 1000 leaves a ragged last warp for the tile write-out, and
    auto-resets write terminal-observation rows, at every observation width."""
    import torch
    n, flags, kernel = ROUTES[route]
    T = 8
    precision = PRECISION_F64 if route == "f64" else PRECISION_MIXED
    p = params_for(coefs, precision, num_obstacles)
    acts = edge_actions(40 + num_obstacles, T, n)
    pinned, paged, dev = (SalpBatch(n, p, seed=3) for _ in range(3))
    for name in ("obs", "terminal_obs", "reward", "terminated", "truncated"):
        setattr(paged, name, np.full_like(getattr(paged, name), 7))       # plain numpy: not page-locked
    a_pinned = pinned.host_buffer((n, 3), np.float32)
    o = pinned.reset()
    np.testing.assert_array_equal(o, paged.reset())
    np.testing.assert_array_equal(o, dev.reset_device().cpu().numpy())
    ended = 0
    for t in range(T):
        a_pinned[:] = acts[t]
        r1 = pinned.step(a_pinned, auto_reset=True, **flags)
        assert pinned.last_step_kernel == kernel
        r2 = paged.step(acts[t].copy(), auto_reset=True, **flags)
        assert paged.last_step_kernel == kernel
        r3 = dev.step_device(torch.from_numpy(acts[t]).cuda(), auto_reset=True, extras=True, **flags)
        assert dev.last_step_kernel == kernel
        torch.cuda.synchronize()
        r3 = [x.cpu().numpy() for x in r3]
        for x, y, z, what in zip(r1, r2, r3, ("obs", "reward", "terminated", "truncated")):
            np.testing.assert_array_equal(x, y, err_msg=f"{what} step {t}: zero-copy vs staged")
            np.testing.assert_array_equal(x, z, err_msg=f"{what} step {t}: zero-copy vs device")
        np.testing.assert_array_equal(pinned.terminal_obs, paged.terminal_obs)
        np.testing.assert_array_equal(pinned.terminal_obs, dev.dev["terminal_obs"].cpu().numpy())
        np.testing.assert_array_equal(pinned.substeps, paged.substeps)
        np.testing.assert_array_equal(pinned.substeps, dev.dev["substeps"].cpu().numpy())
        np.testing.assert_array_equal(pinned.terms, paged.terms)
        np.testing.assert_array_equal(pinned.terms, dev.dev["terms"].cpu().numpy())
        ended += int((r1[2] | r1[3]).sum())
    assert ended > 0
    assert pinned.obs.shape == (n, 6 + 2 * num_obstacles)
    for env in (pinned, paged, dev):
        env.check()


# ---------------------------------------------------------------------------------------------
# 4. the randomised kernel per step, against the host build of the same body
# ---------------------------------------------------------------------------------------------
SWITCHES = {"action": RAND_ACTION, "observation": RAND_OBSERVATION, "dynamics": RAND_DYNAMICS,
            "disturbance": RAND_DISTURBANCE, "latency": RAND_LATENCY,
            "all_but_latency": RAND_ACTION | RAND_OBSERVATION | RAND_DYNAMICS | RAND_DISTURBANCE}
# Worst per-step difference of the GPU kernel from the host build, measured on a B200 (rel_err with
# ASYM_FLOORS -- the dynamics switch makes every coefficient set asymmetric --, obs as in lockstep_compare):
#   observation, dynamics, disturbance, latency: 2.5e-5 (roll rate, dynamics at the defaults; the
#     disturbance's Box-Muller uses the device's fast log / sin / cos), 1.2e-4 on obs (dynamics, asymmetric)
#   with the action switch: 5.7e-3 in-plane (yaw rate), out-of-plane up to 2e3 x the floor.  The device
#     evaluates the +-10 % draw `v (1 + u x)` with one fused multiply-add, the host build (compiled without
#     contraction) as a product and a sum: the two builds fly actions one rounding apart, and the cycle
#     amplifies that, most in the out-of-plane channels, which are therefore not compared there.
RANDOMIZED_RTOL = 3e-4
RANDOMIZED_ACTION_RTOL = 1.5e-2


@pytest.mark.parametrize("coefs", ["default", "asymmetric"])
@pytest.mark.parametrize("switch", list(SWITCHES))
def test_randomized_kernel_vs_host_build(switch, coefs):
    """salp_step_kernel_lat<MIXED_RANDOMIZED> (per-env coefficient draws: always the general form)
    one env-step at a time from identical state against tests/emu, the host build of the same step
    body, which draws the same Philox streams.  A WEAKER reference than the oracle: it catches faults
    of the GPU build of this instantiation (device intrinsics, shared-memory tile, launch, the draws'
    keys on the device), not logic shared with the host build -- that is checked only statistically,
    against the live reference, by test_randomization.py.  Counters, flags and K bit-exact; floats
    within RANDOMIZED_RTOL (in-plane channels, obs and reward within RANDOMIZED_ACTION_RTOL with the
    action switch; see there)."""
    from emu_backend import EmuBatch
    n, T = 256, 10
    p = params_for(coefs)
    p.randomization = SWITCHES[switch]
    action = bool(p.randomization & RAND_ACTION)
    rtol = RANDOMIZED_ACTION_RTOL if action else RANDOMIZED_RTOL
    channels = [c for c in PER_STEP_CHANNELS if not (action and c in SMALL_CHANNELS)]
    gpu, host = SalpBatch(n, p, seed=13), EmuBatch(n, p, seed=13)
    np.testing.assert_allclose(gpu.reset(), host.reset(), rtol=1e-6, atol=1e-6)
    acts = edge_actions(50, T, n)
    worst = {}
    for t in range(T):
        if t:
            for col in FIELDS:
                gpu.set_state(col, host.get_state(col))
        og, rg, teg, trg = gpu.step(acts[t], auto_reset=True)
        assert gpu.last_step_kernel == RANDOMIZED
        oh, rh, teh, trh = host.step(acts[t], auto_reset=True)
        ctx = f"{switch} step {t}"
        np.testing.assert_array_equal(gpu.substeps, host.substeps, err_msg=f"K {ctx}")
        np.testing.assert_array_equal(teg, teh, err_msg=f"terminated {ctx}")
        np.testing.assert_array_equal(trg, trh, err_msg=f"truncated {ctx}")
        for col in ("cycle", "phase", "ep_length", "episode_index", "target_x", "target_y"):
            np.testing.assert_array_equal(gpu.get_state(col), host.get_state(col), err_msg=f"{col} {ctx}")
        errs = {c: float(rel_err(gpu.get_state(c), host.get_state(c), ASYM_FLOORS[c]).max()) for c in channels}
        errs["reward"] = float(rel_err(gpu.terms[:, 7], host.terms[:, 7], 10.0).max())
        errs.update(obs_errors(gpu.terminal_obs, host.terminal_obs, 0.1, "obs"))
        errs.update(obs_errors(og, oh, 0.1, "obs_after_reset"))
        for k, v in errs.items():
            worst[k] = max(worst.get(k, 0.0), v)
        bad = {k: v for k, v in errs.items() if not v <= rtol}
        assert not bad, f"{ctx}: {bad}"
    print(f"randomized {switch} {coefs}: worst", {k: f"{v:.2e}" for k, v in worst.items()})
    assert host.get_state("episode_index").max() > 0       # episode keys advanced (auto-reset)
    gpu.check()
