"""CPU: the device step body, compiled for the host (tests/emu), against the golden traces of
the live Python reference and against the C oracle.  Checks kernel LOGIC without a GPU."""
import numpy as np
import pytest

from emu_backend import EmuBatch, emu_cdll, emu_lane_cdll
from grasp_lab_salp_b200 import PRECISION_F64, PRECISION_MIXED
from oracle.salp_oracle import OracleVecEnv
from parity import (check_blowup_golden, ASYM_FLOORS, AXISYM_CONDITIONS, TOL_F64, MIXED_FLOORS, TOL_MIXED, TOL_MIXED_FREE_RUN,
                    asymmetric_params, axisym_broken, golden_params, lockstep_compare, one_break, sample_scene_pool, load_golden,
                    replay_golden, tumbling, TUMBLING_FLOORS)

GOLDENS = ["ref_fixed10.npz", "ref_edge.npz", "ref_random.npz", "ref_clipped.npz"]


@pytest.mark.parametrize("name", GOLDENS)
def test_emu_f64_matches_reference_trace(name):
    g = load_golden(name)
    env = EmuBatch(g["actions"].shape[0], golden_params(g, precision=PRECISION_F64))
    report = {}
    worst = replay_golden(env, g, report=report, **TOL_F64)
    print(name, "worst rel err", worst, report)
    env.close()


@pytest.mark.parametrize("name", GOLDENS)
def test_emu_mixed_matches_reference_trace(name):
    g = load_golden(name)
    env = EmuBatch(g["actions"].shape[0], golden_params(g, precision=PRECISION_MIXED))
    report = {}
    worst = replay_golden(env, g, report=report, **TOL_MIXED_FREE_RUN)
    print(name, "worst rel err", worst, report)
    env.close()


def _pair(n, precision, g, seed=3, P=6):
    params = golden_params(g, precision=precision)
    prod = EmuBatch(n, params)
    orc = OracleVecEnv(n, params)
    t, o = sample_scene_pool(np.random.default_rng(seed), n, P)
    prod.set_scene_pool(t, o)
    orc.set_scene_pool(t, o)
    return prod, orc


@pytest.mark.parametrize("kind", ["uniform", "clipped"])
def test_emu_mixed_per_step_tolerance_vs_oracle(kind):
    """North-star tolerance: one env-step from identical state, fp32 kernel body vs float64
    oracle: counters/flags bit-exact, 1e-5 relative on the state channels."""
    g = load_golden("ref_random.npz")
    n, T = 64, 12
    prod, orc = _pair(n, PRECISION_MIXED, g)
    rng = np.random.default_rng(11)
    if kind == "uniform":
        acts = rng.uniform([0, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
    else:
        acts = np.clip(rng.normal(size=(T, n, 3)), [0, 0, -1], [1, 1, 1]).astype(np.float32)
    report = {}
    lockstep_compare(prod, orc, acts, resync=True, rtol=TOL_MIXED["rtol"], floor=TOL_MIXED["floor"], floors=MIXED_FLOORS, report=report)
    print(kind, report)


def test_emu_f64_lockstep_vs_oracle_with_autoreset():
    """Free-running with in-kernel auto-reset: reset indices and every counter stay identical."""
    g = load_golden("ref_random.npz")
    n, T = 48, 25
    prod, orc = _pair(n, PRECISION_F64, g)
    acts = np.random.default_rng(5).uniform([0, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
    hist = lockstep_compare(prod, orc, acts, resync=False, rtol=1e-9, floor=1e-6)
    worst = max(max(h.values()) for h in hist)
    assert worst < 1e-7, worst
    assert orc.get_state("episode_index").max() > 1     # some episodes did end and auto-reset


@pytest.mark.parametrize("precision", [PRECISION_F64, PRECISION_MIXED])
def test_emu_cuts_exactly_the_episodes_where_the_reference_raises(precision):
    worst = check_blowup_golden(lambda n, g: EmuBatch(n, golden_params(g, precision=precision)))
    assert worst < (1e-9 if precision == PRECISION_F64 else 1e-5), worst


def test_redundant_shape_updates_are_exact_noops():
    """The fused loop runs the shape update up to the warp-uniform end of the LAST lane's window, so
    a lane may see updates it does not need.  They must not change a single bit: the host build
    that updates after every substep equals the one that updates only inside the env's own
    windows, column for column (this is what makes results independent of warp composition,
    hence of sorting and sharding)."""
    from grasp_lab_salp_b200.batch import SalpBatch
    from grasp_lab_salp_b200.params import FIELDS
    n = 400
    a = SalpBatch(n, seed=3, _cdll=emu_cdll())
    b = SalpBatch(n, seed=3, _cdll=emu_lane_cdll())
    a.reset()
    b.reset()
    rng = np.random.default_rng(0)
    for t in range(5):
        act = rng.uniform([0, 0, -1], [1, 1, 1], size=(n, 3)).astype(np.float32)
        if t == 2:
            act = np.clip(rng.normal(size=(n, 3)), [0, 0, -1], [1, 1, 1]).astype(np.float32)
        a.step(act, auto_reset=True)
        b.step(act, auto_reset=True)
        for col in FIELDS:
            x, y = a.get_state(col), b.get_state(col)
            assert np.array_equal(x, y, equal_nan=True), (t, col)


def test_axisymmetric_form_equals_general_form():
    """The default parameters are axisymmetric (axes 1 and 2 carry the same coefficients); the loop
    then uses a form that shares their coefficient entries and drops identically-zero terms
    (SalpDerived.axisym).  Forcing the general form (SALP_STEP_GENERIC) must give the same bits.
    (Asymmetric parameters take the general form: test_non_default_robot_parameters.)"""
    from grasp_lab_salp_b200.params import FIELDS
    g = load_golden("ref_random.npz")
    n, T = 96, 10
    acts = np.random.default_rng(5).uniform([0, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
    a = EmuBatch(n, golden_params(g, precision=PRECISION_MIXED), seed=8)
    b = EmuBatch(n, golden_params(g, precision=PRECISION_MIXED), seed=8)
    np.testing.assert_array_equal(a.reset(), b.reset())
    for t in range(T):
        ra = a.step(acts[t], auto_reset=True)
        rb = b.step(acts[t], auto_reset=True, generic=True)
        for x, y in zip(ra, rb):
            np.testing.assert_array_equal(x, y)
        np.testing.assert_array_equal(a.terms, b.terms)
    for col in FIELDS:
        np.testing.assert_array_equal(a.get_state(col), b.get_state(col), err_msg=col)


@pytest.mark.parametrize("num_obstacles", [0, 1, 5, 8])
def test_other_obstacle_counts(num_obstacles):
    """Observation width 6 + 2 n, proximity penalty and collision over n obstacles (n = 0: no
    obstacle term at all, salp_robot_env.py:373-383)."""
    g = load_golden("ref_random.npz")
    n, T = 24, 6
    params = golden_params(g, precision=PRECISION_MIXED, num_obstacles=num_obstacles)
    prod, orc = EmuBatch(n, params, seed=7), OracleVecEnv(n, params, seed=7)
    assert prod.obs_dim == 6 + 2 * num_obstacles
    acts = np.random.default_rng(3).uniform([0, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
    lockstep_compare(prod, orc, acts, resync=True, rtol=TOL_MIXED["rtol"], floor=TOL_MIXED["floor"],
                     floors=MIXED_FLOORS, num_obstacles=num_obstacles)


def test_non_default_robot_parameters():
    """Nothing is hard-wired to make_env()'s literals: sea-water density, a heavier and longer body,
    another nozzle, other penalties, and every added-mass and drag family distinct per axis (the
    general form of the loop, roll and pitch driven at real amplitude) -- kernel body vs oracle,
    per-step tolerance with the floors measured for this set (ASYM_FLOORS)."""
    n, T = 48, 8
    for tumble in (False, True):
        for prec, tol in ((PRECISION_F64, dict(rtol=1e-9, floor=1e-3)),
                          (PRECISION_MIXED, dict(rtol=TOL_MIXED["rtol"], floor=TOL_MIXED["floor"],
                                                 floors=TUMBLING_FLOORS if tumble else ASYM_FLOORS))):
            p = asymmetric_params(prec)
            prod, orc = EmuBatch(n, p, seed=11), OracleVecEnv(n, p, seed=11)
            acts = np.random.default_rng(5).uniform([0.1, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
            report = {}
            lockstep_compare(prod, orc, acts, resync=True, report=report, inject=tumbling(n) if tumble else None, **tol)
            print(prec, "tumbling" if tumble else "free", report)
            assert np.abs(orc.get_state("angvel_x")).max() > 1e-4     # roll is driven, not rounding noise


def test_axisymmetric_form_predicate():
    """parity.axisym_broken restates make_derived's predicate: the defaults take the AXI form,
    asymmetric_params() breaks all eight conditions, each one_break() set exactly its own."""
    assert axisym_broken(golden_params(load_golden("ref_random.npz"))) == set()
    assert axisym_broken(asymmetric_params(PRECISION_MIXED)) == set(AXISYM_CONDITIONS)
    for name in AXISYM_CONDITIONS:
        assert axisym_broken(one_break(name)) == {name}
    # fp32 roundings, not the doubles: an axis-2 value one fp64 ulp off is still the AXI form
    p = golden_params(load_golden("ref_random.npz"))
    p.added_mass_force[2] = np.nextafter(p.added_mass_force[1], 1.0)
    assert axisym_broken(p) == set()


@pytest.mark.parametrize("tumble", [False, True], ids=["free", "tumbling"])
@pytest.mark.parametrize("name", AXISYM_CONDITIONS)
@pytest.mark.parametrize("precision", [PRECISION_F64, PRECISION_MIXED])
def test_one_broken_axisymmetry_condition(precision, name, tumble):
    """The defaults with one condition of the axisymmetric-form predicate broken: the general form
    of the loop against the oracle, per step, free and from a tumbling state (parity.tumbling)."""
    n, T = 48, 4
    p = one_break(name, precision)
    prod, orc = EmuBatch(n, p, seed=12), OracleVecEnv(n, p, seed=12)
    acts = np.random.default_rng(6).uniform([0, 0, -1], [1, 1, 1], size=(T, n, 3)).astype(np.float32)
    if precision == PRECISION_F64:
        tol = dict(rtol=1e-9, floor=1e-3)
    else:
        tol = dict(rtol=TOL_MIXED["rtol"], floor=TOL_MIXED["floor"], floors=TUMBLING_FLOORS if tumble else ASYM_FLOORS)
    report = {}
    lockstep_compare(prod, orc, acts, resync=True, report=report, inject=tumbling(n) if tumble else None, **tol)
    print(name, precision, report)


def test_masked_reset_and_zero_substep_cycles():
    g = load_golden("ref_random.npz")
    n = 16
    params = golden_params(g, precision=PRECISION_MIXED)
    prod, orc = EmuBatch(n, params, seed=2), OracleVecEnv(n, params, seed=2)
    prod.reset()
    orc.reset()
    a = np.tile(np.array([[0.5, 0.2, 0.3]], np.float32), (n, 1))
    a[::2] = [0.0, 0.0, 0.0]              # K = 0 cycles: nothing moves, total < 0 (SURVEY 8c edge KAT)
    for _ in range(3):
        prod.step(a)
        orc.step(a)
        np.testing.assert_array_equal(prod.substeps, orc.substeps)
        assert (prod.substeps[::2] == 0).all()
    mask = np.zeros(n, np.uint8)
    mask[[1, 4, 9]] = 1
    o1, o2 = prod.reset(mask).copy(), orc.reset(mask).copy()
    np.testing.assert_allclose(o1, o2, rtol=1e-6, atol=1e-6)
    for col in ("episode_index", "cycle", "ep_length"):
        np.testing.assert_array_equal(prod.get_state(col), orc.get_state(col))
    assert (prod.get_state("cycle")[[1, 4, 9]] == 0).all() and (prod.get_state("cycle")[[0, 2, 3]] == 3).all()
