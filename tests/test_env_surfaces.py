"""The reference-facing surfaces: gymnasium-style SalpRobotEnv and the SB3-VecEnv-shaped
SalpCudaVecEnv.  CPU variants run on the host build of the kernel body (tests/emu); the GPU
variants (marked gpu) run the same checks on the CUDA library."""
import os

import numpy as np
import pytest

from grasp_lab_salp_b200 import PRECISION_F64, Nozzle, Robot, SalpCudaVecEnv, SalpRobotEnv
from oracle.salp_oracle import OracleVecEnv
from parity import golden_params, load_golden

REWARD_KEYS = ["rewards/track", "rewards/heading", "rewards/smooth", "rewards/yaw", "rewards/time",
               "rewards/sideslip", "rewards/obstacle"]


def _cdll(use_gpu):
    if use_gpu:
        return None
    from emu_backend import emu_cdll
    return emu_cdll()


def make_env(cdll):
    """Verbatim body of the reference's make_env() (src/train_robot.py:11-21) on the stand-in classes."""
    nozzle = Nozzle(length1=0.05, length2=0.05, length3=0.05, area=0.00016, mass=1.0)
    robot = Robot(dry_mass=1.0, init_length=0.3, init_width=0.15, max_contraction=0.06, nozzle=nozzle)
    robot.nozzle.set_angles(angle1=0.0, angle2=0.0)
    robot.set_environment(density=1000)
    env = SalpRobotEnv(render_mode=None, robot=robot, precision=PRECISION_F64, _cdll=cdll)
    return env


def _single_env_replays_reference_trace(cdll):
    g = load_golden("ref_fixed10.npz")
    env = make_env(cdll)
    assert env.action_space.shape == (3,) and env.observation_space.shape == (10,)
    env.set_scene(g["targets"][0, 0], g["obstacles"][0, 0])
    obs, info = env.reset(seed=0)
    assert info == {} and obs.dtype == np.float32
    np.testing.assert_allclose(obs, g["first_obs"][0], rtol=1e-6, atol=1e-7)
    np.testing.assert_array_equal(env.target_point, g["targets"][0, 0])
    for t in range(g["actions"].shape[1]):
        obs, rew, done, trunc, info = env.step(g["actions"][0, t])
        assert isinstance(rew, float) and isinstance(done, bool) and isinstance(trunc, bool)
        np.testing.assert_allclose(obs, g["obs"][0, t], rtol=2e-6, atol=1e-6)
        assert rew == pytest.approx(g["reward"][0, t], rel=1e-8, abs=1e-8)
        assert done == bool(g["terminated"][0, t]) and trunc == bool(g["truncated"][0, t])
        for j, k in enumerate(REWARD_KEYS):
            assert info[k] == pytest.approx(g["terms"][0, t, j], rel=1e-8, abs=1e-9)
        assert info["position_history"] == [] and env.robot.cycle == g["cycle"][0, t]
        np.testing.assert_allclose(env.robot.position_world[:2], g["state"][0, t, :2], rtol=1e-9, atol=1e-12)
        if done or trunc:
            env.reset()
    env.close()


def _vec_env_has_sb3_semantics(cdll, n=24, T=40):
    g = load_golden("ref_random.npz")
    params = golden_params(g, precision=PRECISION_F64)
    venv = SalpCudaVecEnv(n, params, seed=3, info_mode="full", _cdll=cdll)
    orc = OracleVecEnv(n, params, seed=3)
    obs = venv.reset()
    np.testing.assert_allclose(obs, orc.reset(), rtol=1e-6, atol=1e-7)
    assert obs.shape == (n, 10) and obs.dtype == np.float32 and len(venv.reset_infos) == n
    assert venv.env_is_wrapped(object) == [False] * n and venv.get_attr("render_mode") == [None] * n
    rng = np.random.default_rng(0)
    returns = np.zeros(n)
    lengths = np.zeros(n, int)
    episodes = 0
    for t in range(T):
        a = rng.uniform([0, 0, -1], [1, 1, 1], size=(n, 3)).astype(np.float32)
        venv.step_async(a)
        obs, rew, dones, infos = venv.step_wait()
        o_obs, o_rew, o_term, o_trunc = orc.step(a, auto_reset=True)
        assert rew.dtype == np.float32 and dones.dtype == bool and len(infos) == n
        np.testing.assert_array_equal(dones, (o_term | o_trunc).astype(bool))
        np.testing.assert_allclose(obs, o_obs, rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(rew, o_rew.astype(np.float32), rtol=1e-5, atol=1e-4)
        returns += o_rew
        lengths += 1
        for i in range(n):
            info = infos[i]
            assert set(REWARD_KEYS) <= set(info)
            if dones[i]:
                episodes += 1
                np.testing.assert_allclose(info["terminal_observation"], orc.terminal_obs[i], rtol=1e-5, atol=1e-6)
                assert info["TimeLimit.truncated"] == bool(o_trunc[i] and not o_term[i])
                assert info["episode"]["l"] == lengths[i]
                assert info["episode"]["r"] == pytest.approx(returns[i], rel=1e-6, abs=1e-6)
                assert info["path_length"] == pytest.approx(orc.metrics[i, 2], rel=1e-6, abs=1e-9)
                assert info["final_distance"] == pytest.approx(orc.metrics[i, 5], rel=1e-6, abs=1e-9)
                returns[i] = 0.0
                lengths[i] = 0
            else:
                assert "terminal_observation" not in info and "episode" not in info
    assert episodes > 0
    # lazy infos: unfinished envs share one empty dict
    lazy = SalpCudaVecEnv(8, params, seed=3, info_mode="lazy", _cdll=cdll)
    lazy.reset()
    _, _, d, infos = lazy.step(np.tile(np.array([[0.5, 0.1, 0.2]], np.float32), (8, 1)))
    assert all((infos[i] == {}) for i in range(8) if not d[i])
    with pytest.raises(ValueError):
        lazy.step_async(np.zeros((3, 3), np.float32))
    venv.close()
    lazy.close()


def test_single_env_replays_reference_trace_emu():
    _single_env_replays_reference_trace(_cdll(False))


def test_vec_env_has_sb3_semantics_emu():
    _vec_env_has_sb3_semantics(_cdll(False))


@pytest.mark.gpu
def test_single_env_replays_reference_trace_gpu():
    _single_env_replays_reference_trace(_cdll(True))


@pytest.mark.gpu
def test_vec_env_has_sb3_semantics_gpu():
    _vec_env_has_sb3_semantics(_cdll(True), n=256, T=40)


def _history_feed(cdll):
    """record=True: info carries the per-substep histories of the cycle (robot.py:681-776); the
    last row is the state the step leaves behind, the row count is K, and tracing does not
    advance the env."""
    g = load_golden("ref_fixed10.npz")
    env = make_env(cdll)
    env.enable_history_recording()
    env.set_scene(g["targets"][0, 0], g["obstacles"][0, 0])
    env.reset()
    for t in range(4):
        a = g["actions"][0, t]
        before = env.robot.position_world.copy()
        h = env._batch.trace_cycle(0, a)
        np.testing.assert_array_equal(env.robot.position_world, before)          # not advanced
        obs, rew, done, trunc, info = env.step(a)
        K = int(g["K"][0, t])
        assert h["substeps"] == K and info["position_history"].shape == (K, 3)
        assert info["length_history"].shape == (K,) and info["width_history"].shape == (K,)
        np.testing.assert_allclose(info["position_history"][-1], env.robot.position_world, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(info["position_history"][-1][:2], g["state"][0, t, :2], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(env.last_history["euler_angle"][-1], env.robot.euler_angle, rtol=1e-12, atol=1e-15)
        assert info["length_history"].min() >= 0.3 - 0.06 * a[0] - 1e-6 and abs(info["length_history"][-1] - 0.3) < 1e-12
        np.testing.assert_allclose(info["length_history"] + info["width_history"], 0.45, rtol=1e-12)
    env.close()


def test_history_feed_emu():
    _history_feed(_cdll(False))


@pytest.mark.gpu
def test_history_feed_gpu():
    _history_feed(_cdll(True))


# ---------------------------------------------------------------------------------------------
# The reference's own consumer of `info`: DetailedMetricsCallback (src/tensorboard_callback.py)
# ---------------------------------------------------------------------------------------------
def _load_reference_callback():
    """The UNMODIFIED DetailedMetricsCallback, imported from the reference sources with a dummy
    `stable_baselines3.common.callbacks.BaseCallback` (SB3 is not installed in this image)."""
    import importlib.util
    import sys
    import types
    from oracle import ref_harness
    d = ref_harness.reference_dir()
    path = None if d is None else os.path.join(d, "tensorboard_callback.py")
    if path is None or not os.path.isfile(path):
        pytest.skip("reference tensorboard_callback.py not available (tools/stage_reference.py)")

    class BaseCallback:               # the part of SB3's BaseCallback that the reference callback touches
        def __init__(self, verbose=0):
            self.verbose = verbose
            self.n_calls = 0
            self.locals = {}
            self.records = {}
            self.logger = types.SimpleNamespace(record=lambda k, v: self.records.__setitem__(k, v))

        def on_step(self):
            self.n_calls += 1
            return self._on_step()

    names = ["stable_baselines3", "stable_baselines3.common", "stable_baselines3.common.callbacks"]
    saved = {k: sys.modules.get(k) for k in names}
    try:
        for k in names:
            sys.modules[k] = types.ModuleType(k)
        sys.modules[names[2]].BaseCallback = BaseCallback
        spec = importlib.util.spec_from_file_location("salp_ref_tensorboard_callback", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod.DetailedMetricsCallback


EPISODE_KEYS = ("r", "l", "success", "truncated", "path_length", "direct_distance", "path_efficiency",
                "final_distance", "initial_distance", "avg_compression", "avg_coast_time", "avg_nozzle_angle",
                "avg_velocity")


def _replay_reference_episodes(cdll, on_step):
    """Drives SalpCudaVecEnv with the actions and scenes of a golden trace of the live reference
    (ref_random.npz), calls on_step(infos, dones) after every step, and returns, in order of episode
    end, what the reference's own env + SB3 Monitor hand out there (recomputed from the golden file):
    Monitor r / l, success / truncation, and the nine navigation / action / velocity metrics of
    salp_robot_env.py:399-447, as {key: [values]} over EPISODE_KEYS."""
    g = load_golden("ref_random.npz")
    acts = g["actions"]
    n, T, _ = acts.shape
    venv = SalpCudaVecEnv(n, golden_params(g, precision=PRECISION_F64), seed=0, info_mode="lazy", _cdll=cdll)
    venv.batch.set_scene_pool(g["targets"], g["obstacles"])
    venv.reset()
    keys = [str(k) for k in g["metric_keys"]]
    want = {k: [] for k in EPISODE_KEYS}
    ret = np.zeros(n)
    length = np.zeros(n, int)
    for t in range(T):
        obs, rew, dones, infos = venv.step(acts[:, t])
        on_step(infos, dones)
        ret += g["reward"][:, t]
        length += 1
        ended = (g["terminated"][:, t] | g["truncated"][:, t]).astype(bool)
        np.testing.assert_array_equal(dones, ended)
        for i in np.flatnonzero(ended):
            want["r"].append(ret[i])
            want["l"].append(length[i])
            tl_trunc = bool(g["truncated"][i, t]) and not bool(g["terminated"][i, t])      # SB3's TimeLimit.truncated
            want["success"].append(0.0 if tl_trunc else 1.0)
            want["truncated"].append(1.0 if tl_trunc else 0.0)
            for k in list(want)[4:]:
                want[k].append(g["metrics"][i, t, keys.index(k)])
            ret[i] = 0.0
            length[i] = 0
    venv.close()
    assert len(want["r"]) >= 20            # the trace does end episodes
    return want


def _assert_episode_values(got, want, rel):
    for k, w in want.items():
        # (the reference averages its float32 action lists in float32, salp_robot_env.py:420-427)
        tol = 1e-6 if k in ("avg_compression", "avg_coast_time", "avg_nozzle_angle") else rel
        np.testing.assert_allclose(np.array(list(got[k]), float), np.array(w, float), rtol=tol, atol=tol, err_msg=k)


def _reference_callback_reads_what_the_reference_env_would_give(cdll, rel):
    """Feeds every step's (infos, dones) of _replay_reference_episodes to the reference's
    DetailedMetricsCallback._on_step; what the callback collected must be what the reference's own
    env + SB3 Monitor would have handed it.  The callback's reward-component deques stay empty, as
    they do with the reference: it looks for `avg_r_track` while the env emits `avg_rewards_track`
    (tensorboard_callback.py:114-123 vs salp_robot_env.py:441-445)."""
    Callback = _load_reference_callback()
    T = load_golden("ref_random.npz")["actions"].shape[1]
    cb = Callback(log_freq=T)

    def on_step(infos, dones):
        cb.locals = {"infos": infos, "dones": dones}
        assert cb.on_step() is True

    want = _replay_reference_episodes(cdll, on_step)
    got = {"r": cb.episode_rewards, "l": cb.episode_lengths, "success": cb.episode_successes,
           "truncated": cb.episode_truncations, "path_length": cb.episode_path_lengths,
           "direct_distance": cb.episode_direct_distances, "path_efficiency": cb.episode_efficiencies,
           "final_distance": cb.episode_final_distances, "initial_distance": cb.episode_initial_distances,
           "avg_compression": cb.episode_compressions, "avg_coast_time": cb.episode_coast_times,
           "avg_nozzle_angle": cb.episode_nozzle_angles, "avg_velocity": cb.episode_velocities}
    _assert_episode_values(got, want, rel)
    assert len(cb.episode_r_tracks) == 0 and len(cb.episode_r_smooths) == 0
    # the aggregated TensorBoard scalars are logged from those deques (log_freq = T)
    assert cb.records["custom/navigation/success_rate"] == pytest.approx(np.mean(want["success"]))
    assert cb.records["custom/path/efficiency"] == pytest.approx(np.mean(want["path_efficiency"]), rel=rel)
    assert cb.records["reward/stats/total_mean"] == pytest.approx(np.mean(want["r"]), rel=rel)


def _episode_infos_match_reference_trace(cdll, rel):
    """What a metrics callback reads at each episode end, taken from the infos directly: Monitor r / l,
    TimeLimit.truncated and the nine metrics must be what the reference handed out in its golden trace.
    Needs nothing outside the repository, unlike the check through the reference's own callback."""
    got = {k: [] for k in EPISODE_KEYS}

    def on_step(infos, dones):
        for i in np.flatnonzero(dones):
            info = infos[i]
            got["r"].append(info["episode"]["r"])
            got["l"].append(info["episode"]["l"])
            got["success"].append(0.0 if info["TimeLimit.truncated"] else 1.0)
            got["truncated"].append(1.0 if info["TimeLimit.truncated"] else 0.0)
            for k in EPISODE_KEYS[4:]:
                got[k].append(info[k])

    _assert_episode_values(got, _replay_reference_episodes(cdll, on_step), rel)


def test_episode_infos_match_reference_trace_cpu():
    _episode_infos_match_reference_trace(_cdll(False), 1e-8)


@pytest.mark.gpu
def test_episode_infos_match_reference_trace_gpu():
    _episode_infos_match_reference_trace(_cdll(True), 1e-8)


def test_reference_metrics_callback_on_the_vec_env_cpu():
    _reference_callback_reads_what_the_reference_env_would_give(_cdll(False), 1e-8)


@pytest.mark.gpu
def test_reference_metrics_callback_on_the_vec_env_gpu():
    _reference_callback_reads_what_the_reference_env_would_give(_cdll(True), 1e-8)


def _set_attr_and_env_method(cdll):
    venv = SalpCudaVecEnv(6, seed=1, info_mode="lazy", _cdll=cdll)
    venv.reset()
    venv.set_attr("target_point", np.array([1.25, -0.5], np.float32), indices=[1, 4])
    tp = venv.get_attr("target_point")
    np.testing.assert_array_equal(tp[1], [1.25, -0.5])
    np.testing.assert_array_equal(tp[4], [1.25, -0.5])
    assert not np.array_equal(tp[0], tp[1])
    venv.set_attr("my_tag", "x", indices=2)
    assert venv.get_attr("my_tag", indices=[2, 3]) == ["x", None]
    out = venv.env_method("reset", indices=[0, 5])
    assert len(out) == 2 and out[0][0].shape == (10,) and out[0][1] == {}
    with pytest.raises(AttributeError):
        venv.env_method("no_such_method")
    venv.close()


def test_set_attr_and_env_method_cpu():
    _set_attr_and_env_method(_cdll(False))
