"""predict, evaluate, save and load of PPO and RecurrentPPO (grasp_lab_salp_b200/ppo.py), the shared evaluation
loop (grasp_lab_salp_b200/evaluation.py) and salp_mlp_act's deterministic mode (csrc/salp_policy.cu).
CPU: evaluate against a host-loop restatement of sb3_contrib's evaluate_policy, predict against the policy's
own step, evaluation leaving training bit-identical, a save / load round trip, and two ranks over gloo.
GPU: the deterministic kernel against torch, the tensor-core predict against fp32 torch, and CUDA-graph runs
with evaluation and with a load into an object whose graphs are already captured."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from grasp_lab_salp_b200.ppo import PPO, HostEnv, PPOConfig, RecurrentPPO
from test_sac import _assert_eval_matches, _host_env

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TIMING = ("rollout_seconds", "update_seconds", "eval_seconds")
EVAL_KEYS = ("eval_return", "eval_success", "eval_length", "eval_seconds")


def _algo(recurrent, env, **kw):
    cfg = dict(n_steps=4, batch_size=8 if recurrent else 12, n_epochs=2, seed=3)
    cfg.update(kw)
    return (RecurrentPPO if recurrent else PPO)(env, PPOConfig(**cfg))


def _contrib_evaluate(model, env, n_episodes):
    """sb3_contrib-aware stable-baselines3 evaluate_policy(deterministic=True) restated as a host loop: env i
    contributes (n_episodes + i) // n episodes; the policy state returned by predict is carried, and
    episode_starts[i] is set to env i's done while env i still counts."""
    n = env.num_envs
    targets = [(n_episodes + i) // n for i in range(n)]
    counts = [0] * n
    rets, lens, succ = [], [], []
    cur_r, cur_l = [0.0] * n, [0] * n
    obs = env.reset_t()
    states, episode_starts = None, np.ones(n, dtype=bool)
    while any(c < t for c, t in zip(counts, targets)):
        actions, states = model.predict(obs, state=states, episode_start=episode_starts, deterministic=True)
        obs, rew, term, trunc, _ = env.step_t(actions)
        r = torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0).double().cpu()
        t, d = term.bool().cpu(), (term.bool() | trunc.bool()).cpu()
        for i in range(n):
            if counts[i] < targets[i]:
                cur_r[i] += r[i].item()
                cur_l[i] += 1
                episode_starts[i] = bool(d[i])
                if d[i]:
                    rets.append(cur_r[i])
                    lens.append(cur_l[i])
                    succ.append(float(t[i]))
                    counts[i] += 1
                    cur_r[i], cur_l[i] = 0.0, 0
    return dict(mean_return=sum(rets) / len(rets), mean_length=sum(lens) / len(rets),
                success_rate=sum(succ) / len(rets), episodes=len(rets))


def _params(algo):
    return [p.detach().clone() for p in algo.policy.parameters()]


def _assert_same_tensors(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def _assert_same_rows(rows0, rows1):
    """Equal history rows apart from timings and evaluation (NaN equals NaN: no episode ended)."""
    strip = lambda r: {k: v for k, v in r.items() if k not in TIMING and k not in EVAL_KEYS}  # noqa: E731
    assert len(rows0) == len(rows1)
    for r0, r1 in zip(rows0, rows1):
        r0, r1 = strip(r0), strip(r1)
        assert r0.keys() == r1.keys()
        for k in r0:
            assert r0[k] == r1[k] or (r0[k] != r0[k] and r1[k] != r1[k]), k


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("recurrent", [False, True])
def test_evaluate_matches_sb3_contrib_quota_restatement(recurrent):
    algo = _algo(recurrent, _host_env(4))
    algo.learn(4 * 4)                              # one iteration: weights away from their initial values
    ref = _contrib_evaluate(algo, _host_env(3, seed=9), 5)     # quotas 1, 2, 2
    ev = algo.evaluate(_host_env(3, seed=9), 5)
    assert ev["episodes"] == 5
    _assert_eval_matches(ev, ref)


def test_recurrent_predict_equals_policy_step_and_leaves_training_state():
    algo = _algo(True, _host_env(4))
    before = [x.clone() for x in algo.state]
    gen = algo.gen.get_state()
    torch.manual_seed(11)
    n = 5
    state = algo.policy.initial_state(n, "cpu")
    pstate = None
    starts = [torch.ones(n, dtype=torch.bool), torch.tensor([0, 1, 0, 0, 1], dtype=torch.bool),
              torch.zeros(n, dtype=torch.bool), torch.tensor([1, 0, 0, 1, 0], dtype=torch.bool)]
    with torch.no_grad():
        for st in starts:
            obs = torch.randn(n, algo.env.obs_dim)
            mean, _, state = algo.policy.step(obs, state, st)
            act, pstate = algo.predict(obs, state=pstate, episode_start=st, deterministic=True)
            assert torch.equal(act, torch.minimum(torch.maximum(mean, algo.low), algo.high))
            assert torch.equal(pstate[0], state[0]) and torch.equal(pstate[1], state[1])
        sampled, _ = algo.predict(obs, state=pstate, deterministic=False)
    assert not torch.equal(sampled, act)
    assert ((sampled >= algo.low) & (sampled <= algo.high)).all()
    for x, y in zip(before, algo.state):          # neither the rollout's actor nor its critic state moved
        assert torch.equal(x, y)
    assert torch.equal(gen, algo.gen.get_state())


def test_mlp_predict_is_the_clipped_actor_mean():
    algo = _algo(False, _host_env(4))
    algo.learn(4 * 4)
    gen = algo.gen.get_state()
    obs = torch.randn(7, algo.env.obs_dim) * 3
    act, state = algo.predict(obs, deterministic=True)
    with torch.no_grad():
        ref = torch.minimum(torch.maximum(algo.policy.actor(obs), algo.low), algo.high)
    assert state is None and torch.equal(act, ref)
    a1, _ = algo.predict(obs)
    a2, _ = algo.predict(obs)
    assert not torch.equal(a1, a2)                # predict's own stream moves on ...
    assert torch.equal(gen, algo.gen.get_state())   # ... and self.gen does not


@pytest.mark.parametrize("recurrent", [False, True])
def test_evaluation_does_not_disturb_training(recurrent):
    runs = []
    for with_eval in (False, True):
        algo = _algo(recurrent, _host_env(4))
        kw = dict(eval_env=_host_env(3, seed=9), eval_every=2 * 4 * 4, n_eval_episodes=3) if with_eval else {}
        stats = algo.learn(5 * 4 * 4, **kw)
        runs.append((stats.history, _params(algo), algo.gen.get_state(), algo._ret_stats.clone()))
    (h0, p0, g0, r0), (h1, p1, g1, r1) = runs
    assert [("eval_return" in r) for r in h1] == [False, True, False, True, False]
    assert not any("eval_return" in r for r in h0)
    assert all(0 <= r["eval_success"] <= 1 and r["eval_length"] >= 1 for r in h1 if "eval_return" in r)
    _assert_same_rows(h0, h1)
    _assert_same_tensors(p0, p1)
    assert torch.equal(g0, g1) and torch.equal(r0, r1)


def _opt_tensors(algo):
    out = []
    for st in algo.opt.state_dict()["state"].values():
        out += [st[k] for k in sorted(st)]
    return out


@pytest.mark.parametrize("recurrent", [False, True])
def test_save_load_round_trip(recurrent, tmp_path):
    a = _algo(recurrent, _host_env(4))
    a.learn(2 * 4 * 4)
    roll = a.collect()                            # a rollout both objects will update on
    path = tmp_path / "ckpt.pt"
    a.save(path)
    b = _algo(recurrent, _host_env(4, seed=6), seed=8)
    b.load(path)
    _assert_same_tensors(_params(a), _params(b))
    _assert_same_tensors(_opt_tensors(a), _opt_tensors(b))
    assert torch.equal(a._ret_stats, b._ret_stats) and torch.equal(a.gen.get_state(), b.gen.get_state())
    assert (a.env_steps, a.iteration) == (b.env_steps, b.iteration) == (3 * 4 * 4, 2)
    assert b._ep_len.abs().sum() == 0 and b._disc_ret.abs().sum() == 0
    if recurrent:
        assert all(x.abs().sum() == 0 for x in b.state) and bool(b.starts.all())
    a.update(roll)
    b.update(roll)
    _assert_same_tensors(_params(a), _params(b))
    b.learn(b.env_steps + 4 * 4)                  # and training goes on
    assert b.iteration == 3


def test_load_refuses_another_policy(tmp_path):
    path = tmp_path / "rppo.pt"
    _algo(True, _host_env(4)).save(path)
    with pytest.raises(ValueError):
        _algo(False, _host_env(4)).load(path)
    path = tmp_path / "ppo.pt"
    _algo(False, _host_env(4)).save(path)
    with pytest.raises(ValueError):
        _algo(False, _host_env(4), hidden=(32, 32)).load(path)
    with pytest.raises(ValueError):
        _algo(True, _host_env(4)).load(path)


EVAL_TOTAL, EVAL_EPISODES = 5, 7        # 3 + 2 envs on two ranks; quotas 1, 1, 1, 2, 2


def _worker(rank, world, port, path, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch
    from emu_backend import emu_cdll
    from grasp_lab_salp_b200.distributed import make_shard
    from grasp_lab_salp_b200.ppo import PPO, HostEnv, PPOConfig
    dist.init_process_group("gloo", rank=rank, world_size=world)
    shard = lambda total, seed: HostEnv(make_shard(total, seed=seed, device=0, _cdll=emu_cdll()))  # noqa: E731
    cfg = PPOConfig(n_steps=4, batch_size=8, n_epochs=2, seed=3)
    algo = PPO(shard(7, 2), cfg)
    ev = algo.evaluate(shard(EVAL_TOTAL, 9), EVAL_EPISODES)
    algo.learn(2 * 4 * 7)
    mine = (algo.gen.get_state().tolist(), algo._ret_stats.tolist())
    algo.save(path)
    fresh = PPO(shard(7, 2), cfg)
    differs = fresh.gen.get_state().tolist() != mine[0]
    fresh.load(path)
    restored = (fresh.gen.get_state().tolist(), fresh._ret_stats.tolist())
    gathered = [None] * world
    dist.gather_object((ev, mine, restored, differs), gathered if rank == 0 else None, dst=0)
    if rank == 0:
        out.put(gathered)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_evaluate_and_checkpoint(tmp_path):
    """PPO over gloo: the sharded evaluate (quotas by global env index, sums all-reduced) equals the
    single-process evaluate on the whole eval env on every rank, and a two-rank save / load gives every rank
    back its own exploration generator and reward-normalisation statistics."""
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29700 + os.getpid() % 90
    procs = [ctx.Process(target=_worker, args=(r, 2, port, str(tmp_path / "ckpt.pt"), out)) for r in range(2)]
    for p in procs:
        p.start()
    gathered = out.get(timeout=400)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    from emu_backend import EmuBatch
    whole = PPO(HostEnv(EmuBatch(7, seed=2)), PPOConfig(n_steps=4, batch_size=8, n_epochs=2, seed=3))
    ref = whole.evaluate(HostEnv(EmuBatch(EVAL_TOTAL, seed=9)), EVAL_EPISODES)
    assert ref["episodes"] == EVAL_EPISODES
    for ev, mine, restored, differs in gathered:
        for key in ("episodes", "mean_length", "success_rate"):
            assert ev[key] == ref[key], key
        assert ev["mean_return"] == pytest.approx(ref["mean_return"], rel=1e-9, abs=0)
        assert restored == mine and differs
    assert gathered[0][1] != gathered[1][1]        # the two ranks' entries are their own


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 5000])
@pytest.mark.parametrize("obs_dim", [10, 16])
def test_fused_mlp_deterministic_mode_matches_torch_mean(n, obs_dim):
    """salp_mlp_act with noise NULL: action = the actor mean, clipped = its Box clip (1e-5 against fp32
    torch); with value NULL the critic is skipped, with value given it is the critic's; logp NULL is not
    written.  The stochastic path keeps logp and value mandatory."""
    import ctypes as C
    from grasp_lab_salp_b200 import _lib
    from grasp_lab_salp_b200.ppo import MlpPolicy
    lib = _lib.load()
    torch.manual_seed(5 + n + obs_dim)
    pol = MlpPolicy(obs_dim, 3).cuda()
    with torch.no_grad():
        pol.actor[4].weight.mul_(30.0)            # means well outside the Box too
        pol.log_std.copy_(torch.tensor([-0.3, 0.1, 0.4]))
    obs = torch.randn(n, obs_dim, device="cuda") * 2
    packed = pol.packed()
    a, clipped = torch.full((n, 3), float("nan"), device="cuda"), torch.full((n, 3), float("nan"), device="cuda")
    v = torch.full((n,), float("nan"), device="cuda")
    lo, hi = (C.c_float * 3)(0.0, 0.0, -1.0), (C.c_float * 3)(1.0, 1.0, 1.0)
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.salp_mlp_act(p(packed), obs_dim, p(obs), None, n, lo, hi, p(a), p(clipped), None, None, stream) == 0
    torch.cuda.synchronize()
    with torch.no_grad():
        mean = pol.actor(obs)
        ref_c = torch.minimum(torch.maximum(mean, torch.tensor([0.0, 0.0, -1.0], device="cuda")),
                              torch.tensor([1.0, 1.0, 1.0], device="cuda"))
        ref_v = pol.value(obs)
    assert (a - mean).abs().max().item() < 1e-5
    assert (clipped - ref_c).abs().max().item() < 1e-5
    assert torch.equal(clipped, torch.minimum(torch.maximum(a, ref_c.new_tensor([0.0, 0.0, -1.0])),
                                              ref_c.new_tensor([1.0, 1.0, 1.0])))
    a2, c2 = torch.empty_like(a), torch.empty_like(a)
    assert lib.salp_mlp_act(p(packed), obs_dim, p(obs), None, n, lo, hi, p(a2), p(c2), None, p(v), stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(a2, a) and torch.equal(c2, clipped)
    assert (v - ref_v).abs().max().item() < 1e-5
    noise, logp = torch.zeros(n, 3, device="cuda"), torch.empty(n, device="cuda")
    assert lib.salp_mlp_act(p(packed), obs_dim, p(obs), p(noise), n, lo, hi, p(a), p(clipped), None, p(v), stream) != 0
    assert lib.salp_mlp_act(p(packed), obs_dim, p(obs), p(noise), n, lo, hi, p(a), p(clipped), p(logp), None, stream) != 0


@pytest.mark.gpu
def test_recurrent_predict_on_tensor_core_cell_tracks_torch():
    """RecurrentPPO.predict with the tcgen05 actor cell against the fp32 torch cell, over a few steps with
    resets, to the bf16 bar of the rollout test (2e-2); more envs than the training env has."""
    from grasp_lab_salp_b200 import SalpBatch, default_params
    from grasp_lab_salp_b200.ppo import DeviceEnv
    algos = [RecurrentPPO(DeviceEnv(SalpBatch(256, default_params(), seed=4)),
                          PPOConfig(n_steps=8, batch_size=8 * 256, seed=2, fused_policy=fused)) for fused in (True, False)]
    assert algos[0]._lstm_fused is not None and algos[1]._lstm_fused is None
    torch.manual_seed(0)
    n = 1000
    states = [None, None]
    for t in range(6):
        obs = torch.randn(n, algos[0].env.obs_dim, device="cuda")
        starts = torch.rand(n, device="cuda") < (1.0 if t == 0 else 0.2)
        acts = []
        for k, algo in enumerate(algos):
            a, states[k] = algo.predict(obs, state=states[k], episode_start=starts, deterministic=True)
            acts.append(a)
        assert (acts[0] - acts[1]).abs().max().item() < 2e-2
        assert (states[0][0] - states[1][0]).abs().max().item() < 2e-2
    algos[0]._eval_cell.check()


@pytest.mark.gpu
@pytest.mark.parametrize("recurrent", [False, True])
def test_cuda_graph_training_with_evaluation_and_load(recurrent, tmp_path):
    from grasp_lab_salp_b200 import SalpBatch, default_params
    from grasp_lab_salp_b200.ppo import DeviceEnv
    n, T = 1024, 8
    cfg = dict(n_steps=T, batch_size=T * 256, n_epochs=2, seed=1, cuda_graphs=True)
    it = T * n
    # evaluation between graph replays leaves the training bit-identical
    runs = []
    for with_eval in (False, True):
        algo = _algo(recurrent, DeviceEnv(SalpBatch(n, default_params(), seed=3)), **cfg)
        kw = dict(eval_env=DeviceEnv(SalpBatch(256, default_params(), seed=9)), eval_every=2 * it,
                  n_eval_episodes=256) if with_eval else {}
        stats = algo.learn(6 * it, **kw)
        torch.cuda.synchronize()
        assert algo._roll_graph is not None and algo._upd_graph is not None
        runs.append((stats.history, _params(algo), algo.gen.get_state()))
    (h0, p0, g0), (h1, p1, g1) = runs
    assert sum("eval_return" in r for r in h1) == 3
    _assert_same_rows(h0, h1)
    _assert_same_tensors(p0, p1)
    assert torch.equal(g0, g1)
    # a load into an object whose graphs are captured restores what a fresh object's load restores, and both
    # then update identically on one rollout, through a newly captured minibatch graph
    path = tmp_path / "ckpt.pt"
    algo.save(path)
    roll = algo.collect()
    captured = _algo(recurrent, DeviceEnv(SalpBatch(n, default_params(), seed=5)), **cfg)
    captured.learn(3 * it)
    assert captured._roll_graph is not None and captured._upd_graph is not None
    captured.load(path)
    assert captured._roll_graph is None and captured._upd_graph is None
    fresh = _algo(recurrent, DeviceEnv(SalpBatch(n, default_params(), seed=6)), **dict(cfg, seed=7))
    fresh.load(path)
    torch.cuda.synchronize()
    _assert_same_tensors(_params(captured), _params(fresh))
    _assert_same_tensors(_opt_tensors(captured), _opt_tensors(fresh))
    assert torch.equal(captured.gen.get_state(), fresh.gen.get_state())
    assert torch.equal(captured._ret_stats, fresh._ret_stats)
    assert (captured.env_steps, captured.iteration) == (fresh.env_steps, fresh.iteration)
    for x in (captured, fresh):
        x.update(roll)
    torch.cuda.synchronize()
    assert captured._upd_graph is not None and fresh._upd_graph is not None
    _assert_same_tensors(_params(captured), _params(fresh))
    assert torch.equal(captured.gen.get_state(), fresh.gen.get_state())
    evs = [x.evaluate(DeviceEnv(SalpBatch(128, default_params(), seed=9)), 128) for x in (captured, fresh)]
    assert evs[0] == evs[1]
    for x in (captured, fresh):                   # and training goes on, the rollout graph captured anew
        x.learn(x.env_steps_global + 2 * it)
        assert x._roll_graph is not None
