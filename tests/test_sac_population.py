"""A population of SAC agents trained side by side (grasp_lab_salp_b200/sac_population.py) and the grouped
rollout actor kernel (salp_sac_act_grouped, csrc/salp_sac.cu).  CPU: initialisation, per-agent gradient steps
against the stable-baselines3 restatement of test_sac.py, per-agent replay, one agent collecting as SAC does,
per-agent evaluation against test_sac.py's evaluate_policy restatement, a short learn() on the host build of
the kernel body, argument checks, save_agent.  GPU: the grouped kernel against salp_sac_act, a
K n-env batch against K separate batches, CUDA-graph equivalence, learning."""
import ctypes as C
import time

import pytest
import torch

from grasp_lab_salp_b200 import _lib
from grasp_lab_salp_b200.sac import SAC, SacActor, SacActorB200, SacActorGroupB200, SACConfig, SacCritic
from grasp_lab_salp_b200.sac_population import SACPopulation
from test_sac import _assert_eval_matches, _host_env, _sb3_evaluate, _sb3_train_step, _TaggedEnv


def _agent_modules(pop, k):
    """Agent k's actor, critic and target as nn.Modules (copies)."""
    D = pop.obs_dim
    mods = (SacActor(D), SacCritic(D), SacCritic(D))
    for m, params in zip(mods, (pop.actor_params, pop.critic_params, pop.target_params)):
        with torch.no_grad():
            for q, p in zip(m.parameters(), params):
                q.copy_(p[k])
    return mods


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def test_initial_networks_match_standalone_sac():
    seeds = [3, 11, 0]
    pop = SACPopulation(_TaggedEnv(n=3 * 2, obs_dim=6), [SACConfig(seed=s) for s in seeds])
    assert pop.num_agents == 3 and pop.n_envs == 2 and pop.slots == 100_000 // 2
    for k, s in enumerate(seeds):
        sac = SAC(_TaggedEnv(n=2, obs_dim=6), SACConfig(seed=s))
        for mine, theirs in ((pop.actor_params, sac.actor), (pop.critic_params, sac.critic),
                             (pop.target_params, sac.critic_target)):
            ps = list(theirs.parameters())
            assert len(ps) == len(mine)
            for a, b in zip(mine, ps):
                assert torch.equal(a[k], b)


@pytest.mark.parametrize("ent_coef", ["auto", "float"])
def test_gradient_steps_match_sb3_restatement_per_agent(ent_coef):
    K, B, D = 3, 64, 6
    lrs, gammas, taus, tents = [3e-4, 1e-4, 3e-4], [0.99, 0.95, 0.99], [0.005, 0.02, 0.005], [-3.0, -1.5, -3.0]
    ents = ["auto"] * K if ent_coef == "auto" else [0.2, 0.05, 0.2]
    seeds = [7, 8, 7]                           # agents 0 and 2: same settings and seed, different batches
    cfgs = [SACConfig(seed=seeds[k], learning_rate=lrs[k], gamma=gammas[k], tau=taus[k], target_entropy=tents[k],
                      ent_coef=ents[k]) for k in range(K)]
    pop = SACPopulation(_TaggedEnv(n=K * 2, obs_dim=D), cfgs)
    torch.manual_seed(1)
    batch = dict(obs=torch.randn(K, B, D), actions=torch.rand(K, B, 3) * 2 - 1, next_obs=torch.randn(K, B, D),
                 rewards=torch.randn(K, B, 1) * 10, dones=(torch.rand(K, B, 1) < 0.2).float())
    eps = (torch.randn(K, B, 3), torch.randn(K, B, 3))
    refs = []
    for k in range(K):
        actor, critic, target = _agent_modules(pop, k)
        log_ent = torch.zeros(1, requires_grad=True) if ent_coef == "auto" else None
        opts = [torch.optim.Adam(actor.parameters(), lr=lrs[k]), torch.optim.Adam(critic.parameters(), lr=lrs[k]),
                None if log_ent is None else torch.optim.Adam([log_ent], lr=lrs[k])]
        ent_t = None if log_ent is not None else torch.tensor(float(ents[k]))
        refs.append((actor, critic, target, log_ent, ent_t, opts))
    was_noise = {}
    for step in (1, 2, 3):
        out = pop.train_step(batch, eps)
        for k, (actor, critic, target, log_ent, ent_t, opts) in enumerate(refs):
            bk = {key: v[k] for key, v in batch.items()}
            ref = _sb3_train_step(actor, critic, target, log_ent, ent_t, opts, bk, (eps[0][k], eps[1][k]),
                                  gammas[k], taus[k], tents[k])
            # batched GEMMs sum in another order than F.linear: 1e-6 relative to max(1, |loss|) (a critic loss
            # near 100 has an fp32 ulp of 7.6e-6); parameters and log_ent_coef to 1e-6 absolute
            for mine, theirs in ((out["critic_loss"][k], ref[0]), (out["actor_loss"][k], ref[1]),
                                 (out["ent_coef_loss"][k] if log_ent is not None else None, ref[2])):
                if theirs is not None:
                    assert abs(mine.item() - theirs.item()) < 1e-6 * max(1.0, abs(theirs.item()))
            if log_ent is not None:
                assert abs(pop.log_ent_coef[k].item() - log_ent.item()) < 1e-6
                assert pop.log_ent_coef[k].item() != 0.0
            # parameters to 1e-6, except where a gradient has been rounding noise below Adam's eps (RMS < 1e-7):
            # there Adam turns a last-bit difference of the gradient into a sizeable fraction of an lr step
            # (measured: at most 0.016 lr per step; bar 0.05)
            for mine, theirs, opt in zip(_agent_modules(pop, k), (actor, critic, target), (opts[0], opts[1], opts[1])):
                for (name, a), b, q in zip(mine.named_parameters(), theirs.parameters(), opt.param_groups[0]["params"]):
                    noise = (opt.state[q]["exp_avg_sq"] / (1 - 0.999 ** step)).sqrt() < 1e-7
                    noise = was_noise[k, name] = noise | was_noise.get((k, name), noise)
                    assert ((a - b).abs() < 1e-6)[~noise].all(), (k, name)
                    assert ((a - b).abs() < 0.05 * lrs[k] * step)[noise].all(), (k, name)
    assert not torch.equal(pop.actor_params[0][0], pop.actor_params[0][2])
    assert not torch.equal(pop.critic_params[2][0], pop.critic_params[2][2])


def test_replay_is_per_agent_on_a_wrapping_ring():
    K, n = 3, 2
    env = _TaggedEnv(n=K * n, obs_dim=6)
    pop = SACPopulation(env, [SACConfig(buffer_size=n * 4, learning_starts=1000, seed=s) for s in range(K)])
    assert pop.slots == 4 and not pop.zero_copy
    for _ in range(11):
        pop._vec_step()
    assert pop.full and pop.pos == 11 % 4 and pop.num_timesteps == 11 * n
    s = pop.sample(3000)
    assert s["obs"].shape == (K, 3000, 6) and s["rewards"].shape == (K, 3000, 1)
    assert not (s["slot"] == pop.pos).any()
    assert set(s["slot"].flatten().tolist()) == {0, 1, 2}
    for k in range(K):
        tags = s["obs"][k, :, 0]                 # the env index each transition came from
        assert set(tags.tolist()) == set(range(k * n, (k + 1) * n))
        assert torch.equal(tags, s["env"][k].float())
        assert torch.equal(s["next_obs"][k, :, 0], tags)
    t_obs, t_next = s["obs"][..., 1], s["next_obs"][..., 1]
    assert ((t_obs == t_next - 1) | (t_obs == -1)).all()


def test_one_agent_collects_like_sac():
    """A population of one collects, keeps episode statistics and samples exactly as SAC does."""
    cfg = SACConfig(buffer_size=3 * 4, learning_starts=1000, seed=1)
    sac, pop = SAC(_TaggedEnv(n=3, obs_dim=6), cfg), SACPopulation(_TaggedEnv(n=3, obs_dim=6), [cfg])
    for _ in range(11):                          # wraps the 4-slot ring
        sac._vec_step()
        pop._vec_step()
    for key in sac.rb:
        assert torch.equal(sac.rb[key], pop.rb[key]), key
    assert (sac.pos, sac.full, sac.num_timesteps) == (pop.pos, pop.full, pop.num_timesteps) == (3, True, 33)
    assert torch.equal(sac._ep, pop._ep) and pop._ep[0, 3].item() == 3
    mine, theirs = pop.sample(500), sac.sample(500)
    for key in theirs:
        assert torch.equal(mine[key][0], theirs[key]), key


def test_evaluate_matches_sb3_quota_restatement_per_agent():
    pop = SACPopulation(_host_env(2 * 2), [SACConfig(seed=3), SACConfig(seed=4)])
    refs = _sb3_evaluate(pop.predict, _host_env(2 * 3, seed=9), 5, agents=2)    # quotas 1, 2, 2 per agent
    ev = pop.evaluate(_host_env(2 * 3, seed=9), 5)
    assert ev["episodes"] == [5, 5] and refs[0] != refs[1]
    for k, ref in enumerate(refs):
        _assert_eval_matches({key: v[k] for key, v in ev.items()}, ref)


def test_short_learn_on_the_kernel_body():
    env = _host_env(2 * 4, seed=4)
    pop = SACPopulation(env, [SACConfig(learning_starts=32, batch_size=16, buffer_size=400, seed=s) for s in (3, 4)])
    rows = pop.learn(4 * 20, log_interval=40)
    assert pop.gradient_steps_done == 20 - 8
    assert len(rows) == 2 and rows[-1]["env_steps"] == 80
    assert set(rows[-1]) == {"env_steps", "gradient_steps", "ent_coef", "critic_loss", "actor_loss", "mean_q",
                             "episodes", "mean_episode_return", "mean_episode_length", "success_rate",
                             "collect_seconds", "train_seconds"}
    for key in ("ent_coef", "critic_loss", "actor_loss", "mean_q", "episodes", "success_rate"):
        assert len(rows[-1][key]) == 2, key
    assert all(torch.isfinite(torch.tensor(rows[-1]["critic_loss"])))
    assert rows[-1]["critic_loss"][0] != rows[-1]["critic_loss"][1]
    ev = pop.evaluate(_host_env(2 * 2, seed=9), n_episodes=2)
    assert ev["episodes"] == [2, 2] and len(ev["success_rate"]) == 2


def test_rejects_bad_input():
    env = _TaggedEnv(n=6, obs_dim=6)
    with pytest.raises(ValueError, match="batch_size"):
        SACPopulation(env, [SACConfig(batch_size=256), SACConfig(batch_size=128)])
    with pytest.raises(ValueError, match="action_low"):
        SACPopulation(env, [SACConfig(), SACConfig(action_low=(0.0, 0.0, 0.0))])
    with pytest.raises(ValueError, match="ent_coef"):
        SACPopulation(env, [SACConfig(ent_coef="auto"), SACConfig(ent_coef=0.1)])
    with pytest.raises(ValueError, match="multiple"):
        SACPopulation(_TaggedEnv(n=5, obs_dim=6), [SACConfig(seed=0), SACConfig(seed=1)])
    lib = _lib.load()
    lo, hi = (C.c_float * 3)(0, 0, -1), (C.c_float * 3)(1, 1, 1)
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    odd = C.c_void_p(p.value + 4)
    assert lib.salp_sac_pack_weights_grouped(*([None] * 8), 2, 10, None, None) == _lib.ERR_INVALID
    for k, d, dst in ((0, 10, p), (2, 0, p), (2, 65, p), (2, 10, odd)):
        assert lib.salp_sac_pack_weights_grouped(*([p] * 8), k, d, dst, None) == _lib.ERR_INVALID
    args = dict(packed=p, k=2, d=10, obs=p, noise=None, n=8, lo=lo, hi=hi, env=p, scaled=p)
    for bad in (dict(k=0), dict(n=0), dict(d=0), dict(d=65), dict(packed=odd), dict(packed=None), dict(obs=None),
                dict(lo=None), dict(hi=None), dict(env=None), dict(scaled=None)):
        a = dict(args, **bad)
        assert lib.salp_sac_act_grouped(a["packed"], a["k"], a["d"], a["obs"], a["noise"], a["n"], a["lo"], a["hi"],
                                        a["env"], a["scaled"], None) == _lib.ERR_INVALID, bad
    with pytest.raises(RuntimeError, match="no CPU path"):
        SacActorGroupB200([q.detach().unsqueeze(0) for q in SacActor(10).parameters()], (0, 0, -1), (1, 1, 1))


def test_save_agent_loads_into_sac(tmp_path):
    K = 2
    env = _TaggedEnv(n=K * 4, obs_dim=6)
    pop = SACPopulation(env, [SACConfig(learning_starts=8, batch_size=16, seed=5, learning_rate=lr)
                              for lr in (3e-4, 1e-3)])
    pop.learn(40)
    trained = SAC(_TaggedEnv(n=4, obs_dim=6), SACConfig(learning_starts=8, batch_size=16, seed=5))
    trained.learn(40)
    ref_path = tmp_path / "sac.pt"
    trained.save(ref_path)
    obs = torch.randn(K * 10, 6)
    a = pop.predict(obs, deterministic=True)
    for k in range(K):
        path = tmp_path / f"agent{k}.pt"
        pop.save_agent(k, path)
        sac = SAC(_TaggedEnv(n=4, obs_dim=6), pop.configs[k])
        assert not torch.equal(sac.predict(obs[k * 10:(k + 1) * 10]), a[k * 10:(k + 1) * 10])
        sac.load(path)
        assert torch.equal(sac.predict(obs[k * 10:(k + 1) * 10]), a[k * 10:(k + 1) * 10])
        for mine, theirs in zip(_agent_modules(pop, k), (sac.actor, sac.critic, sac.critic_target)):
            for x, y in zip(mine.parameters(), theirs.parameters()):
                assert torch.equal(x, y)
        assert sac.log_ent_coef.item() == pop.log_ent_coef[k].item() and sac.num_timesteps == 40
        assert sac.actor_opt.param_groups[0]["lr"] == pop.configs[k].learning_rate
        st = sac.critic_opt.state[sac.critic.q_networks[0][0].weight]
        assert torch.equal(st["exp_avg"], pop.critic_opt.exp_avg[0][k])
        assert float(st["step"]) == float(pop.critic_opt.step_t) > 0
        assert torch.equal(sac.ent_opt.state[sac.log_ent_coef]["exp_avg"].view(()), pop.ent_opt.exp_avg[0][k])
        # the file has the shapes SAC.save writes for a trained SAC, and the loaded agent trains on
        mine, theirs = torch.load(path, weights_only=False), torch.load(ref_path, weights_only=False)
        assert mine.keys() == theirs.keys()
        for key in ("actor", "critic", "critic_target"):
            assert {n: t.shape for n, t in mine[key].items()} == {n: t.shape for n, t in theirs[key].items()}, key
        assert mine["log_ent_coef"].shape == theirs["log_ent_coef"].shape
        for key in ("actor_opt", "critic_opt", "ent_opt"):
            assert mine[key]["param_groups"][0].keys() == theirs[key]["param_groups"][0].keys(), key
            assert ({i: {n: t.shape for n, t in st.items()} for i, st in mine[key]["state"].items()}
                    == {i: {n: t.shape for n, t in st.items()} for i, st in theirs[key]["state"].items()}), key
        before = [p.detach().clone() for p in sac.actor.parameters()]
        sac.learn(80)
        assert sac.gradient_steps_done == 10
        assert all(torch.isfinite(p).all() and not torch.equal(p, q) for p, q in zip(sac.actor.parameters(), before))


def test_refuses_multi_rank_process_group(monkeypatch):
    import torch.distributed as dist
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda: 2)
    with pytest.raises(RuntimeError, match="multi-GPU"):
        SACPopulation(_TaggedEnv(n=4), [SACConfig(seed=0), SACConfig(seed=1)])


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("obs_dim", [6, 10, 22])
@pytest.mark.parametrize("n", [1, 8, 127, 129, 300])
@pytest.mark.parametrize("K", [1, 3, 16])
def test_grouped_actor_kernel_is_bit_identical_per_agent(K, n, obs_dim):
    _check_grouped_against_single_agent_launches(K, n, obs_dim)


@pytest.mark.gpu
@pytest.mark.parametrize("K, n", [(5, 128 * 40), (64, 1024), (200, 8)])
def test_grouped_actor_kernel_reloads_weights_within_a_cta(K, n):
    """More (agent, tile) pairs than SMs: persistent CTAs whose contiguous tile range crosses from one agent to
    the next, so they reload W2, b2 and the heads mid-loop.  The split is the kernel's (salp_sac.cu)."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = (n + 127) // 128
    total = K * tiles
    assert total > sms
    ranges = [(total * b // sms, total * (b + 1) // sms) for b in range(sms)]
    assert any(lo // tiles != (hi - 1) // tiles for lo, hi in ranges if hi > lo)
    _check_grouped_against_single_agent_launches(K, n, 10)


def _check_grouped_against_single_agent_launches(K, n, obs_dim):
    torch.manual_seed(K * 1000 + n + obs_dim)
    actors = [SacActor(obs_dim).cuda() for _ in range(K)]
    with torch.no_grad():                        # spread the log_std heads over the clamp bounds
        for a in actors:
            a.log_std.weight.mul_(10.0)
    lo, hi = [0.0, 0.0, -1.0], [1.0, 1.0, 1.0]
    group = SacActorGroupB200([torch.stack([p.detach() for p in ps]).contiguous()
                               for ps in zip(*(a.parameters() for a in actors))], lo, hi)
    singles = [SacActorB200(a, lo, hi) for a in actors]
    torch.cuda.synchronize()
    written = 256 * 256 * 2 + 4 * (256 * obs_dim + 2 * 256 + 6 * 256 + 6)   # (the rest is alignment padding)
    assert group.packed.numel() == K * singles[0].packed.numel()
    assert torch.equal(group.packed.view(K, -1)[:, :written], torch.stack([s.packed[:written] for s in singles]))
    obs = torch.randn(K * n, obs_dim, device="cuda") * 2
    noise = torch.randn(K * n, 3, device="cuda")
    for nz in (noise, None):
        env_g, a_g = torch.full((K * n, 3), float("nan"), device="cuda"), torch.full((K * n, 3), float("nan"), device="cuda")
        group.act(obs, nz, env_g, a_g)
        for k, s in enumerate(singles):
            rows = slice(k * n, (k + 1) * n)
            env_s, a_s = torch.empty(n, 3, device="cuda"), torch.empty(n, 3, device="cuda")
            s.act(obs[rows].contiguous(), None if nz is None else nz[rows].contiguous(), env_s, a_s)
            assert torch.equal(a_g[rows], a_s) and torch.equal(env_g[rows], env_s), k
    group.check()
    assert torch.isfinite(a_g).all()


@pytest.mark.gpu
def test_grouped_entry_points_check_their_arguments_on_device_pointers():
    """Every other argument a valid device pointer, so only the explicit checks can refuse these calls."""
    lib = _lib.load()
    K, n, D = 2, 8, 10
    nbytes = lib.salp_sac_weight_bytes(D)
    packed = torch.zeros(K * nbytes + 16, dtype=torch.uint8, device="cuda")
    w = torch.zeros(256 * 256 * K, device="cuda")
    obs, out = torch.zeros(K * n, 64, device="cuda"), torch.zeros(K * n, 3, device="cuda")
    ptr = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731
    lo, hi = (C.c_float * 3)(0, 0, -1), (C.c_float * 3)(1, 1, 1)
    pack = dict(k=K, d=D, dst=ptr(packed))
    for bad in (dict(k=0), dict(k=65536), dict(d=0), dict(d=65), dict(dst=ptr(packed, 4))):
        a = dict(pack, **bad)
        assert lib.salp_sac_pack_weights_grouped(*([ptr(w)] * 8), a["k"], a["d"], a["dst"], None) == _lib.ERR_INVALID, bad
    assert lib.salp_sac_pack_weights_grouped(*([ptr(w)] * 8), K, D, ptr(packed), None) == _lib.OK
    act = dict(packed=ptr(packed), k=K, d=D, n=n)
    for bad in (dict(k=0), dict(k=65536), dict(n=0), dict(n=-1), dict(d=0), dict(d=65), dict(packed=ptr(packed, 4))):
        a = dict(act, **bad)
        assert lib.salp_sac_act_grouped(a["packed"], a["k"], a["d"], ptr(obs), None, a["n"], lo, hi, ptr(out), ptr(out),
                                        None) == _lib.ERR_INVALID, bad
    assert lib.salp_sac_act_grouped(ptr(packed), K, D, ptr(obs), None, n, lo, hi, ptr(out), ptr(out), None) == _lib.OK
    assert lib.salp_sac_check() == 0


@pytest.mark.gpu
def test_agent_slice_of_a_batch_steps_like_its_own_batch():
    """Agent k's rows of a K n-env SalpBatch step bit-identically to SalpBatch(n, seed, env_id_offset=k n)
    under the same actions: what a population relies on."""
    from grasp_lab_salp_b200 import SalpBatch, default_params
    from grasp_lab_salp_b200.ppo import DeviceEnv
    K, n, seed = 3, 40, 6
    p = default_params()
    big = DeviceEnv(SalpBatch(K * n, p, seed=seed))
    parts = [DeviceEnv(SalpBatch(n, p, seed=seed, env_id_offset=k * n)) for k in range(K)]
    assert torch.equal(big.reset_t(), torch.cat([e.reset_t() for e in parts]))
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    lo, hi = torch.tensor([0.0, 0.0, -1.0], device="cuda"), torch.tensor([1.0, 1.0, 1.0], device="cuda")
    dones = 0
    for _ in range(50):
        act = lo + torch.rand((K * n, 3), device="cuda", generator=g) * (hi - lo)
        out = [t.clone() for t in big.step_t(act)]
        outs = [[t.clone() for t in e.step_t(act[k * n:(k + 1) * n].contiguous())] for k, e in enumerate(parts)]
        for i, t in enumerate(out):
            assert torch.equal(t, torch.cat([o[i] for o in outs])), i
        dones += int((out[2] | out[3]).sum())
    big.batch.check()
    print("episode ends over 50 steps:", dones)


def _gpu_population(n, seeds, **kw):
    from grasp_lab_salp_b200 import SalpBatch, default_params
    from grasp_lab_salp_b200.ppo import DeviceEnv
    batch = SalpBatch(n * len(seeds), default_params(), seed=seeds[0])
    return SACPopulation(DeviceEnv(batch), [SACConfig(seed=s, **kw) for s in seeds]), batch


@pytest.mark.gpu
def test_population_cuda_graphs_match_eager_training():
    """cuda_graphs=True and eager population training from the same seeds: 300 gradient steps agree to the
    tolerance of test_sac.py's test_cuda_graphs_match_eager_training."""
    res = []
    for graphs in (True, False):
        pop, batch = _gpu_population(64, [2, 3, 4], cuda_graphs=graphs, learning_starts=640, batch_size=256)
        rows = pop.learn(64 * 310, log_interval=64 * 310)
        batch.check()
        res.append((rows[-1], [p.detach().clone() for p in pop.actor_params]))
    (ra, pa), (rb, pb) = res
    assert ra["gradient_steps"] == rb["gradient_steps"] == 300
    print({k: (ra[k], rb[k]) for k in ("critic_loss", "actor_loss", "ent_coef", "mean_q")})
    for k in ("critic_loss", "actor_loss", "ent_coef", "mean_q"):
        for x, y in zip(ra[k], rb[k]):
            assert x == pytest.approx(y, rel=1e-3, abs=1e-3), k
    for x, y in zip(pa, pb):
        assert (x - y).abs().max().item() < 1e-3


@pytest.mark.gpu
def test_population_learns_on_gpu():
    """Four seeds of the reference recipe (8 envs each, 200k env-steps, SB3 defaults; CUDA graphs) as one
    population: every agent clears the bars of test_sac.py's test_sac_learns_on_gpu.  Measured on one B200
    (1000 W): 32.6 s of training, eval success 0.91 / 0.88 / 0.88 / 0.78 from 0.50 / 0.03 / 0.03 / 0.06."""
    from grasp_lab_salp_b200 import SalpBatch, default_params
    from grasp_lab_salp_b200.ppo import DeviceEnv
    K = 4
    pop, batch = _gpu_population(8, list(range(K)), cuda_graphs=True)
    ev_env = DeviceEnv(SalpBatch(K * 32, default_params(), seed=10_000))
    before = pop.evaluate(ev_env, 32)
    t0 = time.perf_counter()
    rows = pop.learn(200_000, log_interval=5000)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    batch.check()
    after = pop.evaluate(ev_env, 32)
    print(f"K={K} population: {wall:.1f} s wall for {pop.gradient_steps_done} gradient steps;",
          "eval before", before, "after", after, "last row", rows[-1])
    for k in range(K):
        assert after["success_rate"][k] >= 0.6 and after["mean_return"][k] > before["mean_return"][k], k
