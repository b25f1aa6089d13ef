"""SAC on the batched simulator (grasp_lab_salp_b200/sac.py) and its rollout-side actor kernel
(csrc/salp_sac.cu).  CPU: one gradient step against a line-by-line restatement of stable-baselines3's
SAC.train(), the squashed-Gaussian log-prob, replay semantics on a wrapping ring, evaluation against a
restatement of SB3's evaluate_policy quotas, the same curve on the host build of the kernel body and on the C
oracle, argument checks, save / load.  GPU: salp_sac_act against float64 and fp32 torch actors, rollout / ring /
CUDA-graph equivalence, learning."""
import copy
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from grasp_lab_salp_b200 import PRECISION_F64, _lib
from grasp_lab_salp_b200.ppo import HostEnv
from grasp_lab_salp_b200.sac import SAC, SacActor, SacActorB200, SACConfig
from parity import golden_params, load_golden


def _host_env(n, seed=4, oracle=False):
    g = load_golden("ref_random.npz")
    p = golden_params(g, precision=PRECISION_F64)
    if oracle:
        from oracle.salp_oracle import OracleVecEnv
        return HostEnv(OracleVecEnv(n, p, seed=seed))
    from emu_backend import EmuBatch
    return HostEnv(EmuBatch(n, p, seed=seed))


class _TaggedEnv:
    """A tiny deterministic env with the HostEnv face: obs carry (env index, step count), episodes end
    by `terminated` every 5th step and by `truncated` every 7th (auto-reset, terminal_obs kept)."""

    def __init__(self, n=3, obs_dim=6):
        self.num_envs, self.obs_dim, self.device = n, obs_dim, torch.device("cpu")
        self.t = 0

    def _obs(self, t):
        o = torch.zeros(self.num_envs, self.obs_dim)
        o[:, 0] = torch.arange(self.num_envs, dtype=torch.float32)
        o[:, 1] = float(t)
        return o

    def reset_t(self):
        self.t = 0
        return self._obs(0)

    def step_t(self, actions):
        self.t += 1
        nxt = self._obs(self.t)
        term = torch.zeros(self.num_envs, dtype=torch.bool)
        trunc = torch.zeros(self.num_envs, dtype=torch.bool)
        term[0] = self.t % 5 == 0
        trunc[1] = self.t % 7 == 0
        done = term | trunc
        obs = nxt.clone()
        obs[done, 1] = -1.0                      # post-reset observation of the finished envs
        rew = actions.sum(1) + 100.0 * self.t
        return obs, rew, term, trunc, nxt


# ------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------
def _sb3_train_step(actor, critic, critic_target, log_ent_coef, ent_coef_tensor, opts, batch, eps, gamma, tau,
                    target_entropy):
    """stable-baselines3 SAC.train(), one gradient step, restated line by line (sb3 2.x, sac.py) with the
    actor's rsample noise given as `eps` (torch.distributions.Normal.rsample: loc + eps * scale)."""
    actor_opt, critic_opt, ent_opt = opts

    def action_log_prob(obs, e):
        latent = actor.latent_pi(obs)
        mean_actions = actor.mu(latent)
        log_std = torch.clamp(actor.log_std(latent), -20, 2)
        action_std = torch.ones_like(mean_actions) * log_std.exp()
        dist = torch.distributions.Normal(mean_actions, action_std)
        gaussian_actions = mean_actions + e * action_std
        actions = torch.tanh(gaussian_actions)
        log_prob = dist.log_prob(gaussian_actions).sum(dim=1)
        log_prob -= torch.sum(torch.log(1 - actions ** 2 + 1e-6), dim=1)
        return actions, log_prob

    def q(net, obs, act):
        qvalue_input = torch.cat([obs, act], dim=1)
        return tuple(q_net(qvalue_input) for q_net in net.q_networks)

    actions_pi, log_prob = action_log_prob(batch["obs"], eps[0])
    log_prob = log_prob.reshape(-1, 1)
    ent_coef_loss = None
    if ent_opt is not None and log_ent_coef is not None:
        ent_coef = torch.exp(log_ent_coef.detach())
        ent_coef_loss = -(log_ent_coef * (log_prob + target_entropy).detach()).mean()
    else:
        ent_coef = ent_coef_tensor
    if ent_coef_loss is not None and ent_opt is not None:
        ent_opt.zero_grad()
        ent_coef_loss.backward()
        ent_opt.step()
    with torch.no_grad():
        next_actions, next_log_prob = action_log_prob(batch["next_obs"], eps[1])
        next_q_values = torch.cat(q(critic_target, batch["next_obs"], next_actions), dim=1)
        next_q_values, _ = torch.min(next_q_values, dim=1, keepdim=True)
        next_q_values = next_q_values - ent_coef * next_log_prob.reshape(-1, 1)
        target_q_values = batch["rewards"] + (1 - batch["dones"]) * gamma * next_q_values
    current_q_values = q(critic, batch["obs"], batch["actions"])
    critic_loss = 0.5 * sum(F.mse_loss(current_q, target_q_values) for current_q in current_q_values)
    critic_opt.zero_grad()
    critic_loss.backward()
    critic_opt.step()
    q_values_pi = torch.cat(q(critic, batch["obs"], actions_pi), dim=1)
    min_qf_pi, _ = torch.min(q_values_pi, dim=1, keepdim=True)
    actor_loss = (ent_coef * log_prob - min_qf_pi).mean()
    actor_opt.zero_grad()
    actor_loss.backward()
    actor_opt.step()
    with torch.no_grad():                        # polyak_update
        for param, target_param in zip(critic.parameters(), critic_target.parameters()):
            target_param.data.mul_(1 - tau)
            torch.add(target_param.data, param.data, alpha=tau, out=target_param.data)
    return critic_loss, actor_loss, ent_coef_loss


def _sb3_evaluate(predict, env, n_episodes, agents=1):
    """stable-baselines3 evaluate_policy(deterministic=True) restated as a host loop over the env's K = `agents`
    slices of m envs: env i of a slice contributes (n_episodes + i) // m episodes to its agent.  Per-agent list of
    dicts of mean_return, mean_length, success_rate and episodes."""
    n = env.num_envs
    m = n // agents
    targets = torch.tensor([(n_episodes + i % m) // m for i in range(n)])
    counts = torch.zeros(n, dtype=torch.long)
    rets, lens, succ = ([[] for _ in range(agents)] for _ in range(3))
    cur_r, cur_l = torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.long)
    obs = env.reset_t()
    while bool((counts < targets).any()):
        a = predict(obs.float(), deterministic=True)
        obs, rew, term, trunc, _ = env.step_t(a)
        r = torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0).double().cpu()
        t, d = term.bool().cpu(), (term.bool() | trunc.bool()).cpu()
        cur_r += r
        cur_l += 1
        for i in torch.nonzero(d & (counts < targets)).flatten().tolist():
            rets[i // m].append(cur_r[i].item())
            lens[i // m].append(cur_l[i].item())
            succ[i // m].append(float(t[i]))
            counts[i] += 1
        cur_r[d] = 0.0
        cur_l[d] = 0
    return [dict(mean_return=sum(r) / len(r), mean_length=sum(ln) / len(r), success_rate=sum(s) / len(r),
                 episodes=len(r)) for r, ln, s in zip(rets, lens, succ)]


def _assert_eval_matches(mine, ref):
    """Episode counts, lengths and success rates exactly, returns to 1e-12 relative."""
    for key in ("episodes", "mean_length", "success_rate"):
        assert mine[key] == ref[key], key
    assert mine["mean_return"] == pytest.approx(ref["mean_return"], rel=1e-12, abs=0)


def test_evaluate_matches_sb3_quota_restatement():
    sac = SAC(_host_env(4), SACConfig(seed=3))
    ref = _sb3_evaluate(sac.predict, _host_env(3, seed=9), 5)[0]     # quotas 1, 2, 2
    ev = sac.evaluate(_host_env(3, seed=9), 5)
    assert ev["episodes"] == 5
    _assert_eval_matches(ev, ref)


@pytest.mark.parametrize("ent_coef", ["auto", 0.2])
def test_gradient_step_matches_sb3_restatement(ent_coef):
    env = _TaggedEnv(n=4, obs_dim=6)
    sac = SAC(env, SACConfig(ent_coef=ent_coef, seed=7))
    torch.manual_seed(1)
    B = 64
    batch = dict(obs=torch.randn(B, 6), actions=torch.rand(B, 3) * 2 - 1, next_obs=torch.randn(B, 6),
                 rewards=torch.randn(B, 1) * 10, dones=(torch.rand(B, 1) < 0.2).float())
    eps = (torch.randn(B, 3), torch.randn(B, 3))
    actor, critic, target = copy.deepcopy(sac.actor), copy.deepcopy(sac.critic), copy.deepcopy(sac.critic_target)
    log_ent = None if sac.log_ent_coef is None else sac.log_ent_coef.detach().clone().requires_grad_(True)
    opts = [torch.optim.Adam(actor.parameters(), lr=3e-4), torch.optim.Adam(critic.parameters(), lr=3e-4),
            None if log_ent is None else torch.optim.Adam([log_ent], lr=3e-4)]
    ent_t = None if sac.auto_ent else torch.tensor(float(ent_coef))
    for _ in range(2):                           # a second step exercises Adam's moments and the target update
        ref = _sb3_train_step(actor, critic, target, log_ent, ent_t, opts, batch, eps, 0.99, 0.005, -3.0)
        out = sac.train_step(batch, eps)
        assert abs(out["critic_loss"].item() - ref[0].item()) < 1e-6
        assert abs(out["actor_loss"].item() - ref[1].item()) < 1e-6
        if sac.auto_ent:
            assert abs(out["ent_coef_loss"].item() - ref[2].item()) < 1e-6
            assert abs(sac.log_ent_coef.item() - log_ent.item()) < 1e-6
            assert sac.log_ent_coef.item() != 0.0
        for mine, theirs in ((sac.actor, actor), (sac.critic, critic), (sac.critic_target, target)):
            for (k, a), (_, b) in zip(mine.state_dict().items(), theirs.state_dict().items()):
                assert (a - b).abs().max().item() < 1e-6, k
    assert not torch.equal(sac.critic_target.state_dict()["q_networks.0.0.weight"],
                           sac.critic.state_dict()["q_networks.0.0.weight"])


def test_networks_match_sb3_defaults():
    torch.manual_seed(0)
    sac = SAC(_TaggedEnv(n=2, obs_dim=10), SACConfig())
    assert [m.out_features for m in sac.actor.latent_pi if hasattr(m, "out_features")] == [256, 256]
    assert (sac.actor.mu.in_features, sac.actor.mu.out_features) == (256, 3)
    assert (sac.actor.log_std.in_features, sac.actor.log_std.out_features) == (256, 3)
    for q in sac.critic.q_networks:
        assert [m.out_features for m in q if hasattr(m, "out_features")] == [256, 256, 1]
        assert q[0].in_features == 13
    for a, b in zip(sac.critic.parameters(), sac.critic_target.parameters()):
        assert torch.equal(a, b)
    w = sac.actor.latent_pi[0].weight           # torch default init: U(-1/sqrt(fan_in), 1/sqrt(fan_in))
    assert w.abs().max().item() <= 1 / math.sqrt(10) and w.abs().max().item() > 0.9 / math.sqrt(10)
    assert sac.log_ent_coef.item() == 0.0 and sac.cfg.target_entropy == -3.0
    assert sac.slots == 100_000 // 2


def test_squashed_gaussian_log_prob_closed_form():
    torch.manual_seed(2)
    actor = SacActor(6).double()
    with torch.no_grad():                        # log_std heads that clamp at both ends
        actor.log_std.bias.copy_(torch.tensor([-30.0, 8.0, 0.0], dtype=torch.float64))
    obs = torch.randn(50, 6, dtype=torch.float64)
    eps = torch.randn(50, 3, dtype=torch.float64) * 0.3
    a, logp = actor.action_log_prob(obs, eps)
    mu, log_std = actor(obs)
    assert (log_std[:, 0] == -20).all() and (log_std[:, 1] == 2).all()
    u = mu + torch.exp(log_std) * eps
    closed = (-0.5 * eps ** 2 - log_std - 0.5 * math.log(2 * math.pi)).sum(1) - torch.log(1 - torch.tanh(u) ** 2 + 1e-6).sum(1)
    np.testing.assert_allclose(a.detach(), torch.tanh(u).detach(), rtol=0, atol=1e-12)
    np.testing.assert_allclose(logp.detach(), closed.detach(), rtol=1e-9, atol=1e-7)


def test_replay_semantics_on_a_wrapping_ring():
    env = _TaggedEnv(n=3, obs_dim=6)
    sac = SAC(env, SACConfig(buffer_size=3 * 4, learning_starts=1000, seed=1))       # 4 slots
    assert sac.slots == 4 and not sac.zero_copy
    lo, hi = torch.tensor([0.0, 0.0, -1.0]), torch.tensor([1.0, 1.0, 1.0])
    steps = []
    for _ in range(11):
        obs_before = sac._obs.clone()
        s = sac.pos
        sac._vec_step()
        steps.append((s, obs_before, sac._env_act.clone(), env.t))
        rb = sac.rb
        # next_obs is terminal_obs on reset rows (step count t) and the following obs elsewhere
        assert torch.equal(rb["next_obs"][s][:, 1], torch.full((3,), float(env.t)))
        assert torch.equal(rb["obs"][s], obs_before)
        # stored done is `terminated` only (env 0 every 5th step); env 1's truncations are not done
        assert rb["done"][s].tolist() == [int(env.t % 5 == 0), 0, 0]
        # warm-up actions: uniform on the Box, stored scaled to [-1, 1]
        a_env = sac._env_act
        assert ((a_env >= lo) & (a_env <= hi)).all()
        np.testing.assert_allclose(rb["act"][s], 2 * (a_env - lo) / (hi - lo) - 1, atol=1e-6)
        assert torch.equal(rb["rew"][s], (a_env.sum(1) + 100.0 * env.t).float())
    assert sac.full and sac.pos == 11 % 4
    # after 11 steps slot pos (3) holds step 8 (t = 8) -- sampling must skip it once wrapped
    sample = sac.sample(4000)
    assert not (sample["slot"] == sac.pos).any()
    assert set(sample["slot"].tolist()) == {0, 1, 2} and set(sample["env"].tolist()) == {0, 1, 2}
    # every sampled transition is one step of one env: obs tag t-1 (or -1 after a reset), next tag t
    t_next = sample["next_obs"][:, 1]
    t_obs = sample["obs"][:, 1]
    assert torch.equal(sample["obs"][:, 0], sample["env"].float())
    assert ((t_obs == t_next - 1) | (t_obs == -1)).all()
    r = sample["rewards"][:, 0] - 100.0 * t_next     # the action sum of that step, within the Box's [-1, 3]
    small = t_next <= 9
    assert ((r >= -1) & (r <= 3))[small].all()
    assert (sample["rewards"][~small, 0] <= 1000.0).all() and (~small).any()    # the learner-side clip
    # before wrapping: only the filled slots
    sac2 = SAC(_TaggedEnv(n=3, obs_dim=6), SACConfig(buffer_size=3 * 4, learning_starts=1000, seed=1))
    sac2._vec_step()
    sac2._vec_step()
    assert set(sac2.sample(500)["slot"].tolist()) == {0, 1}


def test_no_gradient_step_before_learning_starts():
    env = _TaggedEnv(n=4, obs_dim=6)
    sac = SAC(env, SACConfig(learning_starts=20, batch_size=8, seed=0))
    sac.learn(20, log_interval=4)
    assert sac.num_timesteps == 20 and sac.gradient_steps_done == 0
    sac.learn(24, log_interval=4)                 # 24 > 20: the first gradient step
    assert sac.gradient_steps_done == 1
    sac.learn(32, log_interval=4)
    assert sac.gradient_steps_done == 3


def _sac_curve(oracle):
    env = _host_env(8, seed=4, oracle=oracle)
    sac = SAC(env, SACConfig(learning_starts=64, batch_size=32, buffer_size=2000, seed=3))
    rows = sac.learn(8 * 24, log_interval=64)
    return [(r["episodes"], r["critic_loss"], r["actor_loss"], r["ent_coef"]) for r in rows]


def test_same_learning_curve_on_kernel_body_and_oracle():
    """Same SAC, same seed, env = host build of the CUDA step body vs env = C oracle: the curves coincide
    (the envs agree to 1e-9, and a few gradient steps stay far from any decision boundary)."""
    a = _sac_curve(False)
    b = _sac_curve(True)
    assert len(a) == len(b) == 3
    assert np.isfinite(a[-1][1])
    for (ea, ca, aa, ka), (eb, cb, ab, kb) in zip(a, b):
        assert ea == eb
        for x, y in ((ca, cb), (aa, ab), (ka, kb)):
            assert (math.isnan(x) and math.isnan(y)) or x == pytest.approx(y, rel=1e-4, abs=1e-4)


def test_entry_points_and_wrapper_reject_bad_input():
    lib = _lib.load()
    assert lib.salp_sac_weight_bytes(0) == _lib.ERR_INVALID and lib.salp_sac_weight_bytes(65) == _lib.ERR_INVALID
    assert lib.salp_sac_weight_bytes(10) == 256 * 256 * 2 + 4 * (256 * 10 + 512 + 6 * 256 + 6) + 8
    assert lib.salp_sac_weight_bytes(64) % 16 == 0
    assert lib.salp_sac_pack_weights(*([None] * 8), 10, None, None) == _lib.ERR_INVALID
    lo, hi = (C.c_float * 3)(0, 0, -1), (C.c_float * 3)(1, 1, 1)
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    assert lib.salp_sac_act(None, 10, p, None, 8, lo, hi, p, p, None) == _lib.ERR_INVALID
    assert lib.salp_sac_act(p, 10, None, None, 8, lo, hi, p, p, None) == _lib.ERR_INVALID
    assert lib.salp_sac_act(p, 10, p, None, 0, lo, hi, p, p, None) == _lib.ERR_INVALID
    assert lib.salp_sac_act(p, 0, p, None, 8, lo, hi, p, p, None) == _lib.ERR_INVALID
    assert lib.salp_sac_act(p, 65, p, None, 8, lo, hi, p, p, None) == _lib.ERR_INVALID
    assert lib.salp_sac_act(p, 10, p, None, 8, None, hi, p, p, None) == _lib.ERR_INVALID
    assert lib.salp_sac_act(p, 10, p, None, 8, lo, hi, None, p, None) == _lib.ERR_INVALID
    if not torch.cuda.is_available():            # host memory is not a device pointer
        assert lib.salp_sac_act(p, 10, p, None, 8, lo, hi, p, p, None) == _lib.ERR_INVALID
    with pytest.raises(RuntimeError, match="no CPU path"):
        SacActorB200(SacActor(10), (0, 0, -1), (1, 1, 1))


def test_save_load_round_trip(tmp_path):
    env = _TaggedEnv(n=4, obs_dim=6)
    sac = SAC(env, SACConfig(learning_starts=8, batch_size=16, seed=5))
    sac.learn(40)
    obs = torch.randn(10, 6)
    a = sac.predict(obs, deterministic=True)
    path = tmp_path / "sac.pt"
    sac.save(path)
    other = SAC(_TaggedEnv(n=4, obs_dim=6), SACConfig(seed=99))
    assert not torch.equal(other.predict(obs), a)
    other.load(path)
    assert torch.equal(other.predict(obs), a)
    assert other.log_ent_coef.item() == sac.log_ent_coef.item() and other.num_timesteps == 40
    for x, y in zip(other.critic_target.parameters(), sac.critic_target.parameters()):
        assert torch.equal(x, y)


def test_refuses_multi_rank_process_group(monkeypatch):
    import torch.distributed as dist
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda: 2)
    with pytest.raises(RuntimeError, match="multi-GPU"):
        SAC(_TaggedEnv(), SACConfig())


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _actor_reference_f64(actor, obs, noise, lo, hi):
    """float64 actor fed the operands salp_sac_act rounds: h1 = the kernel's fp32 fmaf chain (emulated:
    each fp32 fma is exact in float64 before its rounding to fp32), rounded to bf16; W2 rounded to bf16."""
    w1, b1 = actor.latent_pi[0].weight.double(), actor.latent_pi[0].bias.float()
    x = obs.double()
    acc = b1.unsqueeze(0).expand(obs.shape[0], -1).clone()
    for d in range(obs.shape[1]):
        acc = (acc.double() + x[:, d:d + 1] * w1[:, d]).float()
    h1 = acc.clamp_min(0).bfloat16().double()
    w2 = actor.latent_pi[2].weight.bfloat16().double()
    lat = (h1 @ w2.T + actor.latent_pi[2].bias.double()).clamp_min(0)
    mu = lat @ actor.mu.weight.double().T + actor.mu.bias.double()
    ls = (lat @ actor.log_std.weight.double().T + actor.log_std.bias.double()).clamp(-20, 2)
    u = mu if noise is None else mu + ls.exp() * noise.double()
    a = torch.tanh(u)
    return mu, ls, a, lo.double() + (a + 1) / 2 * (hi.double() - lo.double())


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dim", [6, 10, 22])
@pytest.mark.parametrize("n", [1, 127, 129, 4096 + 37, 65536])
def test_sac_actor_kernel_matches_torch(n, obs_dim):
    """salp_sac_act against (1) a float64 actor fed the same bf16-rounded h1 and W2: 1e-4 relative to
    max(1, |x|) on mu and the clamped log_std (recovered from the kernel's deterministic and noisy outputs),
    with scaled heads whose log_std biases put rows on both sides of the clamp at -20 and 2; and (2) the
    fp32 torch forward of a default-initialised actor: 2e-2 absolute on the scaled and the env action."""
    torch.manual_seed(n + obs_dim)
    actor = SacActor(obs_dim).cuda()
    with torch.no_grad():
        actor.latent_pi[0].weight.mul_(2.0)
        actor.mu.weight.mul_(3.0)
        actor.log_std.weight.mul_(10.0)
    obs = torch.randn(n, obs_dim, device="cuda") * 2
    with torch.no_grad():                        # centre the log_std heads on the clamp bounds: rows on both sides
        raw = actor.log_std(actor.latent_pi(obs)) - actor.log_std.bias
        actor.log_std.bias.copy_(torch.tensor([-20.0, 2.0, -1.0], device="cuda") - raw.median(dim=0).values)
    lo, hi = torch.tensor([0.0, 0.0, -1.0], device="cuda"), torch.tensor([1.0, 1.0, 1.0], device="cuda")
    fused = SacActorB200(actor, lo.tolist(), hi.tolist())
    noise = torch.randn(n, 3, device="cuda")
    env_a, a = torch.full((n, 3), float("nan"), device="cuda"), torch.full((n, 3), float("nan"), device="cuda")
    env_d, a_d = torch.empty_like(env_a), torch.empty_like(a)
    fused.act(obs, noise, env_a, a)
    fused.act(obs, None, env_d, a_d)
    fused.check()
    assert torch.isfinite(a).all() and torch.isfinite(env_a).all()
    with torch.no_grad():
        mu, ls, a_ref, env_ref = _actor_reference_f64(actor, obs, noise, lo, hi)
        _, _, a_ref_d, env_ref_d = _actor_reference_f64(actor, obs, None, lo, hi)
        # mu from the deterministic call (atanh is well conditioned where |a| < 0.99)
        ok = a_d.abs() < 0.99
        mu_k = torch.atanh(a_d.double())
        err_mu = ((mu_k - mu).abs() / mu.abs().clamp_min(1.0))[ok].max().item()
        # clamped log_std from the noisy call where the sample is not saturated
        u_k = torch.atanh(a.double())
        ok2 = (a.abs() < 0.99) & ((u_k - mu_k).abs() > 0.1)       # (u - mu) = std * noise well above atanh's error
        ls_k = torch.log(((u_k - mu_k) / noise.double()).clamp_min(1e-30))
        err_ls = ((ls_k - ls).abs() / ls.abs().clamp_min(1.0))[ok2 & ok].max().item() if (ok2 & ok).any() else 0.0
        if n > 1:
            assert (ls[:, 0] == -20).any() and (ls[:, 1] == 2).any() and (ls[:, 0] > -20).any() and (ls[:, 1] < 2).any()
        err_a64 = max((a.double() - a_ref).abs().max().item(), (a_d.double() - a_ref_d).abs().max().item())
        err_env64 = (env_a.double() - env_ref).abs().max().item()
        # bar (2) on a default-initialised actor: the bf16 rounding of h1 and W2 against fp32 torch
        plain = SacActor(obs_dim).cuda()
        fused_plain = SacActorB200(plain, lo.tolist(), hi.tolist())
        a_p, env_p = torch.empty_like(a), torch.empty_like(env_a)
        a_pd, env_pd = torch.empty_like(a), torch.empty_like(env_a)
        fused_plain.act(obs, noise, env_p, a_p)
        fused_plain.act(obs, None, env_pd, a_pd)
        mean32, ls32 = plain(obs)
        a32 = torch.tanh(mean32 + ls32.exp() * noise)
        a32_d = torch.tanh(mean32)
        err_a32 = max((a_p - a32).abs().max().item(), (a_pd - a32_d).abs().max().item())
        env32 = lo + (a32 + 1) / 2 * (hi - lo)
        err_env32 = (env_p - env32).abs().max().item()
    print(f"n={n} D={obs_dim}: mu {err_mu:.2e}, log_std {err_ls:.2e}, action vs f64 {err_a64:.2e} (env {err_env64:.2e}), "
          f"vs fp32 torch {err_a32:.2e} (env {err_env32:.2e})")
    assert err_mu < 1e-4 and err_ls < 1e-4
    assert err_a64 < 1e-4 and err_env64 < 1e-4
    assert err_a32 < 2e-2 and err_env32 < 2e-2
    # new weights are picked up by pack()
    with torch.no_grad():
        actor.latent_pi[2].weight.mul_(-0.5)
    fused.pack()
    fused.act(obs, None, env_d, a_d)
    with torch.no_grad():
        _, _, a_ref_d, _ = _actor_reference_f64(actor, obs, None, lo, hi)
    assert (a_d.double() - a_ref_d).abs().max().item() < 1e-4
    assert _lib.load().salp_sac_check() == 0


def _gpu_sac(n, seed, **kw):
    from grasp_lab_salp_b200 import SalpBatch, default_params
    from grasp_lab_salp_b200.ppo import DeviceEnv
    batch = SalpBatch(n, default_params(), seed=seed)
    return SAC(DeviceEnv(batch), SACConfig(seed=seed, **kw)), batch


@pytest.mark.gpu
def test_rollout_with_fused_actor_tracks_torch_actor():
    """Same seeds, fused actor vs torch actor: identical first-step observations, replay contents within
    the kernel's tolerance over a few policy steps."""
    rings = []
    for fused in (True, False):
        sac, batch = _gpu_sac(512, 3, fused_actor=fused, learning_starts=0, buffer_size=512 * 8)
        assert (sac.fused is not None) == fused
        for _ in range(3):
            sac._vec_step()
        torch.cuda.synchronize()
        batch.check()
        rings.append({k: v[:3].clone() for k, v in sac.rb.items()})
    assert torch.equal(rings[0]["obs"][0], rings[1]["obs"][0])
    assert (rings[0]["act"][0] - rings[1]["act"][0]).abs().max().item() < 2e-2
    print("act diff per step", [(rings[0]["act"][i] - rings[1]["act"][i]).abs().max().item() for i in range(3)])


@pytest.mark.gpu
def test_zero_copy_ring_equals_copy_fill():
    """The zero-copy ring (step_device(out=...)) holds bit-identical transitions to the copy-based fill."""
    rings = []
    for zero_copy in (True, False):
        sac, batch = _gpu_sac(1000, 5, learning_starts=5 * 1000, buffer_size=1000 * 4)
        sac.zero_copy = zero_copy
        for _ in range(6):                       # wraps the 4-slot ring
            sac._vec_step()
        sac.learn(sac.num_timesteps + 3 * 1000)  # policy steps and gradient steps
        torch.cuda.synchronize()
        batch.check()
        rings.append((sac.rb, sac.pos, sac._ep.clone()))
    (ra, pa, ea), (rb, pb, eb) = rings
    assert pa == pb
    for k in ra:
        live = [s for s in range(4) if s != pa]  # (the slot being filled differs by design)
        assert torch.equal(ra[k][live], rb[k][live]), k
    assert torch.equal(ea, eb)


@pytest.mark.gpu
def test_cuda_graphs_match_eager_training():
    """cuda_graphs=True and eager training from the same seeds: 300 gradient steps agree to fp32
    summation-order tolerance."""
    res = []
    for graphs in (True, False):
        sac, batch = _gpu_sac(64, 2, cuda_graphs=graphs, learning_starts=640, batch_size=256)
        rows = sac.learn(64 * 310, log_interval=64 * 310)
        batch.check()
        res.append((rows[-1], [p.detach().clone() for p in sac.actor.parameters()]))
    (ra, pa), (rb, pb) = res
    assert ra["gradient_steps"] == rb["gradient_steps"] == 300
    print({k: (ra[k], rb[k]) for k in ("critic_loss", "actor_loss", "ent_coef", "mean_q")})
    for k in ("critic_loss", "actor_loss", "ent_coef", "mean_q"):
        assert ra[k] == pytest.approx(rb[k], rel=1e-3, abs=1e-3), k
    for x, y in zip(pa, pb):
        assert (x - y).abs().max().item() < 1e-3


@pytest.mark.gpu
def test_sac_learns_on_gpu():
    """The reference recipe (8 envs, 200k env-steps, SB3 defaults; CUDA graphs) on one B200, about 35 s:
    deterministic evaluation over 32 episodes before and after.  Measured with seeds 0 / 1 / 2
    (profiles/r03_sac_ref_8envs_200k_seed*.jsonl): final eval success 0.906 / 0.969 / 0.906, eval return
    527 / 567 / 537, training-episode success over the last 5000 env-steps 0.90 / 0.88 / 0.89; on this
    test's own evaluation batch seed 0 goes from success 0.50 / return 80 untrained to 0.91 / 525.  The
    bars sit well below the worst seed."""
    from grasp_lab_salp_b200 import SalpBatch, default_params
    from grasp_lab_salp_b200.ppo import DeviceEnv
    sac, batch = _gpu_sac(8, 0, cuda_graphs=True)
    ev_env = DeviceEnv(SalpBatch(32, default_params(), seed=10_000))
    before = sac.evaluate(ev_env, 32)
    rows = sac.learn(200_000, log_interval=5000)
    batch.check()
    after = sac.evaluate(ev_env, 32)
    print("eval before", before, "after", after, "last row", rows[-1])
    assert after["success_rate"] >= 0.6 and after["mean_return"] > before["mean_return"]
    assert rows[-1]["success_rate"] > 0.6
