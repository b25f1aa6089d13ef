"""PPO on device tensors over the batched SALP simulator (SURVEY.md section 8f, rank 1).

Stands in for stable-baselines3 ``PPO("MlpPolicy", vec_env)`` with SB3's defaults (the reference
ships SAC and RecurrentPPO scripts only -- src/train_robot.py:62-69, src/train_robot_recurrent_ppo.py
:85-107 -- and BASELINE.json config 3 asks for "PPO MLP policy ... with 16k envs", so SB3's PPO
defaults are the stand-in, SURVEY section 3.1):

  * policy: separate actor / critic MLPs 64-64 tanh, orthogonal init (gain sqrt(2); 0.01 on the
    action head, 1 on the value head), state-independent log_std = 0, diagonal Gaussian;
    actions are clipped to the Box only when handed to the env (SB3 on-policy collect_rollouts);
  * GAE(gamma = 0.99, lambda = 0.95); on a TimeLimit truncation the reward is bootstrapped with
    gamma * V(terminal_observation), as SB3 does;
  * clipped surrogate (0.2), value coefficient 0.5, entropy coefficient 0, advantage
    normalisation per minibatch, Adam 3e-4, gradient clipping at 0.5, 10 epochs per rollout.

Nothing leaves the GPU: the rollout buffer, the policy forward (cuBLAS GEMMs -- the only dense
algebra here) and ``SalpBatch.step_device`` all work on device tensors; per-iteration statistics
are reduced on device and read back once.  Multi-GPU: one process per GPU, envs sharded
(``distributed.make_shard``), gradients and rollout statistics all-reduced over NCCL.

Both algorithms have SB3's ``predict``, ``evaluate`` (evaluate_policy(deterministic=True), also run by
``learn`` every ``eval_every`` env-steps on an ``eval_env``), ``save`` and ``load`` (torch.save, not SB3's
zip format).  Inference and evaluation use buffers of their own, so they can run between the captured
CUDA graphs of a training run without changing it.

The env is anything with ``num_envs``, ``obs_dim``, ``reset_t() -> obs`` and
``step_t(actions) -> (obs, reward, terminated, truncated, terminal_obs)`` on torch tensors;
``DeviceEnv`` adapts a SalpBatch (CUDA), ``HostEnv`` adapts any numpy backend with the SalpBatch
host face (the CPU oracle and the host build of the kernel body in the tests).
"""
from __future__ import annotations

import math
import time
from dataclasses import dataclass, field

import numpy as np
import torch
import torch.nn as nn

from .evaluation import run_episodes
from .params import sort_by_k_auto


# ------------------------------------------------------------------------------------------------
# env adapters
# ------------------------------------------------------------------------------------------------
class DeviceEnv:
    """SalpBatch device face: zero-copy, asynchronous on the current stream."""

    def __init__(self, batch, sort_by_k="auto"):
        self.batch = batch
        self.num_envs, self.obs_dim = batch.num_envs, batch.obs_dim
        self.device = torch.device("cuda", batch.device)
        self.sort = sort_by_k_auto(batch.num_envs) if sort_by_k == "auto" else bool(sort_by_k)

    def reset_t(self):
        return self.batch.reset_device().clone()

    def step_t(self, actions):
        obs, rew, term, trunc = self.batch.step_device(actions, auto_reset=True, sort_by_k=self.sort)
        return obs, rew, term.bool(), trunc.bool(), self.batch.dev["terminal_obs"]


class HostEnv:
    """Any backend with the numpy face of SalpBatch (oracle, host build of the kernel body)."""

    def __init__(self, backend, device="cpu"):
        self.b = backend
        self.num_envs, self.obs_dim = backend.num_envs, backend.obs_dim
        self.device = torch.device(device)

    def reset_t(self):
        return torch.from_numpy(self.b.reset().copy()).to(self.device)

    def step_t(self, actions):
        obs, rew, term, trunc = self.b.step(actions.detach().cpu().numpy().astype(np.float32), auto_reset=True)
        t = lambda a, dt=None: torch.from_numpy(np.array(a, dtype=dt)).to(self.device)  # noqa: E731
        return (t(obs, np.float32), t(rew, np.float32), t(term, bool), t(trunc, bool),
                t(self.b.terminal_obs, np.float32))


# ------------------------------------------------------------------------------------------------
# policy (SB3 MlpPolicy defaults)
# ------------------------------------------------------------------------------------------------
def _mlp(inp, hidden, out, out_gain):
    layers, d = [], inp
    for h in hidden:
        lin = nn.Linear(d, h)
        nn.init.orthogonal_(lin.weight, gain=math.sqrt(2))
        nn.init.zeros_(lin.bias)
        layers += [lin, nn.Tanh()]
        d = h
    head = nn.Linear(d, out)
    nn.init.orthogonal_(head.weight, gain=out_gain)
    nn.init.zeros_(head.bias)
    return nn.Sequential(*layers, head)


class MlpPolicy(nn.Module):
    def __init__(self, obs_dim=10, act_dim=3, hidden=(64, 64), log_std_init=0.0):
        super().__init__()
        self.actor = _mlp(obs_dim, hidden, act_dim, 0.01)
        self.critic = _mlp(obs_dim, hidden, 1, 1.0)
        self.log_std = nn.Parameter(torch.full((act_dim,), float(log_std_init)))

    def dist(self, obs):
        return torch.distributions.Normal(self.actor(obs), self.log_std.exp(), validate_args=False)

    def value(self, obs):
        return self.critic(obs).squeeze(-1)

    @torch.no_grad()
    def act(self, obs, generator=None):
        mean = self.actor(obs)
        noise = torch.randn(mean.shape, device=mean.device, dtype=mean.dtype, generator=generator)
        a = mean + noise * self.log_std.exp()
        logp = (-0.5 * noise.pow(2) - self.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        return a, logp, self.value(obs)

    def packed(self):
        """All rollout-side parameters as ONE float array in the layout salp_mlp_act expects
        (include/salp_b200.h): actor W1 b1 W2 b2 W3 b3, critic W1 b1 W2 b2 W3 b3, log_std."""
        a, c = self.actor, self.critic
        return torch.cat([t.detach().reshape(-1) for t in (
            a[0].weight, a[0].bias, a[2].weight, a[2].bias, a[4].weight, a[4].bias,
            c[0].weight, c[0].bias, c[2].weight, c[2].bias, c[4].weight, c[4].bias, self.log_std)])

    def evaluate(self, obs, actions):
        """log-prob, entropy, value -- written out (no torch.distributions: its argument validation
        synchronises the stream, which also forbids CUDA-graph capture)."""
        mean = self.actor(obs)
        z = (actions - mean) * (-self.log_std).exp()
        logp = (-0.5 * z.pow(2) - self.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + self.log_std).sum().expand(obs.shape[0])
        return logp, ent, self.value(obs)


# ------------------------------------------------------------------------------------------------
# PPO
# ------------------------------------------------------------------------------------------------
@dataclass
class PPOConfig:
    n_steps: int = 32                 # rollout length per env (SB3 default 2048 is for 1 env)
    n_epochs: int = 10
    batch_size: int = 16384           # minibatch (SB3 default 64 is for 2048-sample rollouts)
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    vf_coef: float = 0.5
    ent_coef: float = 0.0
    max_grad_norm: float = 0.5
    learning_rate: float = 3e-4
    normalize_advantage: bool = True
    reward_clip: float = 1000.0       # |r| cap for the learner only (legitimate rewards are within [-500, 500]); the
                                      # reference env returns finite but astronomically large rewards for cycles next
                                      # to its integrator's stability limit (DESIGN.md 3.3), which would destroy any
                                      # value function; set to 0 to disable
    normalize_reward: bool = True     # learner-side reward scaling, stable-baselines3 VecNormalize(norm_reward=True)
                                      # semantics: r / sqrt(running variance of the discounted return), clipped to
                                      # +-10.  The env's rewards span +-500: un-normalised, the value loss starts at
                                      # 1e5, the critic's gradient dominates the global gradient-norm clip (0.5) and
                                      # the actor's clipped gradient falls below Adam's eps -- the LSTM actor then does
                                      # not move for the first ~15 M env-steps (profiles/README.md, round 1 curve).
                                      # Episode statistics are always reported on the RAW env reward.
    fused_policy: bool = True         # MLP policy on CUDA: the rollout-side forward (both networks, sampling, log-prob,
                                      # clip) is ONE hand-written kernel, salp_mlp_act (csrc/salp_policy.cu); LSTM policy
                                      # on CUDA: both rollout-side LSTM cells run on the tensor cores (csrc/salp_lstm.cu)
    fused_sequence: bool = True       # RecurrentPPO update: both LSTMs over the whole rollout as lstm_seq.LstmSequence
                                      # (two launches per cell, step and direction) instead of nn.LSTMCell stepped T times
    cuda_graphs: bool = False         # MLP PPO on CUDA: replay the whole rollout and each minibatch step as CUDA graphs
    seed: int = 0
    hidden: tuple = (64, 64)
    action_low: tuple = (0.0, 0.0, -1.0)     # the Box of salp_robot_env.py:63-67
    action_high: tuple = (1.0, 1.0, 1.0)


def compute_gae(rewards, values, dones, last_value, gamma, lam):
    """rewards/values/dones: [T, N]; dones[t] = episode ended AT step t (so step t+1 starts a new
    episode).  Returns (advantages, returns), SB3 RolloutBuffer.compute_returns_and_advantage."""
    T = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    last = torch.zeros_like(last_value)
    for t in reversed(range(T)):
        next_value = last_value if t == T - 1 else values[t + 1]
        nonterminal = (~dones[t]).to(rewards.dtype)
        delta = rewards[t] + gamma * next_value * nonterminal - values[t]
        last = delta + gamma * lam * nonterminal * last
        adv[t] = last
    return adv, adv + values


@dataclass
class PPOStats:
    iteration: int = 0
    env_steps: int = 0
    mean_step_reward: float = 0.0
    episodes: int = 0
    mean_episode_return: float = float("nan")
    mean_episode_length: float = float("nan")
    success_rate: float = float("nan")
    approx_kl: float = 0.0
    clip_fraction: float = 0.0
    value_loss: float = 0.0
    policy_loss: float = 0.0
    rollout_seconds: float = 0.0
    update_seconds: float = 0.0
    history: list = field(default_factory=list, repr=False)


class PPO:
    def __init__(self, env, config: PPOConfig | None = None, policy: MlpPolicy | None = None):
        self.env = env
        self.cfg = config or PPOConfig()
        self.device = env.device
        torch.manual_seed(self.cfg.seed)
        self.policy = (policy or MlpPolicy(env.obs_dim, 3, self.cfg.hidden)).to(self.device)
        self.use_graphs = bool(self.cfg.cuda_graphs) and self.device.type == "cuda"
        self.opt = torch.optim.Adam(self.policy.parameters(), lr=self.cfg.learning_rate, eps=1e-5,
                                    capturable=self.use_graphs)
        self.graph_update = self.use_graphs
        self._roll_graph = self._upd_graph = None
        self._roll_calls = self._upd_calls = 0
        self.gen = torch.Generator(device=self.device)
        self._gen_seed = self.cfg.seed + 1          # (+ rank below: shards must not share their exploration noise)
        self.gen.manual_seed(self._gen_seed)
        self.low = torch.tensor(self.cfg.action_low, device=self.device)
        self.high = torch.tensor(self.cfg.action_high, device=self.device)
        self._predict_gen = None                    # stochastic predict(): its own stream, never self.gen
        self._fused = None
        if (self.cfg.fused_policy and self.device.type == "cuda" and isinstance(self.policy, MlpPolicy)
                and tuple(self.cfg.hidden) == (64, 64)):
            import ctypes as C
            from . import _lib
            lib = _lib.load()
            n = env.num_envs
            assert lib.salp_mlp_packed_size(env.obs_dim) == self.policy.packed().numel()
            self._fused = dict(lib=lib, lo=(C.c_float * 3)(*self.cfg.action_low), hi=(C.c_float * 3)(*self.cfg.action_high),
                               a=torch.empty((n, 3), device=self.device), clipped=torch.empty((n, 3), device=self.device),
                               logp=torch.empty(n, device=self.device), v=torch.empty(n, device=self.device), C=C)
        self.obs = env.reset_t()
        n = env.num_envs
        self._ep_ret = torch.zeros(n, device=self.device)
        self._ep_len = torch.zeros(n, device=self.device)
        # running variance of the discounted return (VecNormalize): per-env return accumulator and
        # (count, mean, M2) merged batch-wise on the device (no host round trip, CUDA-graph capturable)
        self._disc_ret = torch.zeros(n, device=self.device, dtype=torch.float64)
        self._ret_stats = torch.tensor([1e-4, 0.0, 1e-4], device=self.device, dtype=torch.float64)
        self.env_steps = 0
        self.iteration = 0
        self.dist_world = 1
        self.global_envs = n        # envs over all ranks: the loop in learn() counts with it so that ranks
        try:                        # holding shards of different sizes still run the same number of iterations
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                self.dist_world = dist.get_world_size()
                g = torch.tensor([n], device=self.device, dtype=torch.int64)
                dist.all_reduce(g)
                self.global_envs = int(g.item())
                for p in self.policy.parameters():          # identical initial weights on every rank
                    dist.broadcast(p.data, src=0)
                self.gen.manual_seed(self._gen_seed + 7919 * dist.get_rank())
                # the minibatch step is captured WITH its NCCL gradient all-reduce (NCCL collectives are
                # capturable); SALP_PPO_GRAPH_ALLREDUCE=0 keeps the multi-GPU update eager
                import os
                if os.environ.get("SALP_PPO_GRAPH_ALLREDUCE", "1") == "0":
                    self.graph_update = False
        except Exception:
            pass

    # ---- rollout ----
    def _alloc_rollout(self):
        env, T, N, dev = self.env, self.cfg.n_steps, self.env.num_envs, self.device
        self._rb = dict(obs=torch.empty((T, N, env.obs_dim), device=dev), act=torch.empty((T, N, 3), device=dev),
                        logp=torch.empty((T, N), device=dev), val=torch.empty((T, N), device=dev),
                        rew=torch.empty((T, N), device=dev), done=torch.empty((T, N), dtype=torch.bool, device=dev),
                        adv=torch.empty((T, N), device=dev), ret=torch.empty((T, N), device=dev),
                        ep=torch.zeros(4, dtype=torch.float64, device=dev), mean_reward=torch.zeros((), device=dev),
                        raw_sum=torch.zeros((), device=dev))

    def _learner_reward(self, raw, done, bootstrap):
        """Reward as the learner sees it: optional VecNormalize-style scaling by the running standard
        deviation of the discounted return (statistics updated in place, device only), the SB3
        time-limit bootstrap gamma * V(terminal_observation) (`bootstrap`, already in the learner's
        units), and the safety clip.  `raw` is the env's reward with non-finite entries zeroed."""
        cfg = self.cfg
        rew = raw
        if cfg.reward_clip > 0:
            rew = raw = raw.clamp(-cfg.reward_clip, cfg.reward_clip)
        if cfg.normalize_reward:
            self._disc_ret.mul_(cfg.gamma).add_(raw.double())
            st = self._ret_stats                       # Chan et al. batch merge of (count, mean, M2)
            nb = float(raw.numel())
            mb = self._disc_ret.mean()
            m2b = (self._disc_ret - mb).pow(2).sum()
            tot = st[0] + nb
            delta = mb - st[1]
            new_mean = st[1] + delta * nb / tot
            new_m2 = st[2] + m2b + delta * delta * st[0] * nb / tot
            st.copy_(torch.stack([tot, new_mean, new_m2]))
            std = (st[2] / st[0]).sqrt().clamp_min(1e-4).float()
            rew = (raw / std).clamp(-10.0, 10.0)
            self._disc_ret.mul_((~done).double())
        return rew + bootstrap

    def _rollout_body(self):
        """T env-steps + GAE, everything in place on persistent device buffers (so that the whole
        body can be captured once and replayed as ONE CUDA graph: policy forward, salp_step and the
        bookkeeping of all T steps, no host round trip)."""
        cfg, env, T, rb = self.cfg, self.env, self.cfg.n_steps, self._rb
        ep = rb["ep"]            # [sum return, sum length, successes, episodes] of the episodes that ended
        ep.zero_()
        rb["raw_sum"].zero_()
        fz = self._fused
        if fz is not None:
            packed = self.policy.packed()             # the weights do not change during a rollout
        for t in range(T):
            if fz is not None:
                # ONE kernel instead of ~20 launches: both networks, sampling, log-prob, Box clip
                noise = torch.randn((env.num_envs, 3), device=self.device, generator=self.gen)
                C = fz["C"]
                rc = fz["lib"].salp_mlp_act(C.c_void_p(packed.data_ptr()), env.obs_dim, C.c_void_p(self.obs.data_ptr()),
                                            C.c_void_p(noise.data_ptr()), env.num_envs, fz["lo"], fz["hi"],
                                            C.c_void_p(fz["a"].data_ptr()), C.c_void_p(fz["clipped"].data_ptr()),
                                            C.c_void_p(fz["logp"].data_ptr()), C.c_void_p(fz["v"].data_ptr()),
                                            C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
                if rc != 0:
                    raise RuntimeError(f"salp_mlp_act failed ({rc})")
                a, logp, v, clipped = fz["a"], fz["logp"], fz["v"], fz["clipped"]
            else:
                a, logp, v = self.policy.act(self.obs, self.gen)
                clipped = torch.minimum(torch.maximum(a, self.low), self.high).float().contiguous()
            rb["obs"][t].copy_(self.obs); rb["act"][t].copy_(a); rb["logp"][t].copy_(logp); rb["val"][t].copy_(v)
            obs, rew, term, trunc, term_obs = env.step_t(clipped)
            done = term | trunc
            timeout = (trunc & ~term).float()
            raw = torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0)       # the env's own reward (Monitor's `r`)
            if cfg.reward_clip > 0:
                raw = raw.clamp(-cfg.reward_clip, cfg.reward_clip)
            with torch.no_grad():                 # SB3: bootstrap truncated episodes with V(terminal_observation)
                rew = self._learner_reward(raw, done, cfg.gamma * self.policy.value(term_obs) * timeout)
            rb["rew"][t].copy_(rew); rb["done"][t].copy_(done); rb["raw_sum"] += raw.sum()
            self._ep_ret += raw
            self._ep_len += 1
            d = done.to(torch.float64)
            ep += torch.stack([(self._ep_ret.double() * d).sum(), (self._ep_len.double() * d).sum(),
                               (term.double() * d).sum(), d.sum()])
            keep = (~done).float()
            self._ep_ret *= keep
            self._ep_len *= keep
            self.obs.copy_(obs)
        with torch.no_grad():
            last_value = self.policy.value(self.obs)
        adv, ret = compute_gae(rb["rew"], rb["val"], rb["done"], last_value, cfg.gamma, cfg.gae_lambda)
        rb["adv"].copy_(adv); rb["ret"].copy_(ret)
        rb["mean_reward"].copy_(rb["raw_sum"] / float(T * env.num_envs))

    def collect(self):
        T, N = self.cfg.n_steps, self.env.num_envs
        if not hasattr(self, "_rb"):
            self._alloc_rollout()
        self._roll_calls += 1
        if self.use_graphs and self._roll_calls >= 2:
            if self._roll_graph is None:          # the first rollout ran eagerly (warm-up); capture now
                g = torch.cuda.CUDAGraph()
                g.register_generator_state(self.gen)
                with torch.cuda.graph(g):
                    self._rollout_body()
                self._roll_graph = g
            self._roll_graph.replay()
        else:
            self._rollout_body()
        self.env_steps += T * N
        rb = self._rb
        flat = lambda x: x.reshape(T * N, *x.shape[2:])  # noqa: E731
        return dict(obs=flat(rb["obs"]), act=flat(rb["act"]), logp=flat(rb["logp"]), val=flat(rb["val"]),
                    adv=flat(rb["adv"]), ret=flat(rb["ret"]), mean_reward=rb["mean_reward"], episodes=rb["ep"])

    # ---- update ----
    def _allreduce_grads(self):
        if self.dist_world == 1:
            return
        import torch.distributed as dist
        grads = [p.grad for p in self.policy.parameters() if p.grad is not None]
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat)                     # ONE bucket: ~40 KB for the 64-64 MLP (latency-bound)
        flat /= self.dist_world
        off = 0
        for g in grads:
            g.copy_(flat[off:off + g.numel()].view_as(g))
            off += g.numel()

    def _minibatch_step(self, roll, idx, stats):
        cfg = self.cfg
        adv = roll["adv"][idx]
        if cfg.normalize_advantage:
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        logp, ent, val = self.policy.evaluate(roll["obs"][idx], roll["act"][idx])
        old = roll["logp"][idx]
        ratio = (logp - old).exp()
        p1, p2 = adv * ratio, adv * ratio.clamp(1 - cfg.clip_range, 1 + cfg.clip_range)
        policy_loss = -torch.minimum(p1, p2).mean()
        value_loss = (roll["ret"][idx] - val).pow(2).mean()
        loss = policy_loss + cfg.vf_coef * value_loss - cfg.ent_coef * ent.mean()
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self._allreduce_grads()
        nn.utils.clip_grad_norm_(self.policy.parameters(), cfg.max_grad_norm)
        self.opt.step()
        with torch.no_grad():                     # statistics stay on the device (one read-back per update)
            lr = logp - old
            stats += torch.stack([((lr.exp() - 1) - lr).mean(), ((ratio - 1).abs() > cfg.clip_range).float().mean(),
                                  value_loss.detach(), policy_loss.detach()])

    def _update_domain(self, roll):
        """(number of items a minibatch is drawn from, items per minibatch): samples for the MLP policy."""
        n = roll["obs"].shape[0]
        return n, min(self.cfg.batch_size, n)

    def update(self, roll):
        cfg = self.cfg
        n, bs = self._update_domain(roll)
        if self.dist_world > 1:       # every rank must issue the same number of gradient all-reduces: uneven
            import torch.distributed as dist      # shards (envs % world != 0) use the smallest shard's count
            t = torch.tensor([n], device=self.device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            n_common = int(t.item())
        else:
            n_common = n
        stats = getattr(self, "_upd_stats", None)
        if stats is None:
            stats = self._upd_stats = torch.zeros(4, device=self.device)
            self._upd_idx = torch.zeros(bs, dtype=torch.long, device=self.device)
        stats.zero_()
        count = 0
        for _ in range(cfg.n_epochs):
            perm = torch.randperm(n, device=self.device, generator=self.gen)
            for s in range(0, n_common - bs + 1, bs):
                self._upd_idx.copy_(perm[s:s + bs])
                self._upd_calls += 1
                if self.graph_update and self._upd_calls > 3:
                    if self._upd_graph is None:   # three eager (real) steps warmed everything up; capture the 4th
                        self.opt.zero_grad(set_to_none=True)
                        g = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(g):
                            self._minibatch_step(roll, self._upd_idx, stats)
                        self._upd_graph = g
                    self._upd_graph.replay()
                else:
                    self._minibatch_step(roll, self._upd_idx, stats)
                count += 1
        kl, clipf, vl, pl = (stats / max(count, 1)).tolist()
        return dict(approx_kl=kl, clip_fraction=clipf, value_loss=vl, policy_loss=pl)

    def allreduce_seconds_per_step(self, reps: int = 50) -> float:
        """Device time of ONE gradient all-reduce of this policy's size (CUDA events, after warm-up):
        multiplied by the optimiser steps of an update it gives the all-reduce share of the update
        (BASELINE.md section 4).  0.0 on one GPU."""
        if self.dist_world == 1:
            return 0.0
        import torch.distributed as dist
        n = sum(p.numel() for p in self.policy.parameters())
        flat = torch.zeros(n, device=self.device)
        for _ in range(5):
            dist.all_reduce(flat)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            dist.all_reduce(flat)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / reps

    def _reduce_stat(self, total, count):
        if self.dist_world > 1:
            import torch.distributed as dist
            t = torch.tensor([total, count], dtype=torch.float64, device=self.device)
            dist.all_reduce(t)                    # rollout statistics: 16 bytes
            total, count = float(t[0]), float(t[1])
        return total / count if count else float("nan"), int(count)

    @property
    def env_steps_global(self) -> int:
        """Env-steps collected over all ranks. Every rank collects the same number of rollouts, so this
        is the same number everywhere even when the shards differ in size."""
        return self.env_steps // self.env.num_envs * self.global_envs

    def learn(self, total_env_steps: int, log=None, eval_env=None, eval_every=0, n_eval_episodes=10) -> PPOStats:
        """Collect and update until env_steps_global >= total_env_steps, one row of statistics per iteration to
        `log`.  With an `eval_env` and `eval_every` > 0, the iteration that reaches the next multiple of
        `eval_every` env-steps runs `evaluate` after its update and its row gains eval_return, eval_success,
        eval_length and eval_seconds (SB3 EvalCallback).  Evaluation leaves the training state untouched."""
        stats = PPOStats()
        next_eval = self.env_steps_global + eval_every if eval_env is not None and eval_every > 0 else None
        while self.env_steps_global < total_env_steps:
            t0 = time.perf_counter()
            roll = self.collect()
            if self.device.type == "cuda":
                torch.cuda.synchronize()
            t1 = time.perf_counter()
            upd = self.update(roll)
            if self.device.type == "cuda":
                torch.cuda.synchronize()
            t2 = time.perf_counter()
            self.iteration += 1
            ep = roll["episodes"].tolist()            # one read-back per iteration
            ne = int(ep[3])
            mean_ret, n_ep = self._reduce_stat(ep[0], ne)
            mean_len, _ = self._reduce_stat(ep[1], ne)
            succ, _ = self._reduce_stat(ep[2], ne)
            mean_rew, _ = self._reduce_stat(float(roll["mean_reward"]), 1)
            row = dict(iteration=self.iteration, env_steps=self.env_steps_global, mean_step_reward=mean_rew,
                       episodes=n_ep, mean_episode_return=mean_ret, mean_episode_length=mean_len, success_rate=succ,
                       rollout_seconds=t1 - t0, update_seconds=t2 - t1, **upd)
            if next_eval is not None and self.env_steps_global >= next_eval:
                t3 = time.perf_counter()
                ev = self.evaluate(eval_env, n_eval_episodes)
                row.update(eval_return=ev["mean_return"], eval_success=ev["success_rate"],
                           eval_length=ev["mean_length"], eval_seconds=time.perf_counter() - t3)
                while next_eval <= self.env_steps_global:
                    next_eval += eval_every
            stats.history.append(row)
            for k, v in row.items():
                setattr(stats, k, v)
            if log:
                log(row)
        return stats

    # ---- inference ----
    def _clip(self, a):
        return torch.minimum(torch.maximum(a, self.low), self.high)

    def _predict_state(self, n, state):
        """The policy state predict() starts from: none for the MLP policy."""
        return None

    def _actor_fn(self, n):
        """The deterministic actor for batches of up to n envs with the weights as they are now (packed once,
        here): f(obs [k, D] contiguous fp32, episode_start [k] bool or None, state) -> (mean, mean clipped to
        the Box).  Buffers are its own, so nothing the rollout or its CUDA graphs read is written.  On CUDA the
        MLP runs as salp_mlp_act in its deterministic mode (no noise, no critic)."""
        fz = self._fused
        if fz is None:
            def f(obs, starts, state):
                mean = self.policy.actor(obs)
                return mean, self._clip(mean)
            return f
        C, lib, D = fz["C"], fz["lib"], self.env.obs_dim
        packed = self.policy.packed()
        mean, clipped = torch.empty((n, 3), device=self.device), torch.empty((n, 3), device=self.device)

        def f(obs, starts, state):
            k = obs.shape[0]
            rc = lib.salp_mlp_act(C.c_void_p(packed.data_ptr()), D, C.c_void_p(obs.data_ptr()), None, k, fz["lo"],
                                  fz["hi"], C.c_void_p(mean.data_ptr()), C.c_void_p(clipped.data_ptr()), None, None,
                                  C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
            if rc != 0:
                raise RuntimeError(f"salp_mlp_act failed ({rc})")
            return mean[:k], clipped[:k]
        return f

    @torch.no_grad()
    def predict(self, obs, state=None, episode_start=None, deterministic=False):
        """stable-baselines3 predict: (actions [N, 3] clipped to the Box, state) for obs [N, obs_dim].  The action
        is the Gaussian mean (deterministic) or a sample drawn from predict's own generator.  `state` and
        `episode_start` matter for RecurrentPPO only (the MLP policy returns state None)."""
        obs = torch.as_tensor(obs, dtype=torch.float32, device=self.device).contiguous()
        if obs.dim() != 2 or obs.shape[1] != self.env.obs_dim:
            raise ValueError(f"obs must be [N, {self.env.obs_dim}]")
        n = obs.shape[0]
        starts = None if episode_start is None else torch.as_tensor(episode_start, dtype=torch.bool,
                                                                     device=self.device).reshape(n).contiguous()
        state = self._predict_state(n, state)
        mean, clipped = self._actor_fn(n)(obs, starts, state)
        if not deterministic:
            if self._predict_gen is None:
                self._predict_gen = torch.Generator(device=self.device)
                self._predict_gen.manual_seed(self.cfg.seed + 2)
            noise = torch.randn(mean.shape, device=self.device, generator=self._predict_gen)
            clipped = self._clip(mean + noise * self.policy.log_std.exp())
        return clipped.clone(), state

    def _shard_span(self, n):
        """(offset of this rank's first env, envs over all ranks) of an eval env sharded over the ranks."""
        if self.dist_world == 1:
            return 0, n
        import torch.distributed as dist
        sizes = [torch.zeros(1, dtype=torch.int64, device=self.device) for _ in range(self.dist_world)]
        dist.all_gather(sizes, torch.tensor([n], dtype=torch.int64, device=self.device))
        sizes = [int(x) for x in sizes]
        return sum(sizes[:dist.get_rank()]), sum(sizes)

    @torch.no_grad()
    def evaluate(self, env, n_episodes=10):
        """Deterministic episodes on `env` (SB3 evaluate_policy(deterministic=True)): env i contributes
        (n_episodes + i) // N episodes; success is `terminated`.  RecurrentPPO starts every env from a zero
        actor state and resets it where an episode ended.  Under torch.distributed each rank steps its shard
        (distributed.make_shard), i counts globally, and every rank returns the same mean_return, mean_length,
        success_rate and episodes.  The env may step up to 15 times past the last recorded episode."""
        n = env.num_envs
        offset, total = self._shard_span(n)
        quotas = (n_episodes + offset + torch.arange(n, device=env.device)) // total
        f, state = self._actor_fn(n), self._predict_state(n, None)
        sums = run_episodes(lambda obs, starts: f(obs.to(self.device).contiguous(), starts, state)[1], env, quotas)
        if self.dist_world > 1:
            import torch.distributed as dist
            dist.all_reduce(sums)
        r, ln, s, e = sums[0].tolist()
        return dict(mean_return=r / e, mean_length=ln / e, success_rate=s / e, episodes=int(e))

    # ---- persistence ----
    def _policy_spec(self):
        p = self.policy
        lstm = getattr(p, "lstm_hidden", None)
        return dict(kind="RecurrentPPO" if lstm else "PPO", obs_dim=self.env.obs_dim, lstm_hidden=lstm,
                    hidden=tuple(m.out_features for m in p.actor if isinstance(m, nn.Linear))[:-1])

    def save(self, path):
        """torch.save (not SB3's zip format) of the policy's state_dict, the Adam state, env_steps (over all
        ranks), iteration, the policy kind and sizes, and per rank the exploration generator state and the
        reward-normalisation statistics.  Under torch.distributed every rank calls it; rank 0 writes."""
        mine = dict(gen=self.gen.get_state(), ret_stats=self._ret_stats.cpu())
        ranks, rank = [mine], 0
        if self.dist_world > 1:
            import torch.distributed as dist
            ranks, rank = [None] * self.dist_world, dist.get_rank()
            dist.all_gather_object(ranks, mine)
        if rank == 0:
            torch.save(dict(spec=self._policy_spec(), policy=self.policy.state_dict(), opt=self.opt.state_dict(),
                            env_steps=self.env_steps_global, iteration=self.iteration, ranks=ranks), path)
        if self.dist_world > 1:
            dist.barrier()

    def load(self, path):
        """Restore what `save` wrote; training then goes on from a reset env, as SB3's learn does after load.
        Parameters are copied in place.  Each rank gets back its own generator state and reward-normalisation
        statistics when the checkpoint was written by as many ranks as there are now; otherwise those keep
        what the constructor set.  Captured CUDA graphs are dropped (the optimiser state they read is
        replaced) and captured again by the next rollout and update.  A checkpoint of another policy kind,
        obs_dim or size raises ValueError."""
        ck = torch.load(path, map_location="cpu", weights_only=False)
        if ck["spec"] != self._policy_spec():
            raise ValueError(f"checkpoint policy {ck['spec']} does not match this one {self._policy_spec()}")
        self.policy.load_state_dict(ck["policy"])
        self.opt.load_state_dict(ck["opt"])
        for g in self.opt.param_groups:           # keep this object's mode, whichever mode wrote the file
            g["capturable"] = self.use_graphs
        for st in self.opt.state.values():
            st["step"] = st["step"].to(self.device) if self.use_graphs else st["step"].cpu()
        ranks = ck["ranks"]
        if len(ranks) == self.dist_world:
            import torch.distributed as dist
            mine = ranks[dist.get_rank() if self.dist_world > 1 else 0]
            self.gen.set_state(mine["gen"])
            self._ret_stats.copy_(mine["ret_stats"])
        self.env_steps = ck["env_steps"] * self.env.num_envs // self.global_envs
        self.iteration = ck["iteration"]
        self._roll_graph = self._upd_graph = None
        self._roll_calls = self._upd_calls = 0
        self.opt.zero_grad(set_to_none=True)
        self._reset_rollout_state()

    def _reset_rollout_state(self):
        """A reset env and zeroed per-env episode state (what SB3's learn starts from after load)."""
        self.obs.copy_(self.env.reset_t())
        self._ep_ret.zero_()
        self._ep_len.zero_()
        self._disc_ret.zero_()


# ------------------------------------------------------------------------------------------------
# RecurrentPPO (sb3_contrib MlpLstmPolicy as configured by src/train_robot_recurrent_ppo.py:85-107)
# ------------------------------------------------------------------------------------------------
class LstmPolicy(nn.Module):
    """lstm_hidden_size = 256, n_lstm_layers = 1, shared_lstm = False, enable_critic_lstm = True
    (train_robot_recurrent_ppo.py:100-105): separate actor / critic LSTMs on the flattened
    observation, each followed by the default 64-64 tanh MLP and a linear head."""

    def __init__(self, obs_dim=10, act_dim=3, lstm_hidden=256, hidden=(64, 64), log_std_init=0.0):
        super().__init__()
        self.lstm_hidden = lstm_hidden
        self.lstm_actor = nn.LSTMCell(obs_dim, lstm_hidden)
        self.lstm_critic = nn.LSTMCell(obs_dim, lstm_hidden)
        self.actor = _mlp(lstm_hidden, hidden, act_dim, 0.01)
        self.critic = _mlp(lstm_hidden, hidden, 1, 1.0)
        self.log_std = nn.Parameter(torch.full((act_dim,), float(log_std_init)))

    def initial_state(self, n, device):
        z = lambda: torch.zeros(n, self.lstm_hidden, device=device)  # noqa: E731
        return (z(), z(), z(), z())

    def step(self, obs, state, starts):
        """One time step.  starts [N] (bool / 0-1): the env began a new episode at this step, so
        its hidden state is reset first (sb3_contrib _process_sequence)."""
        keep = (1.0 - starts.float()).unsqueeze(-1)
        ha, ca, hc, cc = state
        ha, ca = self.lstm_actor(obs, (ha * keep, ca * keep))
        hc, cc = self.lstm_critic(obs, (hc * keep, cc * keep))
        return self.actor(ha), self.critic(hc).squeeze(-1), (ha, ca, hc, cc)

    def peek_value(self, obs, state):
        hc, _ = self.lstm_critic(obs, (state[2], state[3]))
        return self.critic(hc).squeeze(-1)

    def sequence(self, obs, state, starts):
        """The T steps of `step` at once for the learner: obs [T, B, D], starts [T, B] -> (mean [T, B, A],
        value [T, B]).  Both LSTMs run side by side as ONE lstm_seq.LstmSequence (one batched GEMM + one hand-written
        element-wise kernel per step and direction; input projection and weight gradients batched over T x B),
        the 64-64 heads once on the stacked hidden states."""
        from .lstm_seq import lstm_sequence
        T, B = starts.shape
        keep = 1.0 - starts.float()
        ha, hc = lstm_sequence([self.lstm_actor, self.lstm_critic], obs, [state[0], state[2]], [state[1], state[3]], keep)
        mean = self.actor(ha.reshape(T * B, -1)).view(T, B, -1)
        val = self.critic(hc.reshape(T * B, -1)).view(T, B)
        return mean, val


class RecurrentPPO(PPO):
    """PPO with the LSTM policy.  Rollouts carry the per-env LSTM state (reset on done); the
    update replays whole [T, envs] sequences from the stored initial state, so back-propagation
    through time spans the rollout (n_steps) with resets at episode starts.  Minibatches are
    subsets of envs (`batch_size` samples = batch_size // n_steps env sequences)."""

    def __init__(self, env, config: PPOConfig | None = None, policy: LstmPolicy | None = None):
        cfg = config or PPOConfig(n_steps=32, batch_size=32 * 512)
        if policy is None:
            torch.manual_seed(cfg.seed)           # (the base class seeds only after its arguments are built)
            policy = LstmPolicy(env.obs_dim, 3, hidden=cfg.hidden)
        super().__init__(env, cfg, policy)
        self.state = self.policy.initial_state(env.num_envs, self.device)
        self.starts = torch.ones(env.num_envs, dtype=torch.bool, device=self.device)
        # rollout-side LSTM cells on the tensor cores (csrc/salp_lstm.cu): gate GEMM in bf16 with tcgen05,
        # cell update fused behind it; the learner keeps the fp32 torch cells (autograd)
        self._lstm_fused = None
        if (cfg.fused_policy and self.device.type == "cuda" and self.policy.lstm_hidden == 256
                and env.obs_dim <= 64):
            from .lstm import LstmCellB200
            n = env.num_envs
            self._lstm_fused = dict(actor=LstmCellB200(self.policy.lstm_actor, n), critic=LstmCellB200(self.policy.lstm_critic, n),
                                    h=torch.empty((n, 256), device=self.device), c=torch.empty((n, 256), device=self.device))
        self._eval_cell = None      # predict / evaluate's own actor cell: the rollout graph reads the rollout cells

    def _predict_state(self, n, state):
        """The actor LSTM's (h, c) predict() starts from: zeros, or a contiguous copy of the caller's."""
        if state is None:
            return tuple(torch.zeros(n, self.policy.lstm_hidden, device=self.device) for _ in range(2))
        return tuple(torch.as_tensor(x, dtype=torch.float32, device=self.device).reshape(n, -1).clone(
            memory_format=torch.contiguous_format) for x in state)

    def _actor_fn(self, n):
        """As PPO._actor_fn for the actor LSTM and its head (sb3_contrib predict: the critic LSTM is not run);
        `state` = (h, c) is advanced in place, rows with episode_start reset first.  On CUDA the cell is an
        LstmCellB200 of this function's own, built for up to n envs and packed here."""
        actor = self.policy.actor
        if self._lstm_fused is None:
            cell = self.policy.lstm_actor

            def f(obs, starts, state):
                h, c = state
                if starts is not None:
                    keep = (1.0 - starts.float()).unsqueeze(-1)
                    h2, c2 = cell(obs, (h * keep, c * keep))
                else:
                    h2, c2 = cell(obs, (h, c))
                h.copy_(h2)
                c.copy_(c2)
                mean = actor(h)
                return mean, self._clip(mean)
            return f
        from .lstm import LstmCellB200
        if self._eval_cell is None or self._eval_cell.n < n:
            self._eval_cell = LstmCellB200(self.policy.lstm_actor, n)
        cell = self._eval_cell
        cell.pack()

        def f(obs, starts, state):
            cell.step(obs, starts, *state)
            mean = actor(state[0])
            return mean, self._clip(mean)
        return f

    def _reset_rollout_state(self):
        super()._reset_rollout_state()
        for x in self.state:
            x.zero_()
        self.starts.fill_(True)

    def load(self, path):
        super().load(path)
        if self._lstm_fused is not None:
            self._lstm_fused["actor"].pack()
            self._lstm_fused["critic"].pack()

    def _policy_step(self, obs, starts):
        """One rollout step of the policy on self.state (updated in place): (action mean, value)."""
        fz = self._lstm_fused
        if fz is None:
            mean, v, new_state = self.policy.step(obs, self.state, starts)
            for dst, src in zip(self.state, new_state):
                dst.copy_(src)
            return mean, v
        ha, ca, hc, cc = self.state
        fz["actor"].step(obs, starts, ha, ca)
        fz["critic"].step(obs, starts, hc, cc)
        return self.policy.actor(ha), self.policy.critic(hc).squeeze(-1)

    def _peek_value(self, obs, starts=None):
        """V(obs) from the critic's current state WITHOUT advancing it (bootstrap values)."""
        fz = self._lstm_fused
        if fz is None:
            if starts is None:
                return self.policy.peek_value(obs, self.state)
            return self.policy.step(obs, self.state, starts)[1]
        h, _ = fz["critic"].step(obs.contiguous(), starts, self.state[2], self.state[3], fz["h"], fz["c"])
        return self.policy.critic(h).squeeze(-1)

    def _alloc_rollout(self):
        super()._alloc_rollout()
        T, N, dev = self.cfg.n_steps, self.env.num_envs, self.device
        self._rb["starts"] = torch.empty((T, N), dtype=torch.bool, device=dev)
        self._rb["init_state"] = tuple(torch.empty_like(s) for s in self.state)

    def _rollout_body(self):
        """As PPO._rollout_body, carrying the per-env LSTM state in place (reset at episode starts);
        capturable as one CUDA graph: both LSTM cells, the heads, salp_step and the bookkeeping of
        all T steps."""
        cfg, env, T, rb = self.cfg, self.env, self.cfg.n_steps, self._rb
        for dst, src in zip(rb["init_state"], self.state):
            dst.copy_(src)
        ep = rb["ep"]
        ep.zero_()
        rb["raw_sum"].zero_()
        if self._lstm_fused is not None:                # the weights do not change during a rollout
            self._lstm_fused["actor"].pack()
            self._lstm_fused["critic"].pack()
        for t in range(T):
            with torch.no_grad():
                mean, v = self._policy_step(self.obs, self.starts)
                noise = torch.randn(mean.shape, device=self.device, generator=self.gen)
                a = mean + noise * self.policy.log_std.exp()
                logp = (-0.5 * noise.pow(2) - self.policy.log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
            rb["obs"][t].copy_(self.obs); rb["act"][t].copy_(a); rb["logp"][t].copy_(logp); rb["val"][t].copy_(v)
            rb["starts"][t].copy_(self.starts)
            clipped = torch.minimum(torch.maximum(a, self.low), self.high).float().contiguous()
            obs, rew, term, trunc, term_obs = env.step_t(clipped)
            done = term | trunc
            timeout = (trunc & ~term).float()
            raw = torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0)
            if cfg.reward_clip > 0:
                raw = raw.clamp(-cfg.reward_clip, cfg.reward_clip)
            with torch.no_grad():
                rew = self._learner_reward(raw, done, cfg.gamma * self._peek_value(term_obs) * timeout)
            rb["rew"][t].copy_(rew); rb["done"][t].copy_(done); rb["raw_sum"] += raw.sum()
            self._ep_ret += raw
            self._ep_len += 1
            d = done.to(torch.float64)
            ep += torch.stack([(self._ep_ret.double() * d).sum(), (self._ep_len.double() * d).sum(),
                               (term.double() * d).sum(), d.sum()])
            keep = (~done).float()
            self._ep_ret *= keep
            self._ep_len *= keep
            self.obs.copy_(obs)
            self.starts.copy_(done)
        with torch.no_grad():
            last_value = self._peek_value(self.obs, self.starts)
        adv, ret = compute_gae(rb["rew"], rb["val"], rb["done"], last_value, cfg.gamma, cfg.gae_lambda)
        rb["adv"].copy_(adv); rb["ret"].copy_(ret)
        rb["mean_reward"].copy_(rb["raw_sum"] / float(T * env.num_envs))

    def collect(self):
        """Rollout buffers keep their [T, envs] shape (the update replays env sequences)."""
        if not hasattr(self, "_rb"):
            self._alloc_rollout()
        self._roll_calls += 1
        if self.use_graphs and self._roll_calls >= 2:
            if self._roll_graph is None:          # the first rollout ran eagerly (warm-up); capture now
                g = torch.cuda.CUDAGraph()
                g.register_generator_state(self.gen)
                with torch.cuda.graph(g):
                    self._rollout_body()
                self._roll_graph = g
            self._roll_graph.replay()
        else:
            self._rollout_body()
        self.env_steps += self.cfg.n_steps * self.env.num_envs
        rb = self._rb
        return dict(obs=rb["obs"], act=rb["act"], logp=rb["logp"], val=rb["val"], adv=rb["adv"], ret=rb["ret"],
                    starts=rb["starts"], init_state=rb["init_state"], mean_reward=rb["mean_reward"], episodes=rb["ep"])

    def _update_domain(self, roll):
        """Minibatches are subsets of ENVS: whole [T] sequences, batch_size // T of them."""
        T, N = roll["logp"].shape
        return N, max(1, min(N, self.cfg.batch_size // T))

    def _minibatch_step(self, roll, idx, stats):
        """One optimiser step on the env sequences `idx`: BPTT over the rollout from the stored
        initial LSTM state, hidden state reset at episode starts.  No host synchronisation, so it
        can be captured and replayed as a CUDA graph like the MLP step."""
        cfg = self.cfg
        T = roll["logp"].shape[0]
        state = tuple(x[idx] for x in roll["init_state"])
        obs, starts = roll["obs"][:, idx], roll["starts"][:, idx]
        if cfg.fused_sequence:
            mean, val = self.policy.sequence(obs, state, starts)
        else:
            means, vals = [], []
            for t in range(T):
                m, v, state = self.policy.step(obs[t], state, starts[t])
                means.append(m)
                vals.append(v)
            mean, val = torch.stack(means), torch.stack(vals)
        log_std = self.policy.log_std
        z = (roll["act"][:, idx] - mean) * (-log_std).exp()
        logp = (-0.5 * z.pow(2) - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)
        entropy = (0.5 + 0.5 * math.log(2 * math.pi) + log_std).sum()
        old_logp = roll["logp"][:, idx]
        adv = roll["adv"][:, idx]
        if cfg.normalize_advantage:
            adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        ratio = (logp - old_logp).exp()
        policy_loss = -torch.minimum(adv * ratio, adv * ratio.clamp(1 - cfg.clip_range, 1 + cfg.clip_range)).mean()
        value_loss = (roll["ret"][:, idx] - val).pow(2).mean()
        loss = policy_loss + cfg.vf_coef * value_loss - cfg.ent_coef * entropy
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        self._allreduce_grads()
        nn.utils.clip_grad_norm_(self.policy.parameters(), cfg.max_grad_norm)
        self.opt.step()
        with torch.no_grad():
            lr = logp - old_logp
            stats += torch.stack([((lr.exp() - 1) - lr).mean(), ((ratio - 1).abs() > cfg.clip_range).float().mean(),
                                  value_loss.detach(), policy_loss.detach()])
