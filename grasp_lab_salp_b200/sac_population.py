"""A population of K SAC agents trained side by side in one process: seeds and hyper-parameter sweeps of
``sac.SAC`` for the wall time of roughly one run.

``SACPopulation(env, configs)`` trains K = len(configs) agents on one env of K n envs; agent k owns env rows
[k n, (k + 1) n).  Every agent keeps SAC's semantics exactly as ``sac.py`` restates them from
stable-baselines3: warm-up, learning_starts, the per-step order of updates, effective done = `terminated`,
the learner-side reward clip and a ring of buffer_size // n slots.  num_timesteps counts one agent's
env-steps (n per vec step), as in ``SAC``.

Per agent: seed, learning_rate, gamma, tau, target_entropy and ent_coef ("auto" for every agent, or a float
per agent).  Every other SACConfig field is shared and must be equal across configs.

The weights of the K agents are stacked on a leading dimension ([K, out, in] and [K, out]) and every forward
pass is a batched GEMM over it, so one gradient step launches the same kernels whatever K is.  Losses are
per-agent means; their sum is back-propagated, and since the parameter sets are disjoint agent k's gradient is
exactly its own.  ``_StackedAdam`` is torch.optim.Adam per agent with that agent's learning rate.  Rollouts go
through one salp_sac_act_grouped launch per vec step (CUDA, ``fused_actor``).

Agent k's networks start bit-identical to those of ``SAC(env_k, SACConfig(seed=s_k))``.  Randomness is drawn
by one population generator for actions ([K n, 3] at a time) and one for training ([K, B, ...]), so a member
is statistically, not bitwise, the same as a standalone run with its seed.  The replay is one slot-major ring
[S, K n, ...], filled by SAC's zero-copy ``step_device(out=...)`` path, CUDA-graph path or host path
unchanged; the collection loop and the driver (``learn``) are SAC's.
"""
from __future__ import annotations

import collections
import dataclasses
import math

import torch
import torch.nn.functional as F

from .sac import (LOG_STD_MAX, LOG_STD_MIN, SAC, SacActor, SacActorGroupB200, SACConfig, SacCritic,
                  _refuse_multi_rank)

PER_AGENT = ("seed", "learning_rate", "gamma", "tau", "target_entropy", "ent_coef")
BETA1, BETA2, ADAM_EPS = 0.9, 0.999, 1e-8         # torch.optim.Adam's defaults


def _linear(x, w, b):
    """x [K, B, in], w [K, out, in], b [K, out] -> [K, B, out]: K nn.Linear in one batched GEMM."""
    return torch.baddbmm(b.unsqueeze(1), x, w.transpose(1, 2))


def _per_agent(values, like):
    """values [K] broadcast to the shape of each [K, ...] tensor in `like` (materialised: foreach fast path)."""
    return [values.reshape((-1,) + (1,) * (t.dim() - 1)).expand_as(t).contiguous() for t in like]


class _StackedAdam:
    """torch.optim.Adam with its defaults over parameters stacked [K, ...], learning rate lr[k] for agent k.
    All agents step together, so the step count and the bias corrections are shared and only the step size
    is per agent.  Device-side (CUDA-graph capturable), with a launch count that does not depend on K."""

    def __init__(self, params, lr):
        self.params = params
        self.lr = _per_agent(lr, params)
        self.exp_avg = [torch.zeros_like(p) for p in params]
        self.exp_avg_sq = [torch.zeros_like(p) for p in params]
        self.step_t = torch.zeros((), device=params[0].device)

    def zero_grad(self, set_to_none=True):
        for p in self.params:
            p.grad = None

    @torch.no_grad()
    def step(self):
        grads = [p.grad for p in self.params]
        self.step_t += 1
        torch._foreach_lerp_(self.exp_avg, grads, 1 - BETA1)
        torch._foreach_mul_(self.exp_avg_sq, BETA2)
        torch._foreach_addcmul_(self.exp_avg_sq, grads, grads, 1 - BETA2)
        bc1 = 1 - torch.pow(BETA1, self.step_t)
        bc2_sqrt = torch.sqrt(1 - torch.pow(BETA2, self.step_t))
        denom = torch._foreach_sqrt(self.exp_avg_sq)
        torch._foreach_div_(denom, bc2_sqrt)
        torch._foreach_add_(denom, ADAM_EPS)
        update = torch._foreach_div(self.exp_avg, denom)
        torch._foreach_mul_(update, self.lr)
        torch._foreach_div_(update, bc1)
        torch._foreach_sub_(self.params, update)

    def torch_state_dict(self, k, params_k, lr, capturable):
        """Agent k's state as the state_dict of a torch.optim.Adam(params_k, lr) (what SAC.save writes)."""
        opt = torch.optim.Adam(params_k, lr=lr, capturable=capturable)
        for p, m, v in zip(params_k, self.exp_avg, self.exp_avg_sq):
            opt.state[p] = dict(step=torch.tensor(float(self.step_t)), exp_avg=m[k].detach().reshape(p.shape).clone(),
                                exp_avg_sq=v[k].detach().reshape(p.shape).clone())
        return opt.state_dict()


class SACPopulation(SAC):
    def __init__(self, env, configs: list[SACConfig]):
        configs = list(configs)
        K = len(configs)
        if K < 1:
            raise ValueError("a population needs at least one config")
        c0 = configs[0]
        for f in dataclasses.fields(SACConfig):
            if f.name not in PER_AGENT and any(getattr(c, f.name) != getattr(c0, f.name) for c in configs):
                raise ValueError(f"SACConfig.{f.name} must be equal across the population (only "
                                 f"{', '.join(PER_AGENT)} may differ per agent)")
        auto = [isinstance(c.ent_coef, str) for c in configs]
        if any(auto) and not (all(auto) and all(c.ent_coef == "auto" for c in configs)):
            raise ValueError("ent_coef must be 'auto' for every agent or a float for every agent")
        if env.num_envs % K:
            raise ValueError(f"env.num_envs ({env.num_envs}) must be a multiple of the population size ({K})")
        _refuse_multi_rank("SACPopulation")
        self.env, self.configs = env, configs
        self.cfg = cfg = c0                       # (SAC's methods read only its shared fields)
        self.device = dev = env.device
        N, D = env.num_envs, env.obs_dim
        self.num_agents, self.n_total, self.n_envs, self.obs_dim = K, N, N // K, D
        actors, critics = [], []
        for c in configs:                         # SAC's construction order, agent by agent
            torch.manual_seed(c.seed)
            actors.append(SacActor(D))
            critics.append(SacCritic(D))
        self._actor_names = [k for k, _ in actors[0].named_parameters()]
        self._critic_names = [k for k, _ in critics[0].named_parameters()]

        def stack(mods):
            return [torch.stack([p.detach() for p in ps]).to(dev) for ps in zip(*(m.parameters() for m in mods))]
        self.actor_params = [p.requires_grad_(True) for p in stack(actors)]
        self.critic_params = [p.requires_grad_(True) for p in stack(critics)]
        self.target_params = [p.detach().clone() for p in self.critic_params]
        cuda = dev.type == "cuda"
        self.use_graphs = bool(cfg.cuda_graphs) and cuda

        def per_agent(name):
            return torch.tensor([float(getattr(c, name)) for c in configs], device=dev)
        self.lr, self.gamma, self.target_entropy = per_agent("learning_rate"), per_agent("gamma"), per_agent("target_entropy")
        self.tau = per_agent("tau")
        self._tau = _per_agent(self.tau, self.target_params)
        self._keep = _per_agent(torch.tensor([1.0 - c.tau for c in configs], device=dev), self.target_params)
        self.actor_opt = _StackedAdam(self.actor_params, self.lr)
        self.critic_opt = _StackedAdam(self.critic_params, self.lr)
        self.auto_ent = all(auto)
        if self.auto_ent:
            self.log_ent_coef = torch.zeros(K, device=dev, requires_grad=True)     # log 1
            self.ent_opt = _StackedAdam([self.log_ent_coef], self.lr)
        else:
            self.log_ent_coef = None
            self.ent_coef_tensor = per_agent("ent_coef")
        self.fused = None
        if cfg.fused_actor and cuda and D <= 64:
            self.fused = SacActorGroupB200(self.actor_params, cfg.action_low, cfg.action_high)
        # SAC's collection state on one ring of S slots of K n envs (each agent's ring is its n columns), with
        # per-agent statistics; the generators are seeded from the first config
        self._init_collection(max(1, cfg.buffer_size // self.n_envs), per_agent=(K,))

    # ---- networks over the agent dimension ----
    def _actor(self, obs):
        """obs [K, B, D] -> (mu, clamped log_std) [K, B, 3]"""
        w1, b1, w2, b2, w_mu, b_mu, w_ls, b_ls = self.actor_params
        latent = F.relu(_linear(F.relu(_linear(obs, w1, b1)), w2, b2))
        return _linear(latent, w_mu, b_mu), torch.clamp(_linear(latent, w_ls, b_ls), LOG_STD_MIN, LOG_STD_MAX)

    def _action_log_prob(self, obs, eps):
        """SacActor.action_log_prob over [K, B, ...]: actions [K, B, 3], log-prob [K, B]."""
        mean, log_std = self._actor(obs)
        std = torch.ones_like(mean) * log_std.exp()
        u = mean + eps * std
        a = torch.tanh(u)
        logp = (-((u - mean) ** 2) / (2 * std ** 2) - std.log() - math.log(math.sqrt(2 * math.pi))).sum(dim=-1)
        logp = logp - torch.sum(torch.log(1 - a ** 2 + 1e-6), dim=-1)
        return a, logp

    @staticmethod
    def _critic(params, obs, actions):
        """The two Q-nets of `params` (critic or target) -> ([K, B, 1], [K, B, 1])"""
        x = torch.cat([obs, actions], dim=-1)
        qs = []
        for i in range(0, len(params), 6):
            w1, b1, w2, b2, w3, b3 = params[i:i + 6]
            qs.append(_linear(F.relu(_linear(F.relu(_linear(x, w1, b1)), w2, b2)), w3, b3))
        return tuple(qs)

    # ---- acting ----
    def _policy_act(self, obs, env_out, scaled_out, deterministic=False, generator=None):
        """Actor forward of agent k on rows [k m, (k + 1) m) of obs [K m, D] (grouped kernel or torch)."""
        noise = None if deterministic else torch.randn((obs.shape[0], 3), device=self.device, generator=generator)
        if self.fused is not None:
            self.fused.act(obs, noise, env_out, scaled_out)
            return
        with torch.no_grad():
            K = self.num_agents
            mean, log_std = self._actor(obs.reshape(K, -1, self.obs_dim))
            u = mean if noise is None else mean + noise.view(K, -1, 3) * log_std.exp()
            a = torch.tanh(u).reshape(-1, 3)
            scaled_out.copy_(a)
            env_out.copy_(self.low + (a + 1.0) * 0.5 * (self.high - self.low))

    def _random_act(self, env_out, scaled_out):
        u = torch.rand((self.n_total, 3), device=self.device, generator=self.gen_act)
        a_env = self.low + u * (self.high - self.low)
        env_out.copy_(a_env)
        scaled_out.copy_(2.0 * ((a_env - self.low) / (self.high - self.low)) - 1.0)

    # ---- collection ----
    def _bookkeep(self, rew, term, trunc):
        raw = torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0)
        if self.cfg.reward_clip > 0:
            raw = raw.clamp(-self.cfg.reward_clip, self.cfg.reward_clip)
        term, trunc = term.bool(), trunc.bool()
        done = term | trunc
        self._ep_ret += raw
        self._ep_len += 1
        d = done.to(torch.float64)
        per_env = torch.stack([self._ep_ret.double() * d, self._ep_len.double() * d, term.double() * d, d], dim=1)
        self._ep += per_env.view(self.num_agents, -1, 4).sum(1)
        keep = (~done).float()
        self._ep_ret *= keep
        self._ep_len *= keep

    # ---- learning ----
    def sample(self, batch_size):
        """`batch_size` transitions per agent ([K, B, ...]): uniform over (slot, env of that agent) among the
        complete slots; once the ring has wrapped the slot being filled is skipped.  Device-side."""
        S, N, n, K, dev, g = self.slots, self.n_total, self.n_envs, self.num_agents, self.device, self.gen_train
        pos, full = self._pos_t, self._full_t
        count = torch.where(full, torch.full_like(pos, S - 1), pos)
        start = torch.where(full, pos + 1, torch.zeros_like(pos))
        u = torch.rand((K, batch_size), device=dev, generator=g, dtype=torch.float64)
        slot = (start + torch.minimum((u * count).long(), count - 1)) % S
        env = torch.minimum((torch.rand((K, batch_size), device=dev, generator=g, dtype=torch.float64) * n).long(),
                            torch.full_like(slot, n - 1))
        env = env + torch.arange(K, device=dev).unsqueeze(1) * n
        idx = slot * N + env
        rb = self.rb
        rew = torch.nan_to_num(rb["rew"].view(-1)[idx], nan=0.0, posinf=0.0, neginf=0.0)
        if self.cfg.reward_clip > 0:
            rew = rew.clamp(-self.cfg.reward_clip, self.cfg.reward_clip)
        return dict(obs=rb["obs"].view(S * N, -1)[idx], actions=rb["act"].view(S * N, -1)[idx],
                    next_obs=rb["next_obs"].view(S * N, -1)[idx], rewards=rew.unsqueeze(-1),
                    dones=rb["done"].view(-1)[idx].float().unsqueeze(-1), slot=slot, env=env)

    def train_step(self, batch=None, eps=None):
        """One SB3 gradient step of every agent.  `batch` (dict of obs, actions, next_obs [K, B, .], rewards and
        dones [K, B, 1]) and `eps` (the noise of the two actor samples, [K, B, 3] each) are drawn here unless
        given.  Returns per-agent [K] losses."""
        cfg, K = self.cfg, self.num_agents
        if batch is None:
            batch = self.sample(cfg.batch_size)
        B = batch["obs"].shape[1]
        if eps is None:
            eps = (torch.randn((K, B, 3), device=self.device, generator=self.gen_train),
                   torch.randn((K, B, 3), device=self.device, generator=self.gen_train))
        actions_pi, log_prob = self._action_log_prob(batch["obs"], eps[0])
        log_prob = log_prob.unsqueeze(-1)
        if self.auto_ent:
            ent_coef = torch.exp(self.log_ent_coef.detach())
            ent_coef_loss = -(self.log_ent_coef.view(K, 1, 1)
                              * (log_prob + self.target_entropy.view(K, 1, 1)).detach()).mean((1, 2))
            self.ent_opt.zero_grad()
            ent_coef_loss.sum().backward()
            self.ent_opt.step()
        else:
            ent_coef = self.ent_coef_tensor
        alpha = ent_coef.view(K, 1, 1)
        with torch.no_grad():
            next_actions, next_log_prob = self._action_log_prob(batch["next_obs"], eps[1])
            next_q_values = torch.cat(self._critic(self.target_params, batch["next_obs"], next_actions), dim=-1)
            next_q_values, _ = torch.min(next_q_values, dim=-1, keepdim=True)
            next_q_values = next_q_values - alpha * next_log_prob.unsqueeze(-1)
            target_q_values = batch["rewards"] + (1 - batch["dones"]) * self.gamma.view(K, 1, 1) * next_q_values
        current_q_values = self._critic(self.critic_params, batch["obs"], batch["actions"])
        critic_loss = 0.5 * sum(((q - target_q_values) ** 2).mean((1, 2)) for q in current_q_values)
        self.critic_opt.zero_grad()
        critic_loss.sum().backward()
        self.critic_opt.step()
        q_values_pi = torch.cat(self._critic(self.critic_params, batch["obs"], actions_pi), dim=-1)
        min_qf_pi, _ = torch.min(q_values_pi, dim=-1, keepdim=True)
        actor_loss = (alpha * log_prob - min_qf_pi).mean((1, 2))
        self.actor_opt.zero_grad()
        actor_loss.sum().backward()
        self.actor_opt.step()
        self._train_calls += 1
        if (self._train_calls - 1) % cfg.target_update_interval == 0:
            with torch.no_grad():
                torch._foreach_mul_(self.target_params, self._keep)
                torch._foreach_addcmul_(self.target_params, self.critic_params, self._tau)
        with torch.no_grad():
            mean_q = torch.stack([q.mean((1, 2)) for q in current_q_values]).mean(0)
            self._train_stats += torch.stack([critic_loss.detach(), actor_loss.detach(), ent_coef, mean_q,
                                              torch.ones(K, device=self.device)], dim=1)
        return dict(critic_loss=critic_loss, actor_loss=actor_loss, ent_coef=ent_coef,
                    ent_coef_loss=ent_coef_loss if self.auto_ent else None)

    # ---- driver (SAC.learn) ----
    def _row(self, collect_s, train_s, ev):
        ep, ts = self._ep.tolist(), self._train_stats.tolist()
        self._ep.zero_()
        self._train_stats.zero_()
        nan = float("nan")

        def ratio(rows, i, j):
            return [r[i] / r[j] if r[j] else nan for r in rows]
        row = dict(env_steps=self.num_timesteps, gradient_steps=self.gradient_steps_done,
                   ent_coef=ratio(ts, 2, 4), critic_loss=ratio(ts, 0, 4), actor_loss=ratio(ts, 1, 4),
                   mean_q=ratio(ts, 3, 4), episodes=[int(e[3]) for e in ep], mean_episode_return=ratio(ep, 0, 3),
                   mean_episode_length=ratio(ep, 1, 3), success_rate=ratio(ep, 2, 3), collect_seconds=collect_s,
                   train_seconds=train_s)
        if ev:
            row.update(eval_return=ev["mean_return"], eval_success=ev["success_rate"], eval_length=ev["mean_length"])
        return row

    @torch.no_grad()
    def evaluate(self, env, n_episodes=10):
        """Deterministic episodes on an eval env of K m envs, agent k acting on rows [k m, (k + 1) m) with
        SB3's per-env quota within its slice (env i of a slice contributes (n_episodes + i) // m episodes, as
        SAC.evaluate).  Per-agent lists of mean_return, mean_length, success_rate and episodes."""
        K, N = self.num_agents, env.num_envs
        if N % K:
            raise ValueError(f"the eval env's num_envs ({N}) must be a multiple of the population size ({K})")
        m, dev = N // K, env.device
        targets = ((n_episodes + torch.arange(m, device=dev)) // m).repeat(K)
        counts = torch.zeros(N, dtype=torch.long, device=dev)
        sums = torch.zeros((K, 4), dtype=torch.float64, device=dev)        # return, length, successes, episodes
        cur_r = torch.zeros(N, dtype=torch.float64, device=dev)
        cur_l = torch.zeros(N, dtype=torch.float64, device=dev)
        obs = env.reset_t()
        step = 0
        while step % 16 or bool((counts < targets).any()):                # (a finished env records nothing more)
            a = self.predict(obs.float(), deterministic=True)
            obs, rew, term, trunc, _ = env.step_t(a)
            t = term.bool()
            d = t | trunc.bool()
            cur_r += torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0).double()
            cur_l += 1
            rec = d & (counts < targets)
            w = rec.double()
            sums += torch.stack([cur_r * w, cur_l * w, t.double() * w, w], dim=1).view(K, m, 4).sum(1)
            counts += rec.long()
            cur_r.masked_fill_(d, 0.0)
            cur_l.masked_fill_(d, 0.0)
            step += 1
        s = sums.tolist()
        return dict(mean_return=[x[0] / x[3] for x in s], mean_length=[x[1] / x[3] for x in s],
                    success_rate=[x[2] / x[3] for x in s], episodes=[int(x[3]) for x in s])

    # ---- persistence ----
    def save_agent(self, k, path):
        """Agent k in SAC.save's format: ``SAC(env, configs[k]).load(path)`` gives that agent back."""
        cuda, lr = self.device.type == "cuda", self.configs[k].learning_rate

        def state(names, params):
            return collections.OrderedDict((name, p[k].detach().clone()) for name, p in zip(names, params))
        actor, critic = state(self._actor_names, self.actor_params), state(self._critic_names, self.critic_params)
        target = state(self._critic_names, self.target_params)
        log_ent = None if self.log_ent_coef is None else self.log_ent_coef[k:k + 1].detach().cpu()
        ent_opt = None
        if self.auto_ent:
            ent_opt = self.ent_opt.torch_state_dict(k, [self.log_ent_coef[k:k + 1].detach().clone()], lr, cuda)
        torch.save(dict(actor=actor, critic=critic, critic_target=target, log_ent_coef=log_ent,
                        actor_opt=self.actor_opt.torch_state_dict(k, list(actor.values()), lr, cuda),
                        critic_opt=self.critic_opt.torch_state_dict(k, list(critic.values()), lr, cuda),
                        ent_opt=ent_opt, num_timesteps=self.num_timesteps), path)

    def save(self, path):
        raise NotImplementedError("save one member with save_agent(k, path)")

    def load(self, path):
        raise NotImplementedError("a population has no single-agent load; SAC(env, configs[k]).load(path) loads a "
                                  "member saved with save_agent")
