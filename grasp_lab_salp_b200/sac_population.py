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
is statistically, not bitwise, the same as a standalone run with its seed.  This module holds the stacked
learner only: the config checks, collection into one slot-major ring [S, K n, ...], per-agent sampling,
``learn``, its log rows (lists of K) and ``evaluate`` are ``sac._SACDriver``'s, the same code SAC runs.
"""
from __future__ import annotations

import collections

import torch
import torch.nn.functional as F

from .sac import (LOG_STD_MAX, LOG_STD_MIN, SacActor, SacActorGroupB200, SACConfig, SacCritic, _SACDriver,
                  squashed_gaussian)

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


class SACPopulation(_SACDriver):
    def __init__(self, env, configs: list[SACConfig]):
        super().__init__(env, configs)
        configs, cfg, dev, K, D = self.configs, self.cfg, self.device, self.num_agents, self.obs_dim
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

        def per_agent(name):
            return torch.tensor([float(getattr(c, name)) for c in configs], device=dev)
        self.lr, self.gamma, self.target_entropy = per_agent("learning_rate"), per_agent("gamma"), per_agent("target_entropy")
        self.tau = per_agent("tau")
        self._tau = _per_agent(self.tau, self.target_params)
        self._keep = _per_agent(torch.tensor([1.0 - c.tau for c in configs], device=dev), self.target_params)
        self.actor_opt = _StackedAdam(self.actor_params, self.lr)
        self.critic_opt = _StackedAdam(self.critic_params, self.lr)
        if self.auto_ent:
            self.log_ent_coef = torch.zeros(K, device=dev, requires_grad=True)     # log 1
            self.ent_opt = _StackedAdam([self.log_ent_coef], self.lr)
        else:
            self.log_ent_coef = None
            self.ent_coef_tensor = per_agent("ent_coef")
        self.fused = None
        if cfg.fused_actor and dev.type == "cuda" and D <= 64:
            self.fused = SacActorGroupB200(self.actor_params, cfg.action_low, cfg.action_high)
        self._init_collection()

    # ---- networks over the agent dimension ----
    def _actor(self, obs):
        """obs [K, B, D] -> (mu, clamped log_std) [K, B, 3]"""
        w1, b1, w2, b2, w_mu, b_mu, w_ls, b_ls = self.actor_params
        latent = F.relu(_linear(F.relu(_linear(obs, w1, b1)), w2, b2))
        return _linear(latent, w_mu, b_mu), torch.clamp(_linear(latent, w_ls, b_ls), LOG_STD_MIN, LOG_STD_MAX)

    def _policy_forward(self, obs):
        """obs [K m, D], agent k on rows [k m, (k + 1) m) -> (mu, clamped log_std) [K m, 3]"""
        mean, log_std = self._actor(obs.reshape(self.num_agents, -1, self.obs_dim))
        return mean.reshape(-1, 3), log_std.reshape(-1, 3)

    @staticmethod
    def _critic(params, obs, actions):
        """The two Q-nets of `params` (critic or target) -> ([K, B, 1], [K, B, 1])"""
        x = torch.cat([obs, actions], dim=-1)
        qs = []
        for i in range(0, len(params), 6):
            w1, b1, w2, b2, w3, b3 = params[i:i + 6]
            qs.append(_linear(F.relu(_linear(F.relu(_linear(x, w1, b1)), w2, b2)), w3, b3))
        return tuple(qs)

    # ---- learning ----
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
        actions_pi, log_prob = squashed_gaussian(*self._actor(batch["obs"]), eps[0])
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
            next_actions, next_log_prob = squashed_gaussian(*self._actor(batch["next_obs"]), eps[1])
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
