"""SAC on device tensors over the batched SALP simulator: the algorithm the reference trains
(src/train_robot.py: ``SAC("MlpPolicy", vec_env, learning_rate=3e-4, buffer_size=1e5,
learning_starts=1000, batch_size=256, tau=0.005, gamma=0.99)``, 8 envs, 200k steps).

Semantics are stable-baselines3's ``SAC`` with its defaults:

  * actor: Linear(D, 256) ReLU Linear(256, 256) ReLU, then the mu and log_std heads (Linear(256, 3)
    each, log_std clamped to [-20, 2]); squashed Gaussian a = tanh(mu + std eps) with
    log pi = log N(u; mu, std).sum - sum log(1 - tanh(u)^2 + 1e-6);
  * critic: two Q-nets Linear(D + 3, 256) ReLU Linear(256, 256) ReLU Linear(256, 1) on
    [obs, scaled action], a target copy; torch's default nn.Linear init everywhere (SB3 applies no
    orthogonal init to SAC);
  * ent_coef "auto": log_ent_coef starts at log 1, target entropy -3; three Adam optimisers (lr 3e-4);
  * per gradient step, in SB3's order: sample, actor sample + log-prob, entropy-coefficient step
    (alpha taken before it), target under no_grad, critic step (0.5 sum of MSEs), actor step against the
    updated critic, Polyak update (tau 0.005) of the target every step;
  * collection: uniform random actions on the Box while num_timesteps < learning_starts;
    num_timesteps grows by n_envs per vec step; after each vec step, `gradient_steps` gradient steps
    once num_timesteps > learning_starts; the ring holds buffer_size // n_envs slots of n_envs
    transitions, sampled uniformly over (slot, env).
  * done handling: SB3's ReplayBuffer with handle_timeout_termination stores
    done & ~TimeLimit.truncated.  The env flags out-of-bounds, collision and the 500-cycle limit as
    `truncated` (reference salp_robot_env.py:265-276), so the effective done is `terminated` alone and
    all three of those are bootstrapped.  The replay stores exactly that, with the env's unscaled reward.

One deviation: the learner-side reward clip of PPOConfig (``reward_clip``, default 1000, 0 turns it
off; non-finite rewards count as 0), applied when a batch is sampled -- the reference env returns finite
but huge rewards next to its integrator's stability limit (DESIGN.md 3.3).

On CUDA the replay ring is filled without copies: ``SalpBatch.step_device(out=...)`` writes
terminal_obs into next_obs[s], reward / terminated into rew[s] / done[s] and the post-reset obs into
obs[(s + 1) % slots] (where the next actor call reads), and the actor writes the scaled action into
act[s].  obs[s + 1] is thus overwritten one step before the rest of that slot, so once the ring has
wrapped sampling skips the slot being filled (SB3's optimize_memory_usage does the same).  The
rollout-side actor is one kernel (csrc/salp_sac.cu, ``SacActorB200``); the learner is plain torch.
With ``cuda_graphs=True`` one vec step and one gradient step are each replayed as a CUDA graph; the
vec-step graph fills the ring through staging buffers (index_copy_ at a device-side position), since
a captured graph cannot follow a moving slot pointer.

Everything that does not depend on how the learner stores its weights -- the config checks, collection,
replay sampling, ``learn``, its log rows and ``evaluate`` -- is ``_SACDriver``, written for K agents side by
side and shared with ``sac_population.SACPopulation``.  ``SAC`` is its K = 1 case: it adds the nn.Modules,
torch.optim.Adam, the SB3 gradient step (``train_step``) and save / load, and returns agent 0 of the shared
per-agent sample, log rows and evaluation.

The learner runs on CPU too, through ``ppo.HostEnv``.  Multi-GPU SAC is not implemented: under an
initialised torch.distributed with more than one rank the constructor refuses.
"""
from __future__ import annotations

import ctypes as C
import math
import time
from dataclasses import dataclass, fields

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .evaluation import run_episodes

HIDDEN = 256
ACT_DIM = 3
LOG_STD_MIN, LOG_STD_MAX = -20.0, 2.0


@dataclass
class SACConfig:
    learning_rate: float = 3e-4
    buffer_size: int = 100_000        # transitions (the ring has buffer_size // n_envs slots)
    learning_starts: int = 1000
    batch_size: int = 256
    tau: float = 0.005
    gamma: float = 0.99
    gradient_steps: int = 1           # per vec step (train_freq = 1 step)
    ent_coef: object = "auto"         # "auto" (learned, initial value 1) or a float
    target_entropy: float = -3.0      # -act_dim
    target_update_interval: int = 1
    reward_clip: float = 1000.0       # learner-side |r| cap (see module docstring); 0 disables
    fused_actor: bool = True          # CUDA: rollout-side actor as salp_sac_act (csrc/salp_sac.cu)
    cuda_graphs: bool = False         # CUDA: replay the vec step and the gradient step as CUDA graphs
    seed: int = 0
    action_low: tuple = (0.0, 0.0, -1.0)     # the Box of salp_robot_env.py:63-67
    action_high: tuple = (1.0, 1.0, 1.0)


PER_AGENT = ("seed", "learning_rate", "gamma", "tau", "target_entropy", "ent_coef")   # may differ in a population


# ------------------------------------------------------------------------------------------------
# networks (SB3 SACPolicy, net_arch [256, 256])
# ------------------------------------------------------------------------------------------------
def squashed_gaussian(mean, log_std, eps):
    """Reparametrised squashed-Gaussian sample with standard-normal `eps` [..., 3] and its log-prob summed over
    the last dimension, written out exactly as torch.distributions.Normal and SB3's
    SquashedDiagGaussianDistribution compute them."""
    std = torch.ones_like(mean) * log_std.exp()
    u = mean + eps * std
    a = torch.tanh(u)
    logp = (-((u - mean) ** 2) / (2 * std ** 2) - std.log() - math.log(math.sqrt(2 * math.pi))).sum(dim=-1)
    logp = logp - torch.sum(torch.log(1 - a ** 2 + 1e-6), dim=-1)
    return a, logp


class SacActor(nn.Module):
    def __init__(self, obs_dim, act_dim=ACT_DIM, hidden=HIDDEN):
        super().__init__()
        self.latent_pi = nn.Sequential(nn.Linear(obs_dim, hidden), nn.ReLU(), nn.Linear(hidden, hidden), nn.ReLU())
        self.mu = nn.Linear(hidden, act_dim)
        self.log_std = nn.Linear(hidden, act_dim)

    def forward(self, obs):
        """(mu, clamped log_std)"""
        latent = self.latent_pi(obs)
        return self.mu(latent), torch.clamp(self.log_std(latent), LOG_STD_MIN, LOG_STD_MAX)

    def action_log_prob(self, obs, eps):
        """squashed_gaussian of this actor on obs [B, D]: actions [B, 3], log-prob [B]."""
        return squashed_gaussian(*self(obs), eps)


class SacCritic(nn.Module):
    def __init__(self, obs_dim, act_dim=ACT_DIM, hidden=HIDDEN, n_critics=2):
        super().__init__()
        self.q_networks = nn.ModuleList(
            nn.Sequential(nn.Linear(obs_dim + act_dim, hidden), nn.ReLU(), nn.Linear(hidden, hidden), nn.ReLU(),
                          nn.Linear(hidden, 1)) for _ in range(n_critics))

    def forward(self, obs, actions):
        x = torch.cat([obs, actions], dim=1)
        return tuple(q(x) for q in self.q_networks)


class SacActorGroupB200:
    """Rollout-side forward of K SacActors as ONE kernel (salp_sac_act_grouped, csrc/salp_sac.cu): layer 1 in
    fp32 SIMT, layer 2 on the tensor cores with bf16 operands, heads, sampling, tanh and the Box scaling
    fused.  `params` are the eight actor tensors (latent_pi.0 weight / bias, latent_pi.2, mu, log_std) stacked
    [K, ...]; rows [k n, (k + 1) n) of a call belong to agent k.  Call `pack()` after every optimiser step.
    CUDA only -- there is no CPU path."""

    def __init__(self, params, action_low, action_high):
        self.params = params
        w1, w2, w_mu = params[0], params[2], params[4]
        if w1.shape[1] != HIDDEN or tuple(w2.shape[1:]) != (HIDDEN, HIDDEN) or w_mu.shape[1] != ACT_DIM:
            raise ValueError(f"salp_sac_act is built for hidden size {HIDDEN} and {ACT_DIM} actions")
        dev = w1.device
        if dev.type != "cuda":
            raise RuntimeError(f"{type(self).__name__} needs the actor's parameters on a CUDA device (no CPU path)")
        self.lib = _lib.load()
        self.device, self.num_agents, self.obs_dim = dev, w1.shape[0], w1.shape[2]
        self.image_bytes = self.lib.salp_sac_weight_bytes(self.obs_dim)
        if self.image_bytes < 0:
            raise ValueError(f"salp_sac_act supports obs_dim <= 64 (got {self.obs_dim})")
        self.packed = torch.empty(self.num_agents * self.image_bytes, dtype=torch.uint8, device=dev)
        self.lo = (C.c_float * 3)(*action_low)
        self.hi = (C.c_float * 3)(*action_high)
        self.pack()

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _stacked(self):
        return self.params

    def pack(self):
        ps = self._stacked()
        if any(p.dtype != torch.float32 or not p.is_contiguous() for p in ps):
            raise ValueError("the actor's parameters must be contiguous float32")
        rc = self.lib.salp_sac_pack_weights_grouped(*[C.c_void_p(p.data_ptr()) for p in ps], self.num_agents,
                                                    self.obs_dim, C.c_void_p(self.packed.data_ptr()), self._stream())
        if rc != 0:
            raise RuntimeError(f"salp_sac_pack_weights failed ({rc})")

    def act(self, obs, noise, env_action, scaled_action):
        """obs [n, D] fp32 (n a multiple of K); noise [n, 3] standard normal or None (deterministic: tanh(mu));
        writes env_action and scaled_action ([n, 3] fp32, contiguous, may be views into a replay ring)."""
        n = obs.shape[0]
        if not (n > 0 and n % self.num_agents == 0 and obs.shape[1] == self.obs_dim and obs.dtype == torch.float32
                and obs.is_contiguous() and obs.device == self.device):
            raise ValueError(f"obs must be a contiguous float32 [n, {self.obs_dim}] tensor on {self.device}, "
                             f"n a multiple of {self.num_agents}")
        for t in (noise, env_action, scaled_action):
            if t is not None and not (tuple(t.shape) == (n, 3) and t.dtype == torch.float32 and t.is_contiguous()
                                      and t.device == self.device):
                raise ValueError(f"noise / actions must be contiguous float32 [{n}, 3] tensors on {self.device}")
        rc = self.lib.salp_sac_act_grouped(C.c_void_p(self.packed.data_ptr()), self.num_agents, self.obs_dim,
                                           C.c_void_p(obs.data_ptr()), None if noise is None else C.c_void_p(noise.data_ptr()),
                                           n // self.num_agents, self.lo, self.hi, C.c_void_p(env_action.data_ptr()),
                                           C.c_void_p(scaled_action.data_ptr()), self._stream())
        if rc != 0:
            raise RuntimeError(f"salp_sac_act failed ({rc})")
        return env_action, scaled_action

    def check(self):
        if self.lib.salp_sac_check() != 0:
            raise RuntimeError("salp_sac_act: a kernel gave up waiting on its barrier")


class SacActorB200(SacActorGroupB200):
    """Rollout-side forward of one SacActor as ONE kernel (salp_sac_act, the K = 1 case of
    SacActorGroupB200).  `pack()` reads the module's parameters again, so call it after every optimiser
    step.  CUDA only -- there is no CPU path."""

    def __init__(self, actor: SacActor, action_low, action_high):
        self.actor = actor
        super().__init__(self._stacked(), action_low, action_high)

    def _stacked(self):
        a = self.actor
        return [p.detach().unsqueeze(0) for p in (a.latent_pi[0].weight, a.latent_pi[0].bias, a.latent_pi[2].weight,
                                                   a.latent_pi[2].bias, a.mu.weight, a.mu.bias, a.log_std.weight,
                                                   a.log_std.bias)]


# ------------------------------------------------------------------------------------------------
# SAC
# ------------------------------------------------------------------------------------------------
def _refuse_multi_rank(name):
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            raise RuntimeError(f"{name} is single-GPU: multi-GPU SAC (a replay per rank and a gradient all-reduce) "
                               "is not implemented")
    except ImportError:
        pass


class _SACDriver:
    """Everything of SAC that does not depend on how the learner stores its weights, for K = len(configs) agents on
    one env of K n envs, agent k on env rows [k n, (k + 1) n) (SAC is K = 1): the config checks, collection into
    one slot-major replay ring, per-agent sampling, ``learn``, its log rows and ``evaluate``.

    A learner calls ``__init__``, builds its networks, sets ``fused`` (a SacActorGroupB200 or None) and
    ``actor_opt`` / ``critic_opt`` / ``ent_opt``, then calls ``_init_collection``.  It supplies
    ``_policy_forward(obs)``, the torch actor on obs [K m, D] giving (mu, clamped log_std) [K m, 3] with agent k
    on rows [k m, (k + 1) m), and ``train_step()``, one gradient step of every agent on ``sample``'s batch."""

    def __init__(self, env, configs):
        configs = list(configs)
        K = len(configs)
        if K < 1:
            raise ValueError("a population needs at least one config")
        c0 = configs[0]
        for f in fields(SACConfig):
            if f.name not in PER_AGENT and any(getattr(c, f.name) != getattr(c0, f.name) for c in configs):
                raise ValueError(f"SACConfig.{f.name} must be equal across the population (only "
                                 f"{', '.join(PER_AGENT)} may differ per agent)")
        auto = [isinstance(c.ent_coef, str) for c in configs]
        if any(auto) and not (all(auto) and all(c.ent_coef == "auto" for c in configs)):
            raise ValueError("ent_coef must be 'auto' for every agent or a float for every agent")
        if env.num_envs % K:
            raise ValueError(f"env.num_envs ({env.num_envs}) must be a multiple of the population size ({K})")
        _refuse_multi_rank(type(self).__name__)
        self.env, self.configs = env, configs
        self.cfg = c0                             # (read for the fields shared by every agent)
        self.device = env.device
        N = env.num_envs
        self.num_agents, self.n_total, self.n_envs, self.obs_dim = K, N, N // K, env.obs_dim
        self.use_graphs = bool(c0.cuda_graphs) and self.device.type == "cuda"
        self.auto_ent = all(auto)

    def _init_collection(self):
        """Generators, replay ring, staging buffers, statistics, counters and graph slots of the collection loop
        and the driver, then the first reset.  The ring has buffer_size // n slots of K n envs (agent k's ring is
        its n columns); the generators are seeded from the first config."""
        cfg, env, dev = self.cfg, self.env, self.device
        K, N, D = self.num_agents, self.n_total, self.obs_dim
        self.gen_act = torch.Generator(device=dev)
        self.gen_act.manual_seed(cfg.seed + 1)
        self.gen_train = torch.Generator(device=dev)
        self.gen_train.manual_seed(cfg.seed + 2)
        self.low = torch.tensor(cfg.action_low, device=dev)
        self.high = torch.tensor(cfg.action_high, device=dev)

        # replay ring: S slots of N envs
        S = self.slots = max(1, cfg.buffer_size // self.n_envs)
        self.rb = dict(obs=torch.zeros((S, N, D), device=dev), next_obs=torch.zeros((S, N, D), device=dev),
                       act=torch.zeros((S, N, 3), device=dev), rew=torch.zeros((S, N), device=dev),
                       done=torch.zeros((S, N), dtype=torch.uint8, device=dev))
        self.pos, self.full = 0, False
        self._pos_t = torch.zeros(1, dtype=torch.long, device=dev)
        self._full_t = torch.zeros(1, dtype=torch.bool, device=dev)
        self.zero_copy = dev.type == "cuda" and hasattr(env, "batch") and not self.use_graphs
        self._trunc = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._env_act = torch.zeros((N, 3), device=dev)
        self._scaled = torch.zeros((N, 3), device=dev)
        self._obs = torch.zeros((N, D), device=dev)

        self._ep_ret = torch.zeros(N, device=dev)
        self._ep_len = torch.zeros(N, device=dev)
        self._ep = torch.zeros((K, 4), dtype=torch.float64, device=dev)   # sum return, sum length, successes, episodes
        self._train_stats = torch.zeros((K, 5), device=dev)               # critic loss, actor loss, alpha, mean Q, count
        self.num_timesteps = 0
        self.gradient_steps_done = 0
        self._graph_vec = {}
        self._graph_train = None
        self._policy_steps = self._train_calls = 0

        obs0 = env.reset_t()
        self._obs.copy_(obs0)
        if self.zero_copy:
            self.rb["obs"][0].copy_(obs0)

    # ---- acting ----
    def _policy_act(self, obs, env_out, scaled_out, deterministic=False, generator=None):
        """Actor forward of agent k on rows [k m, (k + 1) m) of obs [K m, D] into env_out / scaled_out (fused
        kernel or torch)."""
        noise = None if deterministic else torch.randn((obs.shape[0], 3), device=self.device, generator=generator)
        if self.fused is not None:
            self.fused.act(obs, noise, env_out, scaled_out)
            return
        with torch.no_grad():
            mean, log_std = self._policy_forward(obs)
            u = mean if noise is None else mean + noise * log_std.exp()
            a = torch.tanh(u)
            scaled_out.copy_(a)
            env_out.copy_(self.low + (a + 1.0) * 0.5 * (self.high - self.low))

    def _random_act(self, env_out, scaled_out):
        """SB3 warm-up: action_space.sample() (uniform on the Box), stored as scale_action() of it."""
        u = torch.rand((self.n_total, 3), device=self.device, generator=self.gen_act)
        a_env = self.low + u * (self.high - self.low)
        env_out.copy_(a_env)
        scaled_out.copy_(2.0 * ((a_env - self.low) / (self.high - self.low)) - 1.0)

    @torch.no_grad()
    def predict(self, obs, deterministic=True):
        """Env-space actions [n, 3] for obs [n, D] (SB3 predict); agent k acts on rows [k m, (k + 1) m)."""
        obs = obs.to(self.device, torch.float32).contiguous()
        env_out = torch.empty((obs.shape[0], 3), device=self.device)
        scaled = torch.empty_like(env_out)
        self._policy_act(obs, env_out, scaled, deterministic=deterministic, generator=self.gen_act)
        return env_out

    # ---- collection ----
    def _clip_reward(self, rew):
        """The learner-side reward clip: non-finite rewards count as 0, then |r| <= reward_clip (0 disables it)."""
        rew = torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0)
        if self.cfg.reward_clip > 0:
            rew = rew.clamp(-self.cfg.reward_clip, self.cfg.reward_clip)
        return rew

    def _bookkeep(self, rew, term, trunc):
        raw = self._clip_reward(rew)
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

    def _vec_step_body(self, random):
        """One vec step into the ring at the current position."""
        rb, S = self.rb, self.slots
        if self.zero_copy:
            s, s1 = self.pos, (self.pos + 1) % S
            obs = rb["obs"][s]
            if random:
                self._random_act(self._env_act, rb["act"][s])
            else:
                self._policy_act(obs, self._env_act, rb["act"][s], generator=self.gen_act)
            self.env.batch.step_device(self._env_act, auto_reset=True, sort_by_k=self.env.sort,
                                       out=dict(obs=rb["obs"][s1], reward=rb["rew"][s], terminated=rb["done"][s],
                                                truncated=self._trunc, terminal_obs=rb["next_obs"][s]))
            self._bookkeep(rb["rew"][s], rb["done"][s], self._trunc)
        else:
            if random:
                self._random_act(self._env_act, self._scaled)
            else:
                self._policy_act(self._obs, self._env_act, self._scaled, generator=self.gen_act)
            obs, rew, term, trunc, term_obs = self.env.step_t(self._env_act)
            p = self._pos_t
            rb["obs"].index_copy_(0, p, self._obs[None])
            rb["act"].index_copy_(0, p, self._scaled[None])
            rb["next_obs"].index_copy_(0, p, term_obs[None].float())
            rb["rew"].index_copy_(0, p, rew[None].float())
            rb["done"].index_copy_(0, p, term[None].to(torch.uint8))
            self._obs.copy_(obs)
            self._bookkeep(rew, term, trunc)
        self._pos_t.add_(1).remainder_(S)
        self._full_t |= self._pos_t == 0

    def _vec_step(self):
        random = self.num_timesteps < self.cfg.learning_starts
        if not random:
            self._policy_steps += 1
        if self.use_graphs and self._policy_steps >= 3:        # two eager policy steps warm up first
            g = self._graph_vec.get("policy")
            if g is None:
                g = torch.cuda.CUDAGraph()
                g.register_generator_state(self.gen_act)
                with torch.cuda.graph(g):
                    self._vec_step_body(False)
                self._graph_vec["policy"] = g
            g.replay()
        else:
            self._vec_step_body(random)
        self.pos = (self.pos + 1) % self.slots
        self.full = self.full or self.pos == 0
        self.num_timesteps += self.n_envs

    # ---- learning ----
    def sample(self, batch_size):
        """`batch_size` transitions per agent ([K, B, ...]): uniform over (slot, env of that agent) among the
        complete slots; once the ring has wrapped the slot being filled is skipped.  Device-side (capturable): the
        fill level lives in device tensors."""
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
        rew = self._clip_reward(rb["rew"].view(-1)[idx])
        return dict(obs=rb["obs"].view(S * N, -1)[idx], actions=rb["act"].view(S * N, -1)[idx],
                    next_obs=rb["next_obs"].view(S * N, -1)[idx], rewards=rew.unsqueeze(-1),
                    dones=rb["done"].view(-1)[idx].float().unsqueeze(-1), slot=slot, env=env)

    def _train(self):
        for _ in range(self.cfg.gradient_steps):
            # (the graph holds the Polyak update of every step: target_update_interval 1 only)
            if self.use_graphs and self.cfg.target_update_interval == 1 and self.gradient_steps_done >= 3:
                if self._graph_train is None:   # three eager steps warmed up cuBLAS and the optimisers
                    for o in self._optimisers():
                        o.zero_grad(set_to_none=True)
                    g = torch.cuda.CUDAGraph()
                    g.register_generator_state(self.gen_train)
                    with torch.cuda.graph(g):
                        self.train_step()
                    self._graph_train = g
                self._graph_train.replay()
            else:
                self.train_step()
            self.gradient_steps_done += 1
        if self.fused is not None:
            self.fused.pack()

    def _optimisers(self):
        return [self.actor_opt, self.critic_opt] + ([self.ent_opt] if self.auto_ent else [])

    # ---- driver ----
    def _sync(self):
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)

    def learn(self, total_timesteps, log=None, log_interval=1000, eval_env=None, eval_every=0, n_eval_episodes=10):
        """Collect and train until num_timesteps >= total_timesteps.  Every `log_interval` env-steps (and
        at the end) a row of statistics goes to `log`; every `eval_every` env-steps, with an `eval_env`,
        `evaluate` runs first and its result joins the row."""
        history = []
        collect_s = train_s = 0.0
        next_log = self.num_timesteps + log_interval
        next_eval = self.num_timesteps + eval_every if eval_every else None
        ev = {}
        while self.num_timesteps < total_timesteps:
            t0 = time.perf_counter()
            self._vec_step()
            self._sync()
            t1 = time.perf_counter()
            collect_s += t1 - t0
            if self.num_timesteps > self.cfg.learning_starts:
                self._train()
                self._sync()
                train_s += time.perf_counter() - t1
            if eval_env is not None and next_eval is not None and self.num_timesteps >= next_eval:
                ev = self.evaluate(eval_env, n_eval_episodes)
                next_eval += eval_every
            if self.num_timesteps >= next_log or self.num_timesteps >= total_timesteps:
                row = self._row(collect_s, train_s)
                if ev:
                    row.update(eval_return=ev["mean_return"], eval_success=ev["success_rate"],
                               eval_length=ev["mean_length"])
                history.append(row)
                if log:
                    log(row)
                next_log += log_interval
                collect_s = train_s = 0.0
                ev = {}
        return history

    def _row(self, collect_s, train_s):
        """The training and episode statistics since the last row (per agent: lists of K), which it zeroes."""
        ep, ts = self._ep.tolist(), self._train_stats.tolist()
        self._ep.zero_()
        self._train_stats.zero_()
        nan = float("nan")

        def ratio(rows, i, j):
            return [r[i] / r[j] if r[j] else nan for r in rows]
        return dict(env_steps=self.num_timesteps, gradient_steps=self.gradient_steps_done,
                    ent_coef=ratio(ts, 2, 4), critic_loss=ratio(ts, 0, 4), actor_loss=ratio(ts, 1, 4),
                    mean_q=ratio(ts, 3, 4), episodes=[int(e[3]) for e in ep], mean_episode_return=ratio(ep, 0, 3),
                    mean_episode_length=ratio(ep, 1, 3), success_rate=ratio(ep, 2, 3), collect_seconds=collect_s,
                    train_seconds=train_s)

    @torch.no_grad()
    def evaluate(self, env, n_episodes=10):
        """Deterministic episodes (SB3 EvalCallback(deterministic=True) via evaluate_policy) on an eval env of
        K m envs, agent k acting on rows [k m, (k + 1) m): env i of a slice contributes (n_episodes + i) // m
        episodes.  Per-agent lists of mean_return, mean_length, success_rate and episodes.  The quotas are read
        back every 16 steps, so the env may step up to 15 times past the last recorded episode."""
        K, N = self.num_agents, env.num_envs
        if N % K:
            raise ValueError(f"the eval env's num_envs ({N}) must be a multiple of the population size ({K})")
        m = N // K
        quotas = ((n_episodes + torch.arange(m, device=env.device)) // m).repeat(K)
        s = run_episodes(lambda obs, starts: self.predict(obs, deterministic=True), env, quotas, K).tolist()
        return dict(mean_return=[x[0] / x[3] for x in s], mean_length=[x[1] / x[3] for x in s],
                    success_rate=[x[2] / x[3] for x in s], episodes=[int(x[3]) for x in s])


class SAC(_SACDriver):
    def __init__(self, env, config: SACConfig | None = None):
        super().__init__(env, [config or SACConfig()])
        cfg, dev, D = self.cfg, self.device, self.obs_dim
        torch.manual_seed(cfg.seed)
        self.actor = SacActor(D).to(dev)
        self.critic = SacCritic(D).to(dev)
        self.critic_target = SacCritic(D).to(dev)
        self.critic_target.load_state_dict(self.critic.state_dict())
        self.critic_target.requires_grad_(False)
        cuda = dev.type == "cuda"
        adam = dict(lr=cfg.learning_rate, capturable=cuda)
        self.actor_opt = torch.optim.Adam(self.actor.parameters(), **adam)
        self.critic_opt = torch.optim.Adam(self.critic.parameters(), **adam)
        if self.auto_ent:
            self.log_ent_coef = torch.log(torch.ones(1, device=dev)).requires_grad_(True)
            self.ent_opt = torch.optim.Adam([self.log_ent_coef], **adam)
        else:
            self.log_ent_coef = None
            self.ent_coef_tensor = torch.tensor(float(cfg.ent_coef), device=dev)
        self.fused = None
        if cfg.fused_actor and cuda and D <= 64:
            self.fused = SacActorB200(self.actor, cfg.action_low, cfg.action_high)
        self._init_collection()

    def _policy_forward(self, obs):
        return self.actor(obs)

    def sample(self, batch_size):
        """`batch_size` transitions [B, ...], uniform over (slot, env) among the complete slots; once the ring has
        wrapped the slot being filled is skipped.  Device-side (capturable)."""
        return {k: v[0] for k, v in super().sample(batch_size).items()}

    def train_step(self, batch=None, eps=None):
        """One SB3 gradient step.  `batch` (dict of obs, actions, next_obs, rewards [B, 1], dones [B, 1])
        and `eps` (standard-normal noise of the two actor samples) are drawn here unless given."""
        cfg = self.cfg
        if batch is None:
            batch = self.sample(cfg.batch_size)
        B = batch["obs"].shape[0]
        if eps is None:
            eps = (torch.randn((B, 3), device=self.device, generator=self.gen_train),
                   torch.randn((B, 3), device=self.device, generator=self.gen_train))
        actions_pi, log_prob = self.actor.action_log_prob(batch["obs"], eps[0])
        log_prob = log_prob.reshape(-1, 1)
        if self.auto_ent:
            ent_coef = torch.exp(self.log_ent_coef.detach())
            ent_coef_loss = -(self.log_ent_coef * (log_prob + cfg.target_entropy).detach()).mean()
            self.ent_opt.zero_grad()
            ent_coef_loss.backward()
            self.ent_opt.step()
        else:
            ent_coef = self.ent_coef_tensor
        with torch.no_grad():
            next_actions, next_log_prob = self.actor.action_log_prob(batch["next_obs"], eps[1])
            next_q_values = torch.cat(self.critic_target(batch["next_obs"], next_actions), dim=1)
            next_q_values, _ = torch.min(next_q_values, dim=1, keepdim=True)
            next_q_values = next_q_values - ent_coef * next_log_prob.reshape(-1, 1)
            target_q_values = batch["rewards"] + (1 - batch["dones"]) * cfg.gamma * next_q_values
        current_q_values = self.critic(batch["obs"], batch["actions"])
        critic_loss = 0.5 * sum(F.mse_loss(current_q, target_q_values) for current_q in current_q_values)
        self.critic_opt.zero_grad()
        critic_loss.backward()
        self.critic_opt.step()
        q_values_pi = torch.cat(self.critic(batch["obs"], actions_pi), dim=1)
        min_qf_pi, _ = torch.min(q_values_pi, dim=1, keepdim=True)
        actor_loss = (ent_coef * log_prob - min_qf_pi).mean()
        self.actor_opt.zero_grad()
        actor_loss.backward()
        self.actor_opt.step()
        self._train_calls += 1
        if (self._train_calls - 1) % cfg.target_update_interval == 0:
            with torch.no_grad():
                tp, sp = list(self.critic_target.parameters()), list(self.critic.parameters())
                torch._foreach_mul_(tp, 1 - cfg.tau)
                torch._foreach_add_(tp, sp, alpha=cfg.tau)
        with torch.no_grad():
            mean_q = torch.stack([q.mean() for q in current_q_values]).mean()
            self._train_stats += torch.stack([critic_loss.detach(), actor_loss.detach(), ent_coef.reshape(()),
                                              mean_q, torch.ones((), device=self.device)])
        return dict(critic_loss=critic_loss, actor_loss=actor_loss, ent_coef=ent_coef,
                    ent_coef_loss=ent_coef_loss if self.auto_ent else None)

    def _row(self, collect_s, train_s):
        return {k: v[0] if isinstance(v, list) else v for k, v in super()._row(collect_s, train_s).items()}

    def evaluate(self, env, n_episodes=10):
        """The shared evaluation with scalar results: env i contributes (n_episodes + i) // n_envs episodes."""
        return {k: v[0] for k, v in super().evaluate(env, n_episodes).items()}

    # ---- persistence ----
    def save(self, path):
        """torch.save of the networks, log_ent_coef and the optimiser states (not SB3's zip format)."""
        torch.save(dict(actor=self.actor.state_dict(), critic=self.critic.state_dict(),
                        critic_target=self.critic_target.state_dict(),
                        log_ent_coef=None if self.log_ent_coef is None else self.log_ent_coef.detach().cpu(),
                        actor_opt=self.actor_opt.state_dict(), critic_opt=self.critic_opt.state_dict(),
                        ent_opt=self.ent_opt.state_dict() if self.auto_ent else None,
                        num_timesteps=self.num_timesteps), path)

    def load(self, path):
        st = torch.load(path, map_location=self.device, weights_only=False)
        self.actor.load_state_dict(st["actor"])
        self.critic.load_state_dict(st["critic"])
        self.critic_target.load_state_dict(st["critic_target"])
        if self.auto_ent and st["log_ent_coef"] is not None:
            with torch.no_grad():
                self.log_ent_coef.copy_(st["log_ent_coef"].to(self.device))
            self.ent_opt.load_state_dict(st["ent_opt"])
        self.actor_opt.load_state_dict(st["actor_opt"])
        self.critic_opt.load_state_dict(st["critic_opt"])
        self.num_timesteps = st["num_timesteps"]
        if self.fused is not None:
            self.fused.pack()
