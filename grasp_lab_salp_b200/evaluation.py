"""The device-side evaluation loop shared by every trainer (stable-baselines3 evaluate_policy semantics).

Env i records its first quotas[i] episodes; the loop runs until every env has met its quota.  The quotas are
read back every 16 steps, not every step, so the env may step up to 15 times past the last recorded episode
(a finished env records nothing more).
"""
from __future__ import annotations

import torch


@torch.no_grad()
def run_episodes(act, env, quotas, groups=1):
    """Step `env` with `act(obs, episode_start) -> env actions` from a reset until env i has ended quotas[i]
    episodes.  episode_start [N] bool is true where an episode begins at this step (all true at the reset).
    The env's rows form `groups` contiguous slices of equal size (N a multiple of `groups`).  Returns float64
    [groups, 4]: per slice, the sums of episode return, episode length, successes (`terminated`) and the
    episode count."""
    N, dev = env.num_envs, env.device
    counts = torch.zeros(N, dtype=torch.long, device=dev)
    sums = torch.zeros((groups, 4), dtype=torch.float64, device=dev)
    cur_r = torch.zeros(N, dtype=torch.float64, device=dev)
    cur_l = torch.zeros(N, dtype=torch.float64, device=dev)
    obs = env.reset_t()
    starts = torch.ones(N, dtype=torch.bool, device=dev)
    step = 0
    while step % 16 or bool((counts < quotas).any()):
        a = act(obs.float(), starts)
        obs, rew, term, trunc, _ = env.step_t(a)
        t = term.bool()
        d = t | trunc.bool()
        cur_r += torch.nan_to_num(rew, nan=0.0, posinf=0.0, neginf=0.0).double()
        cur_l += 1
        rec = d & (counts < quotas)
        w = rec.double()
        sums += torch.stack([cur_r * w, cur_l * w, t.double() * w, w], dim=1).view(groups, N // groups, 4).sum(1)
        counts += rec.long()
        cur_r.masked_fill_(d, 0.0)
        cur_l.masked_fill_(d, 0.0)
        starts = d
        step += 1
    return sums
