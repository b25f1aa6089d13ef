#!/usr/bin/env python
"""Train SAC (grasp_lab_salp_b200/sac.py) on the batched GPU simulator.  The defaults are the
reference recipe (src/train_robot.py: 8 envs, 200k steps, SB3's SAC defaults):

    python tools/train_sac.py --out sac_curve.jsonl
    python tools/train_sac.py --envs 1024 --total-steps 5000000 --gradient-steps 4 --batch-size 4096 \\
        --buffer-size 2000000 --learning-starts 100000 --cuda-graphs

Writes one JSON line every --log-every env-steps (env steps, gradient steps, alpha, critic and actor
loss, mean Q, episode return / length / success, eval return / success, collect and train seconds) and
ends with a summary line (env-steps/s including the learner, gradient steps/s).

--agents K trains seeds seed .. seed + K - 1 as one population (grasp_lab_salp_b200/sac_population.py) on
K --envs envs, with K --eval-envs envs for evaluation; --learning-rate, --gamma, --tau and --target-entropy
take one value or K comma-separated values.  Per-agent values in rows and the summary are lists of K, and
--total-steps and env_steps count one agent's env-steps:

    python tools/train_sac.py --agents 16 --cuda-graphs --out sac_population16.jsonl
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from grasp_lab_salp_b200 import SalpBatch, default_params  # noqa: E402
from grasp_lab_salp_b200.ppo import DeviceEnv  # noqa: E402
from grasp_lab_salp_b200.sac import SAC, SACConfig  # noqa: E402
from grasp_lab_salp_b200.sac_population import SACPopulation  # noqa: E402


def per_agent(ap, name, text, k):
    """One value for every agent, or k comma-separated values."""
    vals = [float(v) for v in text.split(",")]
    if len(vals) == 1:
        return vals * k
    if len(vals) != k:
        ap.error(f"--{name} takes one value or {k} comma-separated values (got {len(vals)})")
    return vals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8)
    ap.add_argument("--total-steps", type=int, default=200_000)
    ap.add_argument("--gradient-steps", type=int, default=1)
    ap.add_argument("--batch-size", type=int, default=256)
    ap.add_argument("--buffer-size", type=int, default=100_000)
    ap.add_argument("--learning-starts", type=int, default=1000)
    ap.add_argument("--cuda-graphs", action="store_true", help="replay the vec step and the gradient step as CUDA graphs")
    ap.add_argument("--eval-every", type=int, default=10_000, help="env-steps between deterministic evaluations (0: none)")
    ap.add_argument("--eval-episodes", type=int, default=32)
    ap.add_argument("--eval-envs", type=int, default=32)
    ap.add_argument("--log-every", type=int, default=5000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--save", default=None, help="torch.save the trained agent here (with --agents: PATH.agentK)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--agents", type=int, default=None,
                    help="train seeds seed .. seed+K-1 as one population of K agents, each on --envs envs")
    ap.add_argument("--learning-rate", default="3e-4", help="one value, or one per agent (comma-separated)")
    ap.add_argument("--gamma", default="0.99", help="one value, or one per agent (comma-separated)")
    ap.add_argument("--tau", default="0.005", help="one value, or one per agent (comma-separated)")
    ap.add_argument("--target-entropy", default="-3", help="one value, or one per agent (comma-separated)")
    args = ap.parse_args()
    params = default_params()
    K = args.agents or 1
    if K < 1:
        ap.error("--agents must be >= 1")
    hp = {name: per_agent(ap, name.replace("_", "-"), getattr(args, name), K)
          for name in ("learning_rate", "gamma", "tau", "target_entropy")}
    env = DeviceEnv(SalpBatch(K * args.envs, params, seed=args.seed))
    eval_env = DeviceEnv(SalpBatch(K * args.eval_envs, params, seed=10_000 + args.seed)) if args.eval_every else None
    cfgs = [SACConfig(gradient_steps=args.gradient_steps, batch_size=args.batch_size, buffer_size=args.buffer_size,
                      learning_starts=args.learning_starts, cuda_graphs=args.cuda_graphs, seed=args.seed + k,
                      **{name: v[k] for name, v in hp.items()}) for k in range(K)]
    sac = SAC(env, cfgs[0]) if args.agents is None else SACPopulation(env, cfgs)
    out = open(args.out, "w") if args.out else None
    t0 = time.perf_counter()

    def log(row):
        row = dict(row, wall_seconds=time.perf_counter() - t0)
        line = json.dumps(row)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    rows = sac.learn(args.total_steps, log=log, log_interval=args.log_every, eval_env=eval_env,
                     eval_every=args.eval_every, n_eval_episodes=args.eval_episodes)
    env.batch.check()
    wall = time.perf_counter() - t0
    collect = sum(r["collect_seconds"] for r in rows)
    train = sum(r["train_seconds"] for r in rows)
    evals = [r for r in rows if "eval_return" in r]
    summary = dict(summary=True, card=torch.cuda.get_device_name(), envs=args.envs, env_steps=sac.num_timesteps,
                   gradient_steps=sac.gradient_steps_done, cuda_graphs=sac.use_graphs, fused_actor=sac.fused is not None,
                   wall_seconds=wall, collect_seconds=collect, train_seconds=train,
                   env_steps_per_sec_incl_learner=sac.num_timesteps / wall,
                   gradient_steps_per_sec=sac.gradient_steps_done / train if train > 0 else 0.0,
                   final_eval_return=evals[-1]["eval_return"] if evals else None,
                   final_eval_success=evals[-1]["eval_success"] if evals else None)
    if args.agents is not None:
        summary.update(agents=K, seeds=[c.seed for c in cfgs], **hp)
    log(summary)
    if args.save:
        if args.agents is None:
            sac.save(args.save)
        else:
            for k in range(K):
                sac.save_agent(k, f"{args.save}.agent{k}")


if __name__ == "__main__":
    main()
