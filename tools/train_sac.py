#!/usr/bin/env python
"""Train SAC (grasp_lab_salp_b200/sac.py) on the batched GPU simulator.  The defaults are the
reference recipe (src/train_robot.py: 8 envs, 200k steps, SB3's SAC defaults):

    python tools/train_sac.py --out sac_curve.jsonl
    python tools/train_sac.py --envs 1024 --total-steps 5000000 --gradient-steps 4 --batch-size 4096 \\
        --buffer-size 2000000 --learning-starts 100000 --cuda-graphs

Writes one JSON line every --log-every env-steps (env steps, gradient steps, alpha, critic and actor
loss, mean Q, episode return / length / success, eval return / success, collect and train seconds) and
ends with a summary line (env-steps/s including the learner, gradient steps/s).
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
    ap.add_argument("--save", default=None, help="torch.save the trained agent here")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    params = default_params()
    env = DeviceEnv(SalpBatch(args.envs, params, seed=args.seed))
    eval_env = DeviceEnv(SalpBatch(args.eval_envs, params, seed=10_000 + args.seed)) if args.eval_every else None
    sac = SAC(env, SACConfig(gradient_steps=args.gradient_steps, batch_size=args.batch_size, buffer_size=args.buffer_size,
                             learning_starts=args.learning_starts, cuda_graphs=args.cuda_graphs, seed=args.seed))
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
    log(summary)
    if args.save:
        sac.save(args.save)


if __name__ == "__main__":
    main()
