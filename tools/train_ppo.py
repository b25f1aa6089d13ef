#!/usr/bin/env python
"""Train PPO (MLP policy, SB3 defaults; --recurrent: LSTM policy of train_robot_recurrent_ppo.py) on the
batched GPU simulator -- BASELINE configs 3 and 4.

    python tools/train_ppo.py --envs 16384 --total-steps 10000000 --out gpurun_out/ppo_curve.jsonl
    torchrun --nproc-per-node 8 tools/train_ppo.py --envs 65536 ...      (envs = whole job, sharded)

Writes one JSON line per PPO iteration (env_steps, mean step reward, mean episode return /
length, success rate, approx KL, wall seconds for rollout and update).  With --eval-every, the iteration
that reaches each multiple of it also runs a deterministic evaluation on a separate env (eval_return,
eval_success, eval_length, eval_seconds); --save-best keeps the model with the best eval_return so far
(SB3 EvalCallback's best_model_save_path), --save writes the final model, --load resumes from a file.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from grasp_lab_salp_b200 import PRECISION_F64, PRECISION_MIXED, default_params  # noqa: E402
from grasp_lab_salp_b200.distributed import make_shard, world_info  # noqa: E402
from grasp_lab_salp_b200.ppo import PPO, DeviceEnv, PPOConfig, RecurrentPPO  # noqa: E402


class FreshEnv:
    """An eval env rebuilt from its seed at every reset: every evaluation meets the same scenes, so that
    evaluations during training compare like with like and a saved model's evaluation can be repeated in
    another process (--evaluate-only)."""

    def __init__(self, make):
        self.make, self.env = make, make()
        self.num_envs, self.obs_dim, self.device = self.env.num_envs, self.env.obs_dim, self.env.device

    def reset_t(self):
        self.env = self.make()
        return self.env.reset_t()

    def step_t(self, actions):
        return self.env.step_t(actions)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--total-steps", type=int, default=10_000_000)
    ap.add_argument("--n-steps", type=int, default=32)
    ap.add_argument("--n-epochs", type=int, default=10)
    ap.add_argument("--batch-size", type=int, default=16384)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--precision", choices=["mixed", "f64"], default="mixed")
    ap.add_argument("--recurrent", action="store_true", help="RecurrentPPO, LSTM(256) actor and critic (config 4)")
    ap.add_argument("--cuda-graphs", action="store_true", help="replay rollout and minibatch steps as CUDA graphs")
    ap.add_argument("--eval-every", type=int, default=0, help="env-steps between deterministic evaluations")
    ap.add_argument("--eval-envs", type=int, default=64)
    ap.add_argument("--eval-episodes", type=int, default=64)
    ap.add_argument("--save", default=None, help="write the final model here (torch.save)")
    ap.add_argument("--save-best", default=None, help="write the model with the best eval_return so far here")
    ap.add_argument("--load", default=None, help="resume from a file written by --save / --save-best")
    ap.add_argument("--evaluate-only", action="store_true",
                    help="with --load: evaluate the loaded model once on the eval env, print the result and exit")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, local, world = world_info()
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    params = default_params(precision=PRECISION_MIXED if args.precision == "mixed" else PRECISION_F64)
    batch = make_shard(args.envs, params, seed=args.seed)
    algo = RecurrentPPO if args.recurrent else PPO
    ppo = algo(DeviceEnv(batch), PPOConfig(n_steps=args.n_steps, n_epochs=args.n_epochs, batch_size=args.batch_size,
                                           seed=args.seed, cuda_graphs=args.cuda_graphs))
    if args.load:
        ppo.load(args.load)
    eval_env = FreshEnv(lambda: DeviceEnv(make_shard(args.eval_envs, params, seed=10_000 + args.seed)))
    if args.evaluate_only:
        ev = ppo.evaluate(eval_env, args.eval_episodes)
        if rank == 0:
            print(json.dumps(dict(ev, evaluate_only=True, load=args.load)), flush=True)
        return
    out = open(args.out, "w") if (args.out and rank == 0) else None
    t0 = time.perf_counter()
    best = [float("-inf")]

    def log(row):
        if args.save_best and "eval_return" in row and row["eval_return"] > best[0]:
            best[0] = row["eval_return"]
            ppo.save(args.save_best)               # (every rank: save gathers the per-rank state)
        if rank == 0:
            row = dict(row, wall_seconds=time.perf_counter() - t0)
            line = json.dumps(row)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
                out.flush()

    stats = ppo.learn(args.total_steps, log=log, eval_env=eval_env if args.eval_every else None,
                      eval_every=args.eval_every, n_eval_episodes=args.eval_episodes)
    batch.check()
    if args.save:
        ppo.save(args.save)
    evals = [h for h in stats.history if "eval_return" in h]
    ar = ppo.allreduce_seconds_per_step()
    if rank == 0:
        wall = time.perf_counter() - t0
        sim = sum(h["rollout_seconds"] for h in stats.history)
        upd = sum(h["update_seconds"] for h in stats.history)
        n_params = sum(p.numel() for p in ppo.policy.parameters())
        steps_per_update = ppo._upd_calls / max(1, len(stats.history))
        print(json.dumps({"summary": True, "envs": args.envs, "gpus": world, "env_steps": stats.env_steps,
                          "update_seconds_total": upd, "rollout_seconds_total": sim,
                          "policy_parameters": n_params, "optimiser_steps_per_update": steps_per_update,
                          "allreduce_seconds_per_optimiser_step": ar,
                          "allreduce_share_of_update": (ar * ppo._upd_calls / upd) if upd > 0 else 0.0,
                          "update_cuda_graph": bool(ppo.graph_update),
                          "wall_seconds": wall, "env_steps_per_sec_incl_learner": stats.env_steps / wall,
                          "env_steps_per_sec_rollout_only": stats.env_steps / sim,
                          "final_success_rate": stats.success_rate,
                          "final_mean_episode_return": stats.mean_episode_return,
                          "final_eval_success": evals[-1]["eval_success"] if evals else None,
                          "final_eval_return": evals[-1]["eval_return"] if evals else None,
                          "eval_seconds_total": sum(h["eval_seconds"] for h in evals)}), flush=True)
    if world > 1:
        # (no destroy_process_group(): with NCCL collectives captured in CUDA graphs it blocked at exit on
        #  8 GPUs; leave at once instead)
        sys.stdout.flush()
        if out:
            out.close()
        os._exit(0)


if __name__ == "__main__":
    main()
