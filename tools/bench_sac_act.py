#!/usr/bin/env python
"""Time salp_sac_act (csrc/salp_sac.cu) against the torch forward of the same SAC actor (eager, and
replayed as a CUDA graph) at several env counts; one JSON line per size, first a line with the card.

    python tools/bench_sac_act.py [--sizes 8,4096,16384,65536] [--obs-dim 10] [--iters 2000] [--out FILE]
    python tools/bench_sac_act.py --agents 1,4,16,64 [--sizes 8,1024] ...

With --agents, the grouped kernel instead: salp_sac_act_grouped over K actors of `size` envs each, one
launch, against K back-to-back salp_sac_act launches on the same rows, one line per (K, size).

Each timing is CUDA events around `iters` back-to-back launches after a warm-up.  FLOP and byte counts
come from the shapes: 2 N (D 256 + 256 256 + 256 6) flop; obs, noise and both action outputs plus the
packed weights once per launch.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from grasp_lab_salp_b200.sac import SacActor, SacActorB200, SacActorGroupB200  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(card=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip().splitlines()[:1])


def time_it(fn, iters):
    for _ in range(20):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters          # microseconds per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="8,4096,16384,65536")
    ap.add_argument("--obs-dim", type=int, default=10)
    ap.add_argument("--iters", type=int, default=2000)
    ap.add_argument("--out", default=None)
    ap.add_argument("--agents", default=None, help="comma-separated population sizes: time salp_sac_act_grouped")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sac_act.py needs a CUDA device")
    out = open(args.out, "w") if args.out else None

    def emit(row):
        line = json.dumps(row)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    emit(card())
    torch.manual_seed(0)
    D = args.obs_dim
    if args.agents:
        return bench_grouped(args, emit)
    actor = SacActor(D).cuda()
    lo, hi = torch.tensor([0.0, 0.0, -1.0], device="cuda"), torch.tensor([1.0, 1.0, 1.0], device="cuda")
    fused = SacActorB200(actor, lo.tolist(), hi.tolist())
    for n in [int(s) for s in args.sizes.split(",")]:
        obs = torch.randn(n, D, device="cuda")
        noise = torch.randn(n, 3, device="cuda")
        env_a, a = torch.empty(n, 3, device="cuda"), torch.empty(n, 3, device="cuda")

        def torch_fwd():
            with torch.no_grad():
                mu, ls = actor(obs)
                u = torch.tanh(mu + ls.exp() * noise)
                a.copy_(u)
                env_a.copy_(lo + (u + 1) * 0.5 * (hi - lo))

        torch_fwd()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            torch_fwd()
        t_k = time_it(lambda: fused.act(obs, noise, env_a, a), args.iters)
        t_e = time_it(torch_fwd, args.iters)
        t_g = time_it(g.replay, args.iters)
        fused.check()
        flop = 2.0 * n * (D * 256 + 256 * 256 + 256 * 6)
        nbytes = n * (D + 3 + 6) * 4 + fused.packed.numel()
        emit(dict(envs=n, obs_dim=D, salp_sac_act_us=round(t_k, 2), torch_eager_us=round(t_e, 2),
                  torch_graph_us=round(t_g, 2), kernel_tflops=round(flop / t_k * 1e-6, 2),
                  kernel_gbytes_per_s=round(nbytes / t_k * 1e-3, 1), torch_graph_tflops=round(flop / t_g * 1e-6, 2),
                  speedup_vs_graph=round(t_g / t_k, 2)))


def bench_grouped(args, emit):
    D = args.obs_dim
    lo, hi = [0.0, 0.0, -1.0], [1.0, 1.0, 1.0]
    for K in [int(k) for k in args.agents.split(",")]:
        actors = [SacActor(D).cuda() for _ in range(K)]
        group = SacActorGroupB200([torch.stack([p.detach() for p in ps]).contiguous()
                                   for ps in zip(*(a.parameters() for a in actors))], lo, hi)
        singles = [SacActorB200(a, lo, hi) for a in actors]
        for n in [int(s) for s in args.sizes.split(",")]:
            obs = torch.randn(K * n, D, device="cuda")
            noise = torch.randn(K * n, 3, device="cuda")
            env_a, a = torch.empty(K * n, 3, device="cuda"), torch.empty(K * n, 3, device="cuda")
            rows = [(obs[k * n:(k + 1) * n], noise[k * n:(k + 1) * n], env_a[k * n:(k + 1) * n], a[k * n:(k + 1) * n])
                    for k in range(K)]

            def one_by_one():
                for s, r in zip(singles, rows):
                    s.act(*r)
            t_g = time_it(lambda: group.act(obs, noise, env_a, a), args.iters)
            t_s = time_it(one_by_one, max(1, args.iters // K))
            group.check()
            emit(dict(agents=K, envs_per_agent=n, obs_dim=D, grouped_us=round(t_g, 2), k_single_launches_us=round(t_s, 2),
                      speedup=round(t_s / t_g, 2), grouped_us_per_agent=round(t_g / K, 2)))


if __name__ == "__main__":
    main()
