#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched SALP simulator on N B200s (device-timed, whole box).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W     # the CPU implementation of the path
    python bench.py --steps K --warmup W --dump-outputs DIR   # + what the last timed step returned, as .npy

A *step* is one vectorised SalpRobotEnv.step() over every env of the rank (auto-reset on, one
full breathing cycle = K_i in [0, 1348] physics substeps per env).  Workload at N = 1:
BASELINE.json configs[1] -- 4096 batched envs, uniform-random Box actions (SURVEY 8d input A),
Philox scenes; for N > 1 every GPU gets its own 4096 envs (weak scaling, no data-path
collective: envs are independent; global env ids keep the per-env random streams
shard-invariant).

Timing: W warm-up steps, then K steps, each bracketed by its own CUDA event pair on the
launching stream; between steps the L2 is flushed (a 256 MiB memset, outside the event pairs)
and that step's substep total is reduced.  value = envs * K / sum(step durations), max over
ranks (all-reduce MAX).  e2e = the same workload through the host-buffer C-ABI call
(salp_step_host: pinned host actions -> H2D -> kernel -> D2H of obs/reward/flags/terminal obs,
one stream sync), wall-clocked around K synchronous calls.

cpu_baseline / --impl reference: the reference's OWN CPU path -- the unmodified Python SalpRobotEnv
under a SubprocVecEnv-equivalent (oracle/ref_vecenv.py: one process per host core, pipes, lock-step,
worker-side auto-reset; src/train_robot.py:25-26) -- when its sources are staged (baseline/_ref/src,
tools/stage_reference.py) and numba is importable; the plain-C port (oracle/salp_oracle.c) is timed
beside it (`cpu_baseline_port`) and is the fallback.

roofline: the dominant (only significant) kernel is the step kernel the library reports
(salp_last_step_kernel); it is bound by the FP32 SIMT
pipe, not HBM and not tensor cores (SURVEY 8d: ~0.66 KB of state traffic against ~3.5e5 flop
per env-step), so `bound` is "fp32" and `achieved` = substeps/s * 500 flop (SURVEY 8d's
canonical per-substep count of the reference formulation) against the FFMA rate this same run
measures with salp_probe_fp32_peak (MEASURED_PEAKS.json has no FP32 SIMT figure; nominal
148 SM * 128 lanes * 2 * 1.965 GHz = 74.4 TFLOP/s is quoted beside it).  The HBM view is
reported too (`hbm`), against MEASURED_PEAKS.json.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from

FLOP_PER_SUBSTEP = 500.0            # SURVEY.md 8(d) "ALGORITHMIC work per unit"
NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12
METRIC = "env-steps/sec"


def workload(n):
    return f"{n} batched envs per GPU, uniform-random Box actions, auto-reset, 1 cycle (0..1348 substeps) per env-step"


def common_config(n, gpus):
    """Identical in both arms (the driver compares the two lines' `config`)."""
    return {"workload": workload(n), "envs_per_gpu": n, "global_envs": n * gpus,
            "actions": "uniform Box (SURVEY 8d input A)", "auto_reset": True, "parallelism": f"env-shard x{gpus}"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["cuda", "reference"], default="cuda")
    ap.add_argument("--envs", type=int, default=4096, help="envs per GPU (BASELINE configs[1]: 4096)")
    ap.add_argument("--precision", choices=["mixed", "f64"], default="mixed")
    ap.add_argument("--sort-by-k", choices=["auto", "on", "off"], default="auto")
    ap.add_argument("--no-sweep", action="store_true", help="skip the env-count sweep (config 5) extras")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (rank 0's envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl cuda)")
    return args


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (plain-C restatement of the reference's Python), one process per core,
# like the reference's SubprocVecEnv (src/train_robot.py:26).
# ------------------------------------------------------------------------------------------------
_W = {}


def _cpu_worker_init(n_envs, seed):
    import numpy as np
    from oracle.salp_oracle import OracleVecEnv
    _W["env"] = OracleVecEnv(n_envs, seed=seed)
    _W["env"].reset()
    _W["rng"] = np.random.default_rng(seed)
    _W["n"] = n_envs


def _cpu_worker_steps(steps):
    env, rng, n = _W["env"], _W["rng"], _W["n"]
    sub = 0
    for _ in range(steps):
        a = rng.uniform([0, 0, -1], [1, 1, 1], size=(n, 3)).astype("float32")
        env.step(a, auto_reset=True)
        sub += int(env.substeps.sum())
    return n * steps, sub


class CpuArm:
    """`cores` worker processes, `envs_per_worker` oracle envs each."""

    def __init__(self, cores, envs_per_worker):
        import multiprocessing as mp
        from oracle import salp_oracle
        salp_oracle.build()
        self.cores = cores
        self.envs_per_worker = envs_per_worker
        ctx = mp.get_context("fork")
        self.pools = [ctx.Pool(1, initializer=_cpu_worker_init, initargs=(envs_per_worker, 1000 + i))
                      for i in range(cores)]

    def run(self, steps):
        t0 = time.perf_counter()
        res = [p.apply_async(_cpu_worker_steps, (steps,)) for p in self.pools]
        out = [r.get() for r in res]
        dt = time.perf_counter() - t0
        return sum(o[0] for o in out), sum(o[1] for o in out), dt

    def close(self):
        for p in self.pools:
            p.terminate()


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def port_baseline(seconds, total_envs=4096):
    """The plain-C port on the host cores: `total_envs` envs split over one process per core, as many
    vectorised steps as fit in ~`seconds`."""
    cores = host_cores()
    per = max(1, total_envs // cores)
    arm = CpuArm(cores, per)
    try:
        arm.run(1)                                   # warm-up / page-in
        n1, _, dt1 = arm.run(1)
        steps = max(1, min(200, int(seconds / max(dt1, 1e-3))))
        n, sub, dt = arm.run(steps)
    finally:
        arm.close()
    return {"value": n / dt, "unit": METRIC, "cores": cores, "kind": "port",
            "substeps_per_sec": sub / dt, "mean_substeps": sub / n,
            "sample": f"{per * cores} envs ({per}/process x {cores} processes) x {steps} vectorised steps of the "
                      f"same workload, oracle/salp_oracle.c (gcc -O2 scalar float64 port of the reference's Python)"}


def reference_available():
    try:
        from oracle import ref_harness
        return ref_harness.available()
    except Exception:
        return False


def reference_baseline(vec_steps, warmup, n_envs=None):
    """The reference's own CPU path: unmodified Python SalpRobotEnv x `cores`, one process each,
    lock-step vector steps (SubprocVecEnv semantics, src/train_robot.py:25-26)."""
    from oracle import ref_vecenv
    cores = n_envs or host_cores()
    n, sub, dt = ref_vecenv.time_reference(cores, vec_steps, warmup)
    return {"value": n / dt, "unit": METRIC, "cores": cores, "kind": "reference", "seconds": dt,
            "substeps_per_sec": sub / dt, "mean_substeps": sub / max(n, 1),
            "sample": f"{cores} envs (1 per process, {cores} processes, pipes, lock-step) x {vec_steps} vector steps after "
                      f"{warmup} warm-up steps (numba JIT done before the fork) of the same workload: the UNMODIFIED "
                      f"Python reference (SalpRobotEnv under a SubprocVecEnv-equivalent, oracle/ref_vecenv.py)",
            "reference_files": ref_vecenv.manifest()}


def cpu_baseline(seconds, total_envs=4096):
    """`cpu_baseline` of the CUDA arm's line: the reference's own path if its sources travelled
    (kind "reference", ~`seconds` of lock-step vector steps), the C port beside it.  The reference
    runs in a FRESH interpreter (this file with --impl reference): numba's LAPACK binding failed to
    import inside a process that had already initialised torch + CUDA on the GPU box."""
    import subprocess
    port = port_baseline(seconds, total_envs)
    if not reference_available():
        port["reference_unavailable"] = "reference sources not staged (tools/stage_reference.py) or numba missing"
        return port, None
    steps = max(4, int(seconds / (3 * 0.55)))
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps),
                            "--warmup", "1", "--envs", str(total_envs)], capture_output=True, text=True, timeout=600)
        ref = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        if ref.get("kind") == "reference":
            return ref, port
        port["reference_unavailable"] = "the reference arm fell back to the port: " + r.stderr.strip().splitlines()[-1][:300]
    except Exception as e:
        port["reference_unavailable"] = f"{type(e).__name__}: {e}"
    return port, None


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    n = args.envs
    base = None
    if reference_available():
        # one bench "step" = R lock-step vector steps of `cores` reference envs (a bounded sample of the
        # n-env batch); R sized so that (K + W) steps stay within ~2 minutes (a vector step waits for
        # its slowest env: ~0.55 s)
        R = max(1, min(3, int(120.0 / (0.55 * max(1, args.steps + args.warmup)))))
        try:
            base = reference_baseline(vec_steps=args.steps * R, warmup=max(3, args.warmup * R))
            base["sample"] = f"each step = {R} lock-step vector step(s); " + base["sample"]
        except Exception as e:
            import traceback
            base = None
            traceback.print_exc()
            sys.stderr.write(f"reference arm: Python reference failed ({type(e).__name__}: {e}); timing the C port\n")
    if base is None:
        # fallback: the C port; bounded per-step sample sized so that (K + W) steps take ~2 minutes
        probe = CpuArm(cores, 8)
        probe.run(1)
        m, _, dt = probe.run(2)
        probe.close()
        rate = m / dt
        budget = 120.0 / max(1, args.steps + args.warmup)
        per = int(max(1, min(max(1, n // cores), rate * budget / cores)))
        arm = CpuArm(cores, per)
        try:
            arm.run(max(1, args.warmup))
            m, sub, dt = arm.run(args.steps)
        finally:
            arm.close()
        base = {"value": m / dt, "unit": METRIC, "cores": cores, "kind": "port", "seconds": dt, "substeps_per_sec": sub / dt,
                "sample": f"each step = {per * cores} envs ({per}/process x {cores} processes) of the workload; "
                          "oracle/salp_oracle.c, the plain-C float64 port (reference sources not staged or numba missing)"}
    value = base["value"]
    line = {
        "metric": METRIC, "value": value, "unit": METRIC, "impl": "reference", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * base["seconds"] / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": common_config(n, args.gpus),
        "cpu_baseline": base,
        "substeps_per_sec": base["substeps_per_sec"],
        "e2e": {"value": value, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi fields of the profiling recipe, through NVML)
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self):
        self._stop_evt.set()
        if self.ok:
            self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------
def time_steps(torch, batch, action_pool, steps, warmup, sort_by_k, flush, collect_substeps=True):
    """Returns (sum of per-step device ms, total substeps, launches) for `steps` timed steps."""
    A = action_pool.shape[0]
    for i in range(warmup):
        batch.step_device(action_pool[i % A], auto_reset=True, sort_by_k=sort_by_k)
    torch.cuda.synchronize()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    sub_total = torch.zeros((), dtype=torch.int64, device=action_pool.device)
    l0 = batch.launch_count
    for i in range(steps):
        a = action_pool[(warmup + i) % A]
        starts[i].record()
        batch.step_device(a, auto_reset=True, sort_by_k=sort_by_k)
        ends[i].record()
        if collect_substeps:
            sub_total += batch.dev["substeps"].sum()
        if flush is not None:
            flush.zero_()                      # evict L2 between timed steps (outside the event pairs)
    torch.cuda.synchronize()
    launches = batch.launch_count - l0
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    return ms, int(sub_total.item()), launches


def run_cuda_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from grasp_lab_salp_b200 import PRECISION_F64, PRECISION_MIXED, SalpBatch, _lib, default_params
    from grasp_lab_salp_b200.params import sort_by_k_auto

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the SALP simulator has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # keep stdout for the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    n = args.envs
    prec = PRECISION_MIXED if args.precision == "mixed" else PRECISION_F64
    params = default_params(precision=prec)
    lib = _lib.load()

    def make_batch(n_envs):
        b = SalpBatch(n_envs, params, seed=0, env_id_offset=rank * n_envs, device=local)
        b.reset_device()
        return b

    def action_pool(n_envs, A=32):
        g = torch.Generator(device=dev)
        g.manual_seed(1234 + rank)
        u = torch.rand((A, n_envs, 3), generator=g, device=dev, dtype=torch.float32)
        u[..., 2] = u[..., 2] * 2 - 1
        return u.contiguous()

    def sort_flag(n_envs):
        if args.sort_by_k == "auto":
            return sort_by_k_auto(n_envs)    # one warp per SM sub-partition or less: the longest warp decides
        return args.sort_by_k == "on"

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    # ---- FP32 peak probe (roofline denominator) ----
    tf = _lib.C.c_double(0.0)
    rc = lib.salp_probe_fp32_peak(local, 300, _lib.C.byref(tf))
    fp32_peak = float(tf.value) if rc == 0 and tf.value > 0 else None

    batch = make_batch(n)
    pool = action_pool(n)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    ms, substeps, launches = time_steps(torch, batch, pool, args.steps, args.warmup, sort_flag(n), flush)
    barrier()
    clocks = sampler.stop()
    batch.check()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batch)
    step_kernel_name = batch.last_step_kernel          # what the launcher picked (salp_last_step_kernel)
    ms = max_over_ranks(ms)
    total_env_steps = sum_over_ranks(float(n * args.steps))
    total_substeps = sum_over_ranks(float(substeps))
    sec = ms * 1e-3
    value = total_env_steps / sec
    sub_rate = total_substeps / sec
    achieved_tf = sub_rate / world * FLOP_PER_SUBSTEP / 1e12      # per GPU
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    bytes_per_env_step = state_bytes_per_env_step(params)
    hbm_achieved = (total_env_steps / world) * bytes_per_env_step / sec / 1e9

    # ---- e2e: host buffers through the C ABI (salp_step_host), H2D + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        hb = SalpBatch(n, params, seed=0, env_id_offset=rank * n, device=local)
        hb.reset()
        host_actions = [hb.host_buffer((n, 3), np.float32) for _ in range(8)]
        pool_h = pool[:8].cpu().numpy()
        for k in range(8):
            host_actions[k][:] = pool_h[k]
        for i in range(max(3, args.warmup)):
            hb.step(host_actions[i % 8], auto_reset=True, sort_by_k=sort_flag(n), extras=False)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            hb.step(host_actions[i % 8], auto_reset=True, sort_by_k=sort_flag(n), extras=False)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        barrier()
        D = params.obs_dim
        e2e = {"value": total_env_steps / dt, "unit": METRIC, "h2d_bytes_per_step": n * 3 * 4,
               "d2h_bytes_per_step": n * (D * 4 * 2 + 4 + 1 + 1), "ms_per_step": 1e3 * dt / args.steps,
               "api": "SalpBatch.step -> salp_step_host (page-locked host buffers, wall clock around synchronous calls; "
                      + ("staged H2D/D2H copies" if sort_flag(n) else "kernel reads/writes the mapped host buffers directly") + ")"}
        hb.close()

    # ---- env-count sweep (BASELINE config 5) : where the GPU saturates ----
    sweep = None
    if not args.no_sweep:
        sweep = []
        for ne in (1024, 8192, 16384, 65536, 262144, 1048576):     # (8192 and 16384: BASELINE configs 4 and 3)
            b = make_batch(ne)
            p = action_pool(ne, A=8)
            st = max(5, min(40, int(4e6 // ne) + 5))
            m, s, _ = time_steps(torch, b, p, st, 3, sort_flag(ne), flush)
            m = max_over_ranks(m)
            tot = sum_over_ranks(float(ne * st))
            ssum = sum_over_ranks(float(s))
            row = {"envs_per_gpu": ne, "steps": st, "env_steps_per_sec": tot / (m * 1e-3),
                   "substeps_per_sec": ssum / (m * 1e-3), "sort_by_k": sort_flag(ne),
                   "fp32_tflops_per_gpu": ssum / world / (m * 1e-3) * FLOP_PER_SUBSTEP / 1e12}
            if fp32_peak:
                row["frac_of_measured_fp32"] = row["fp32_tflops_per_gpu"] / fp32_peak
            row["kernel"] = b.last_step_kernel
            if not args.no_e2e:      # the same rows through salp_step_host (page-locked host buffers, wall clock)
                b.reset()
                ha = [b.host_buffer((ne, 3), np.float32) for _ in range(2)]
                ph = p[:2].cpu().numpy()
                ha[0][:] = ph[0]
                ha[1][:] = ph[1]
                for k in range(3):
                    b.step(ha[k % 2], auto_reset=True, sort_by_k=sort_flag(ne), extras=False)
                es = max(5, st // 2)
                barrier()
                t0 = time.perf_counter()
                for k in range(es):
                    b.step(ha[k % 2], auto_reset=True, sort_by_k=sort_flag(ne), extras=False)
                dt_h = max_over_ranks(time.perf_counter() - t0)
                row["e2e_env_steps_per_sec"] = sum_over_ranks(float(ne * es)) / dt_h
            sweep.append(row)
            b.close()
            del b, p

    # ---- synthetic input B (SURVEY 8d): actions of a random-init Gaussian policy, N(0, 1) clipped to
    # the Box -> ~50 % of a0/a1 are exactly 0 and ~16 % exactly 1: bimodal K ----
    input_b = None
    if not args.no_sweep:
        input_b = []
        for ne in sorted({n, 262144}):
            b = make_batch(ne)
            g = torch.Generator(device=dev)
            g.manual_seed(4321 + rank)
            p = torch.randn((8, ne, 3), generator=g, device=dev, dtype=torch.float32)
            p[..., :2].clamp_(0.0, 1.0)
            p[..., 2].clamp_(-1.0, 1.0)
            st = max(5, min(40, int(4e6 // ne) + 5))
            m, ssum, _ = time_steps(torch, b, p.contiguous(), st, 3, sort_flag(ne), flush)
            b.step_device(p[0], auto_reset=True, sort_by_k=sort_flag(ne), extras=True)
            K = b.dev["substeps"].float()
            edges = [0, 1, 50, 150, 350, 700, 1000, 1200, 1349]
            hist = torch.histogram(K.cpu(), bins=torch.tensor(edges, dtype=torch.float32))[0]
            m = max_over_ranks(m)
            input_b.append({"envs_per_gpu": ne, "steps": st, "sort_by_k": sort_flag(ne),
                            "env_steps_per_sec": sum_over_ranks(float(ne * st)) / (m * 1e-3),
                            "substeps_per_sec": sum_over_ranks(float(ssum)) / (m * 1e-3),
                            "mean_substeps_per_env_step": float(ssum) / (ne * st),
                            "K_histogram": {"edges": edges, "share": [round(float(x) / ne, 4) for x in hist]}})
            b.close()
            del b, p

    cpu = cpu_port = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, cpu_port = cpu_baseline(args.cpu_seconds, total_envs=n)

    if rank == 0:
        peak = fp32_peak or NOMINAL_FP32_TFLOPS
        line = {
            "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if prec == PRECISION_MIXED else "f64", "data": "synthetic",
            "config": common_config(n, world),
            "config_detail": {"precision": args.precision, "sort_by_k": sort_flag(n), "l2": "flushed between timed steps "
                              "(256 MiB memset outside the per-step event pairs)"},
            "substeps_per_sec": sub_rate, "mean_substeps_per_env_step": total_substeps / total_env_steps,
            "roofline": {"bound": "fp32", "achieved": achieved_tf, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak, "traffic": ncu_traffic(n, args.precision),
                         "traffic_source": "profiles/traffic.json (ncu --set full capture of this workload, committed; not measured in this run)",
                         "peak_source": ("measured in this run: salp_probe_fp32_peak (FFMA, 2048 thr/SM)"
                                         if fp32_peak else "nominal"),
                         "nominal_peak": NOMINAL_FP32_TFLOPS, "frac_of_nominal": achieved_tf / NOMINAL_FP32_TFLOPS,
                         "flop_per_substep": FLOP_PER_SUBSTEP, "kernel": step_kernel_name,
                         "hbm": {"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": hbm_achieved / hbm_peak, "bytes_per_env_step": bytes_per_env_step,
                                 "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}},
            "clocks": clocks, "gpu_launches": int(launches),
        }
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if cpu_port:
            line["cpu_baseline_port"] = cpu_port
        if sweep:
            line["sweep"] = sweep
        if input_b:
            line["input_b_gaussian_policy_actions"] = input_b
        emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20
DUMP_OUTPUTS = ("obs", "reward", "terminated", "truncated", "terminal_obs", "substeps")


def dump_outputs(out_dir, batch):
    """What the last timed step handed its caller -- SalpBatch.step_device's (obs, reward, terminated,
    truncated) and the terminal_obs / substeps beside them -- as float32 DIR/<name>.npy (flags and
    substep counts are exact in float32).  Above DUMP_BYTES in all, the same rows of every array are
    written for a fixed, seeded sample of envs, and their indices as env_index.npy."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    n = batch.num_envs
    outs = {k: batch.dev[k].cpu().numpy().astype(np.float32) for k in DUMP_OUTPUTS}
    row_bytes = sum(a[0].nbytes for a in outs.values())
    budget = DUMP_BYTES - 128 * (len(outs) + 1)        # less one .npy header per file
    if n * row_bytes > budget:
        m = budget // (row_bytes + 8)
        idx = np.sort(np.random.default_rng(0).choice(n, m, replace=False))
        outs = {k: a[idx] for k, a in outs.items()}
        outs["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in outs.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def ncu_traffic(envs, precision):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE step-kernel launch from the committed
    `ncu --set full` capture of this workload (profiles/traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(f"{precision}:{envs}")
    except Exception:
        return None


def state_bytes_per_env_step(params):
    """Algorithmic HBM bytes of one env-step: every state column read + written once, plus the
    I/O rows (actions in; obs, reward, flags, terminal obs, substeps out)."""
    from grasp_lab_salp_b200.params import NUM_F64_FIELDS
    D = params.obs_dim
    cols = NUM_F64_FIELDS * 8 + (6 + 2 * params.num_obstacles) * 4 + 4 * 4
    return 2 * cols + 12 + (2 * D * 4 + 4 + 2 + 4)


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line goes to the process's original stdout; everything else any library
    prints (NCCL's version banner, torchrun notices) has been rerouted to stderr."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: re-launch under torchrun, one rank per GPU
        port = 29500 + (os.getpid() % 2000)
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                                   f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
                                   "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    run_cuda_arm(args)


if __name__ == "__main__":
    main()
