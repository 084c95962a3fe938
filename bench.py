#!/usr/bin/env python
"""bench.py -- env-steps/s of the hot path on B200 (contract: see the task statement).

Workload (BASELINE.json configs[1]): Lorenz targeting env, 65,536 parallel envs per GPU, FP64
RK4 with S=16 substeps per control interval (the smallest power of two that meets the
rtol-1e-9 bar against adaptive integration, tests/test_rk4_vs_scipy.py), random actions.

One bench "step" = one rollout chunk: T control intervals for every env, executed by ONE
launch of the fused rollout kernel (`cl_rollout`).  Inputs: a pre-generated random action
tensor f32 [T, 3, n_pad] resident in HBM; outputs streamed to HBM every interval: obs f32
[T, 6, n_pad], reward f64 [T, n_pad], done u8 [T, n_pad].  With T=256 the per-step streams
(201 MB in, 554 MB out) exceed the 126 MB L2, so no timed iteration finds its inputs cached.

`value`   = all ranks' env-steps / max-over-ranks device time (CUDA events), inputs in HBM.
`e2e`     = the same env, same metric, driven through the SB3-facing VecEnv API
            (`step_async(actions)` / `step_wait()`) with HOST buffers: per control interval a
            caller-owned (pageable) float32 ndarray of actions -- what stock SB3 passes -- is staged
            into pinned memory and crosses PCIe, and obs/reward/done come back as host arrays, all
            inside the timed region (the variant whose policy writes straight into the env's pinned
            staging buffer is reported next to it).
`cfg4`    = (N > 1 only) BASELINE.json configs[3]: 1,048,576 envs per GPU, FP64 and FP32, episode-
            statistics all-reduce after EVERY step, device-timed, max over ranks.
`roofline`= the fused rollout kernel against the FP64-FMA peak measured live by a
            register-resident DFMA chain (MEASURED_PEAKS.json carries no FP64 number), plus
            its HBM side against MEASURED_PEAKS.json's copy bandwidth.
`cpu_baseline` / `--impl reference` = the oracle's C restatement (OpenMP, all host cores) on
            a bounded sample of the same workload; the reference itself is single-env
            Python (~2.7e4 steps/s/core, BASELINE.md) and cannot travel to the GPU box.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
FLOP_PER_SUBSTEP = 87          # SURVEY 8d: Lorenz RK4 substep with 3-channel ZOH control
BYTES_PER_ENV_STEP = 12 + 24 + 8 + 1   # action f32x3 in; obs f32x6, reward f64, done u8 out
# per kind: (algorithmic flop per substep, bytes per env-step in the rollout streams, dtype, FMA width)
KIND_INFO = {
    "lorenz_rk4": (87, 12 + 24 + 8 + 1, "f64", 8),
    "lorenz_rk4_f32": (87, 12 + 24 + 4 + 1, "f32", 4),
    "pmsm_rk4": (2 * 91, 8 + 24 + 8 + 1, "f64", 8),     # master + slave, 91 flop each (SURVEY 8d)
}


ENV_TYPE = {"lorenz_rk4": "EnvLorenzRK4<double>", "lorenz_rk4_f32": "EnvLorenzRK4<float>", "pmsm_rk4": "EnvPMSMRK4"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--chunk", type=int, default=256, help="control intervals per bench step (T)")
    ap.add_argument("--substeps", type=int, default=16)
    ap.add_argument("--kind", default="lorenz_rk4")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg4", action="store_true", help="N>1: skip the 1,048,576-envs-per-GPU FP64/FP32 sub-record")
    ap.add_argument("--e2e-chunks", type=int, default=4, help="bench steps timed on the host-buffer path")
    ap.add_argument("--param-jitter", type=float, default=0.0,
                    help="per-env parameter randomisation: each env's sigma/rho/beta (sigma/gamma for PMSM) "
                         "is the nominal value times U(1-j, 1+j) (BASELINE.json configs[2])")
    ap.add_argument("--stats-every", type=int, default=16,
                    help="N>1: all-reduce the 64 B episode-statistics vector every this many bench steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (obs, reward, done) and "
                         "the env state it left, for a fixed seeded sample of envs, as DIR/<name>.npy "
                         "(float32/float64, at most 64 MB in all; rank r of several writes <name>_rank<r>.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def workload_config(args, world):
    return {
        "workload": (f"Lorenz targeting env (RK4 x {args.substeps} substeps, dt=0.01, FP64), "
                     f"{args.envs_per_gpu} envs/GPU, random actions (BASELINE.json configs[1])")
        if args.kind == "lorenz_rk4" else f"{args.kind} (RK4 x {args.substeps}), {args.envs_per_gpu} envs/GPU, random actions",
        "kind": args.kind, "envs_per_gpu": args.envs_per_gpu, "total_envs": args.envs_per_gpu * world,
        "substeps": args.substeps, "control_intervals_per_step": args.chunk, "param_jitter": args.param_jitter,
        "parallelism": f"env-slab x{world} (no data-path collective; 64 B NCCL stats all-reduce every "
                       f"{args.stats_every} steps on a side stream)",
        "l2": "per-step action/obs/reward streams (>=750 MB) exceed the 126 MB L2; env state "
              "(3 MB) lives in registers across the whole launch",
    }


DUMP_BYTES = 60 << 20   # --dump-outputs: array bytes of all ranks together (files under 64 MB)


def sample_outputs(batch, out, budget):
    """Host copies of what the last rollout returned -- obs [T, obs_dim, k], reward [T, k], done flags [T, k]
    (as float32) -- and of the env state [n_state, k] it left, for k envs drawn with a fixed seed: all of them
    when they fit in `budget` bytes."""
    import numpy as np
    import torch
    N, T = batch.num_envs, out["reward"].shape[0]
    per_env = (T * (batch.obs_dim * out["obs"].element_size() + out["reward"].element_size() + 4)
               + batch.state.shape[0] * batch.state.element_size())
    k = min(N, budget // per_env)
    ix = torch.as_tensor(np.sort(np.random.default_rng(0).choice(N, k, replace=False)), device=batch.device)
    return {"obs": out["obs"].index_select(2, ix).cpu().numpy(),
            "reward": out["reward"].index_select(1, ix).cpu().numpy(),
            "done": out["done"].index_select(1, ix).float().cpu().numpy(),
            "state": batch.state.index_select(1, ix).cpu().numpy()}


# ---------------------------------------------------------------- clocks sampler
class ClockSampler:
    """`nvidia-smi -lms` in the background for the duration of the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.th = index, [], None, None

    def _read(self):
        for ln in self.proc.stdout:
            cols = [c.strip() for c in ln.strip().split(",")]
            if len(cols) >= 6:
                self.rows.append(cols)

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
            time.sleep(0.3)   # let the first samples arrive before the timed region starts
        except Exception:  # noqa: BLE001
            self.proc = None
        return self

    def mark(self):
        return len(self.rows)

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:  # noqa: BLE001
                self.proc.kill()
            self.th.join(timeout=5)

    def summary(self, lo=0, hi=None):
        rows = self.rows[lo:hi] or self.rows
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in rows)]
        mx = float(rows[0][1]) if rows[0][1].replace(".", "").isdigit() else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(rows)}


# ---------------------------------------------------------------- CPU arms (oracle port)
def cpu_arm(args, budget_s):
    """Oracle C port, OpenMP on all host cores, on a bounded sample of the same workload.
    Returns (env_steps_per_s, cores, sample_text, T_sample, elapsed)."""
    from oracle import api as O
    n = args.envs_per_gpu
    threads = len(os.sched_getaffinity(0))   # all host cores, whatever OMP_NUM_THREADS torchrun exported
    O.set_threads(threads)
    orc = O.Oracle(args.kind, n, flags=O.F_AUTORESET, seed=0, substeps=args.substeps,
                   dt=0.001 if args.kind == "pmsm_rk4" else 0.01, act_limit=1.0, act_gain=50.0, max_episode_steps=1000,
                   param_jitter=args.param_jitter)
    orc.reset()
    t0 = time.perf_counter(); orc.rollout_timed(1); dt1 = time.perf_counter() - t0   # also warms up
    T = max(1, min(4096, int(budget_s / max(dt1, 1e-6))))
    t0 = time.perf_counter(); orc.rollout_timed(T); el = time.perf_counter() - t0
    sample = (f"{n} envs x {T} control intervals ({args.kind}, RK4 x {args.substeps}, synthetic Philox actions), "
              f"oracle/chaos_oracle.c -O2 OpenMP x{threads}, {el:.2f} s")
    # the same port on ONE core (the reference's gym path is single-threaded): ~2 s sample
    O.set_threads(1)
    T1 = max(1, int(2.0 / max(dt1 * threads, 1e-6)))
    t0 = time.perf_counter(); orc.rollout_timed(T1); el1 = time.perf_counter() - t0
    O.set_threads(threads)
    return n * T / el, threads, sample, n * T1 / el1, el


def run_reference(args):
    """--impl reference: the CPU implementation of the path on this box's host cores."""
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import api as O
    n = args.envs_per_gpu
    threads = len(os.sched_getaffinity(0))   # all host cores, whatever OMP_NUM_THREADS torchrun exported
    O.set_threads(threads)
    orc = O.Oracle(args.kind, n, flags=O.F_AUTORESET, seed=0, substeps=args.substeps,
                   dt=0.001 if args.kind == "pmsm_rk4" else 0.01, act_limit=1.0, act_gain=50.0, max_episode_steps=1000,
                   param_jitter=args.param_jitter)
    orc.reset()
    t0 = time.perf_counter(); orc.rollout_timed(1); dt1 = time.perf_counter() - t0
    # bounded sample per step: about 0.1 s of CPU work, whole run capped near 2 minutes
    per_step_budget = min(0.1, 120.0 / max(args.steps + args.warmup, 1))
    T = max(1, int(per_step_budget / max(dt1, 1e-6)))
    for _ in range(args.warmup):
        orc.rollout_timed(T)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.rollout_timed(T)
    el = time.perf_counter() - t0
    value = n * T * args.steps / el
    cfg = workload_config(args, max(world, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg, "reference_sample_intervals_per_step": T,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n} envs x {T} control intervals per step x {args.steps} steps, "
                                   f"oracle/chaos_oracle.c (C restatement, OpenMP x{threads}); the reference "
                                   f"itself is single-env Python and is not present on this box"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------- the B200 arm
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from gym_lorenz_b200 import distributed as D
    from gym_lorenz_b200.core import ChaosBatch, measure_fma_peak
    from gym_lorenz_b200.vec_env import BatchedChaosVecEnv

    rank, world, local = D.init_process_group()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one rank per GPU: each rank keeps to its own cores of its GPU's NUMA node (before any pinned
    # allocation, so first touch places the staging buffers there) -- see distributed.pin_rank_to_cores
    cores = D.pin_rank_to_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    slab = D.weak_slab(args.envs_per_gpu, world, rank)
    N, T, S = slab.num_envs, args.chunk, args.substeps
    flop_sub, bytes_step, dtype_name, fma_bytes = KIND_INFO[args.kind]

    env_dt = 0.001 if args.kind == "pmsm_rk4" else 0.01
    batch = ChaosBatch(args.kind, N, device=dev, seed=0, env_id_base=slab.env_id_base, substeps=S,
                       dt=env_dt, autoreset=True, max_episode_steps=1000, param_jitter=args.param_jitter)
    batch.reset()
    NP = batch.n_pad
    # synthetic random actions, SoA time-major, resident in HBM before the timed region
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    act_soa = torch.rand((T, batch.act_dim, NP), generator=g, device=dev, dtype=torch.float32) * 2 - 1
    actions = act_soa[:, :, :N].permute(0, 2, 1)       # [T, N, A] view, env stride 1
    out = {"obs": torch.empty((T, batch.obs_dim, NP), dtype=torch.float32, device=dev),
           "reward": torch.empty((T, NP), dtype=batch.real, device=dev),
           "done": torch.empty((T, NP), dtype=torch.uint8, device=dev)}
    side = torch.cuda.Stream(device=dev)

    step_no = [0]

    def one_step():
        batch.rollout(T, actions, out=out)
        step_no[0] += 1
        if world > 1 and step_no[0] % args.stats_every == 0:
            # cumulative episode statistics, all-reduced on a side stream off the critical path
            st = batch.stats_tensor(clear=False)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                D.allreduce_stats(st)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()
    l0 = batch.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        m0 = clk.mark()
        e0.record()
        for _ in range(args.steps):
            one_step()
        e1.record()
        barrier()
        l1 = batch.launch_count
        m1 = clk.mark()
        # what the last timed step computed, before the passes below overwrite `out` and advance the envs
        dumped = sample_outputs(batch, out, DUMP_BYTES // world) if args.dump_outputs else None
        # kernel-only duration of the dominant kernel (rollout launches back to back, same stream)
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(args.steps):
            batch.rollout(T, actions, out=out)
        k1.record()
        torch.cuda.synchronize(dev)
        # short runs (small --steps): keep the same load running, untimed, until the sampler has
        # seen >= 0.6 s of it, so that `clocks` describes the GPU under THIS load, not idle
        t_load = time.perf_counter()
        while (time.perf_counter() - t_load) < 0.6 and (clk.mark() - m0) < 10:
            for _ in range(20):
                batch.rollout(T, actions, out=out)
            torch.cuda.synchronize(dev)
        m2 = clk.mark()
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        sfx = f"_rank{rank}" if world > 1 else ""
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{name}{sfx}.npy"), a)
    kern_ms = k0.elapsed_time(k1) / args.steps
    clocks = clk.summary(m0, max(m2, m0 + 1))
    clocks["samples_in_timed_region"] = m1 - m0
    ms = e0.elapsed_time(e1)
    launches = l1 - l0
    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_all = float(tmax.item())
    env_steps = float(N) * T * args.steps * world
    value = env_steps / (ms_all * 1e-3)
    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)"
        fp64_peak = measure_fma_peak(local, fma_bytes, 0.2)
        flops = float(N) * T * S * flop_sub
        ach = flops / (kern_ms * 1e-3) * 1e-12
        gbs = float(N) * T * bytes_step / (kern_ms * 1e-3) * 1e-9
        dyn = batch.dyn_launch_count > 0
        sm_local = batch.sm_launch_count > 0
        plain = ", PLAIN=true" if batch.plain_launch_count > 0 else ""   # which instantiation launch_env picked
        traffic = traffic_detail = None
        try:   # DRAM bytes per launch from the committed ncu --set full capture of this exact workload
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            w = tj["workload"]
            if (w["kind"], w["envs"], w["chunk"], w["substeps"]) == (args.kind, N, T, S) and dyn:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                traffic_detail = {"dram_bytes_read": tj["dram_bytes_read"], "dram_bytes_write": tj["dram_bytes_write"],
                                  "algorithmic_bytes": int(N) * T * bytes_step, "source": tj["source"]}
        except Exception:  # noqa: BLE001
            pass
        roofline = {
            "kernel": (f"cl::k_rollout_sm<{ENV_TYPE[args.kind]}> (fused T-interval rollout; per SM: resident env-warps in registers, "
                       f"guest env-warps chunked through a shared-memory queue, actions by tensor copies)" if sm_local
                       else f"cl::k_rollout_dyn<{ENV_TYPE[args.kind]}{plain}> (fused T-interval rollout, env-warp x chunk tasks)" if dyn
                       else f"cl::k_step<{ENV_TYPE[args.kind]}, ROLL=true{plain}> (fused T-interval rollout)"),
            "bound": "fp64" if fma_bytes == 8 else "fp32", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": ach / fp64_peak if fp64_peak > 0 else None, "traffic": traffic, "traffic_detail": traffic_detail,
            "peak_source": "DFMA-chain micro-kernel (cl_measure_fma_peak) run in this process, 2 flop/FMA; "
                           "MEASURED_PEAKS.json has no FP64 entry",
            "algorithmic_flop_per_substep": flop_sub,
            # the integrator works on z - rho (envs_northstar.cuh): 45 FP64-pipe instructions = 82 executed
            # flop per substep for the 87 algorithmic ones, so the 2-flop-per-FMA ceiling is 87 / 90
            "executed_fp64_instr_per_substep": 45, "executed_flop_per_substep": 82,
            "fma_issue_ceiling": 87.0 / (2 * 45),
            "kernel_ms_per_launch": kern_ms,
            "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                    "bytes_per_env_step": bytes_step, "peak_source": hbm_src},
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_all / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": dtype_name, "data": "synthetic",
            "config": workload_config(args, world), "substeps_per_s": value * S,
            "roofline": roofline, "clocks": clocks, "gpu_launches": int(launches),
            "block_size": batch.block_size,
        }

    # ---- e2e: the SB3-facing VecEnv API with host buffers -------------------------------------
    # Per control interval: the caller's (pageable) action array is staged into pinned host memory by the
    # library's staging lanes while the step kernel, already launched, reads it slice by slice; obs / reward /
    # done travel device->host; `infos` bookkeeping for finished episodes included.
    e2e = None
    if not args.no_e2e:
        env = BatchedChaosVecEnv(args.kind, N, device=dev, seed=0, env_id_base=slab.env_id_base,
                                 substeps=S, dt=env_dt, max_episode_steps=1000, param_jitter=args.param_jitter)
        env.reset()
        rng = np.random.default_rng(rank)
        host_actions = [rng.uniform(-1, 1, (N, env.batch.act_dim)).astype(np.float32) for _ in range(8)]
        chunks = max(1, min(args.e2e_chunks, args.steps))
        for k in range(32):
            env.step(host_actions[k % 8])
        barrier()
        # headline: a caller-owned ndarray every step (stock SB3: collect_rollouts passes the policy's
        # freshly produced action array)
        t0 = time.perf_counter()
        acc = 0.0
        for k in range(chunks * T):
            obs, rew, dones, infos = env.step(host_actions[k % 8])
            acc += float(rew[0])
        torch.cuda.synchronize(dev)
        el = time.perf_counter() - t0
        tm = torch.tensor([el], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        # side number: the policy writes its actions straight into the env's pinned staging buffer
        pin = env.batch.host_action_buffer()          # pinned f32 [N, act_dim]
        pin[:] = host_actions[0]
        for k in range(8):
            env.step(pin)
        t0 = time.perf_counter()
        for k in range(T):
            obs, rew, dones, infos = env.step(pin)
        torch.cuda.synchronize(dev)
        el_pin = (time.perf_counter() - t0) / T
        e2e = {"value": float(N) * T * chunks * world / float(tm.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(env.batch.h2d_bytes_per_step * T),
               "d2h_bytes_per_step": int(env.batch.d2h_bytes_per_step * T),
               "api": "BatchedChaosVecEnv.step_async(actions)/step_wait() (SB3 VecEnv contract); a caller-owned pageable "
                      "float32 ndarray of actions every step, obs/reward/done returned as host arrays; "
                      f"{T} control intervals per bench step, {chunks} bench steps timed, wall clock, max over ranks",
               "us_per_control_interval": float(tm.item()) / (chunks * T) * 1e6,
               "us_per_control_interval_pinned_inputs_rank0": el_pin * 1e6,
               "host_cores_of_rank0": len(cores)}
        env.close()

    cfg4 = None
    if world > 1 and not args.no_cfg4:
        cfg4 = run_cfg4(args, torch, dist, D, ChaosBatch, measure_fma_peak, rank, world, local, dev)

    if rank == 0:
        line["e2e"] = e2e
        if cfg4 is not None:
            line["cfg4"] = cfg4
        if not args.no_cpu_baseline and world == 1:
            v, cores, sample, v1, _ = cpu_arm(args, budget_s=12.0)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "single_core_value": v1,
                                    "note": "C/OpenMP restatement of the reference's scheme (oracle/chaos_oracle.c); the "
                                            "unmodified Python reference cannot travel to the GPU box -- in the build "
                                            "container its env classes ran at 1.2e4-2.5e4 steps/s on one core "
                                            "(profiles/r01_reference_python_container.json), ~100x below this port's "
                                            "single-core rate, so every ratio against this baseline is conservative"}
        print(json.dumps(line), flush=True)
    batch.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_cfg4(args, torch, dist, D, ChaosBatch, measure_fma_peak, rank, world, local, dev):
    """BASELINE.json configs[3]: 8 Mi envs over 8 GPUs = 1,048,576 envs per rank (weak scaling at any N),
    Lorenz RK4 x 16, FP64 and FP32, the 64 B episode-statistics vector all-reduced (NCCL) after EVERY
    rollout step.  Device-timed with CUDA events, max over ranks.  Returns the sub-record (rank 0) or None."""
    n, T, S, steps = 1 << 20, 16, 16, 12
    rec = {"envs_per_gpu": n, "total_envs": n * world, "control_intervals_per_step": T, "substeps": S, "steps": steps,
           "stats_allreduce": "every step"}
    for kind, key, fb in (("lorenz_rk4", "f64", 8), ("lorenz_rk4_f32", "f32", 4)):
        batch = ChaosBatch(kind, n, device=dev, seed=0, env_id_base=rank * n, substeps=S, dt=0.01, autoreset=True,
                           max_episode_steps=1000)
        batch.reset()
        NP = batch.n_pad
        g = torch.Generator(device=dev).manual_seed(99 + rank)
        act = torch.rand((T, batch.act_dim, NP), generator=g, device=dev, dtype=torch.float32) * 2 - 1
        actions = act[:, :, :n].permute(0, 2, 1)
        out = {"obs": torch.empty((T, batch.obs_dim, NP), dtype=torch.float32, device=dev),
               "reward": torch.empty((T, NP), dtype=batch.real, device=dev),
               "done": torch.empty((T, NP), dtype=torch.uint8, device=dev)}

        def step():
            batch.rollout(T, actions, out=out)
            D.allreduce_stats(batch.stats_tensor(clear=False))

        for _ in range(3):
            step()
        dist.barrier(); torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        dist.barrier(); torch.cuda.synchronize(dev)
        tmax = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item()) / steps
        value = float(n) * T * world / (ms * 1e-3)
        peak = measure_fma_peak(local, fb, 0.2) if rank == 0 else 0.0
        rec[key] = {"value": value, "unit": UNIT, "ms_per_step": ms,
                    "tflops_per_gpu": value / world * S * 87 * 1e-12,
                    "frac": (value / world * S * 87 * 1e-12 / peak) if peak > 0 else None, "peak_tflops": peak}
        batch.close()
        del act, actions, out
        torch.cuda.empty_cache()
    return rec if rank == 0 else None


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
