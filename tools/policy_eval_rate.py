#!/usr/bin/env python
"""Rate of deterministic policy evaluation (the reference's test_evaluate.py workflow: frozen VecNormalize,
model.predict(obs, deterministic=True) every control interval, then steady-state MAE/RMSE, settling time and
control energy) on hr_sync and pmsm_sync, N in {4,096, 65,536}, T = 2000.  Three arms, each warmed up, then
alternated REPS times and timed with CUDA events:
  fused  -- rl_ops.evaluate_policy: one cl_policy_rollout launch, metrics accumulated in registers;
  eager  -- torch loop: policy (float32 MLP, TF32 off) -> ChaosBatch.step -> err / ctrl stored as f64
            [T][c][N] -> rl_ops.eval_metrics;
  graph  -- the same loop captured as one CUDA graph (env in graph mode) and replayed.
With --variant-lib (a build with -DCL_POLICY_W_PARAM=1, tools/build_variant.sh) the fused arm is also run with
the weights as a __grid_constant__ kernel parameter instead of shared memory, alternated with the default build
in the same process.  Reports env-steps/s and the MLP's algorithmic rate (9,216 flop per env-step) as a share
of the measured FFMA peak (ChaosBatch-independent micro-kernel, measure_fma_peak(dtype_bytes=4)).
Writes one JSON line per (kind, N, arm) to --out; the GPU name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from gym_lorenz_b200 import _lib as L, rl_ops  # noqa: E402
from gym_lorenz_b200.core import ChaosBatch, measure_fma_peak  # noqa: E402

FLOP_PER_ENV_STEP = 2 * (6 * 64 + 64 * 64 + 64 * 2)   # 9,216: the MLP's multiply-adds


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


def modules(dev):
    torch.manual_seed(0)
    pnet = torch.nn.Sequential(torch.nn.Linear(6, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh())
    anet = torch.nn.Linear(64, 2)
    return pnet.to(dev), anet.to(dev)


def variant_lib(path):
    lib = C.CDLL(path)
    for name, res, args in L.SYMBOLS:
        if name == "cl_policy_rollout":
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    return lib


def timed(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def run_case(kind, n, T, reps, var_lib, fma_peak, info):
    dev = torch.device("cuda:0")
    b = ChaosBatch(kind, n, seed=1, autoreset=False, max_episode_steps=100000, add_noise=True,
                   **({"eval_mode": True} if kind == "hr_sync" else {}))
    b.reset()
    pnet, anet = modules(dev)
    params = rl_ops.pack_policy((pnet, anet), dev, kind)
    norm = None
    if kind == "pmsm_sync":
        art = json.load(open(os.path.join(ROOT, "tests", "golden", "sb3_artefacts.json")))["runs"]["0.50"]
        import types
        norm = rl_ops.DeviceVecNormalize(types.SimpleNamespace(batch=b, num_envs=n), training=False)
        norm.obs_rms.mean.copy_(torch.tensor(art["obs_mean"], dtype=torch.float64))
        norm.obs_rms.var.copy_(torch.tensor(art["obs_var"], dtype=torch.float64))
    obs = b._view(b.obs_planes)
    err = torch.empty((T, 3, n), dtype=torch.float64, device=dev)
    ctrl = torch.empty((T, 2, n), dtype=torch.float64, device=dev)
    xn = torch.empty((n, 6), dtype=torch.float32, device=dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    main_lib = b.lib

    def fused(lib=main_lib):
        b.lib = lib
        try:
            rl_ops.evaluate_policy(b, params, T, normalize=norm)
        finally:
            b.lib = main_lib

    @torch.no_grad()
    def loop():
        for t in range(T):
            x = obs if norm is None else norm.normalize_obs(obs, xn)
            a = torch.clamp(anet(pnet(x)), -1.0, 1.0)
            o, _, _ = b.step(a)
            err[t].copy_(o[:, :3].t())
            ctrl[t].copy_(a.t())
        return rl_ops.eval_metrics(err, ctrl, dt=0.001)

    arms = {"fused": fused, "eager": loop}
    if var_lib is not None:
        arms["fused_wparam"] = lambda: fused(var_lib)
    for fn in arms.values():   # warm-up (module load, cuBLAS heuristics, allocator)
        fn()
    torch.cuda.synchronize()
    b.set_graph_mode(True)
    loop()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        loop()
    g.replay()
    arms["graph"] = g.replay
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    b.set_graph_mode(False)
    rows = []
    for k, ts in times.items():
        ts = sorted(ts)
        med = ts[len(ts) // 2]
        rate = n * T / med
        tflops = rate * FLOP_PER_ENV_STEP / 1e12
        rows.append({"kind": kind, "n": n, "T": T, "arm": k, "seconds_median": med, "seconds_all": ts,
                     "env_steps_per_s": rate, "mlp_tflops": tflops, "ffma_peak_tflops": fma_peak,
                     "mlp_share_of_ffma_peak": tflops / fma_peak, **info})
    b.close()
    del g
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="policy_eval_rate.jsonl")
    ap.add_argument("--T", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--envs", default="4096,65536")
    ap.add_argument("--kinds", default="hr_sync,pmsm_sync")
    ap.add_argument("--variant-lib", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("policy_eval_rate needs a GPU")
    info = gpu_info()
    var_lib = variant_lib(a.variant_lib) if a.variant_lib else None
    fma_peak = measure_fma_peak(0, dtype_bytes=4, seconds=0.5)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for kind in a.kinds.split(","):
            for n in (int(x) for x in a.envs.split(",")):
                for row in run_case(kind, n, a.T, a.reps, var_lib, fma_peak, info):
                    f.write(json.dumps(row) + "\n")
                    f.flush()
                    print(f'{kind:10s} N={n:6d} {row["arm"]:13s} {row["seconds_median"] * 1e3:9.2f} ms '
                          f'{row["env_steps_per_s"]:.3e} env-steps/s  MLP {row["mlp_tflops"]:6.2f} TFLOP/s '
                          f'= {row["mlp_share_of_ffma_peak"]:.3f} of FFMA peak', flush=True)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
