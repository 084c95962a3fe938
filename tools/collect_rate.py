#!/usr/bin/env python
"""Rate of PPO / A2C rollout collection (SB3 OnPolicyAlgorithm.collect_rollouts: actor-critic forward,
Gaussian sample, env step, TimeLimit bootstrap, buffer rows, GAE) on hr_sync and pmsm_sync.  Cases: both
kinds at 4,096 and 65,536 envs with n_steps = 256, plus hr_sync at 65,536 envs with n_steps = 2048
(code/train.py's PPO setting).  Three arms, each on its own batch, warmed up, then alternated REPS times and
timed with CUDA events (median reported):
  fused  -- rl_ops.FusedRolloutCollector: one cl_policy_collect launch + the GAE kernel;
  eager  -- rl_ops.DeviceRolloutCollector with the same-shaped torch actor-critic (TF32 off);
  graph  -- the same collector with its whole n_steps loop captured as one CUDA graph.
pmsm_sync runs with the frozen VecNormalize of tests/golden/sb3_artefacts.json, as the reference's A2C
pipeline normalises observations.  Reports env-steps/s and the MLP's algorithmic rate (18,304 flop per
env-step: actor 9,216 + critic 9,088) as a share of the FFMA peak measured in the same run
(measure_fma_peak(dtype_bytes=4)).  Writes one JSON line per (kind, N, T, arm) to --out; the GPU name and
power limit are read in the same run."""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from gym_lorenz_b200 import rl_ops  # noqa: E402
from gym_lorenz_b200.core import measure_fma_peak  # noqa: E402
from gym_lorenz_b200.vec_env import BatchedChaosVecEnv  # noqa: E402

FLOP_PER_ENV_STEP = 2 * (6 * 64 + 64 * 64 + 64 * 2) + 2 * (6 * 64 + 64 * 64 + 64 * 1)   # 18,304
CASES = [("hr_sync", 4096, 256), ("pmsm_sync", 4096, 256), ("hr_sync", 65536, 256), ("pmsm_sync", 65536, 256),
         ("hr_sync", 65536, 2048)]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if r.returncode == 0 else ("?", "?")
    return {"gpu": name, "power_limit": power}


class ActorCritic(torch.nn.Module):
    """SB3 ActorCriticPolicy parameter names (net_arch [64, 64], Tanh); forward is the collector interface."""

    def __init__(self):
        super().__init__()
        torch.manual_seed(0)
        mlp = lambda: torch.nn.Sequential(torch.nn.Linear(6, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64),
                                          torch.nn.Tanh())
        self.mlp_extractor = torch.nn.Module()
        self.mlp_extractor.policy_net, self.mlp_extractor.value_net = mlp(), mlp()
        self.action_net, self.value_net = torch.nn.Linear(64, 2), torch.nn.Linear(64, 1)
        self.log_std = torch.nn.Parameter(torch.full((2,), -0.5))

    def forward(self, obs):
        mu, std = self.action_net(self.mlp_extractor.policy_net(obs)), self.log_std.exp()
        a = mu + std * torch.randn_like(mu)
        # torch Normal.log_prob written out: the distribution's argument validation would synchronise
        logp = (-((a - mu) ** 2) / (2 * std ** 2) - std.log() - math.log(math.sqrt(2 * math.pi))).sum(-1)
        return a, self.value_net(self.mlp_extractor.value_net(obs)).squeeze(-1), logp


def normalizer(venv, kind):
    if kind != "pmsm_sync":
        return None
    art = json.load(open(os.path.join(ROOT, "tests", "golden", "sb3_artefacts.json")))["runs"]["0.50"]
    vn = rl_ops.DeviceVecNormalize(venv, training=False, norm_reward=False, clip_obs=art["clip_obs"],
                                   epsilon=art["epsilon"])
    vn.obs_rms.mean.copy_(torch.tensor(art["obs_mean"], dtype=torch.float64))
    vn.obs_rms.var.copy_(torch.tensor(art["obs_var"], dtype=torch.float64))
    return vn


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3


def run_case(kind, n, T, reps, fma_peak, info):
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    pol = ActorCritic().to(dev)
    venvs, arms = [], {}
    for arm in ("fused", "eager", "graph"):
        venv = BatchedChaosVecEnv(kind, n, seed=1)
        venvs.append(venv)
        norm = normalizer(venv, kind)
        if arm == "fused":
            col = rl_ops.FusedRolloutCollector(venv, pol, T, normalize=norm)
        else:
            col = rl_ops.DeviceRolloutCollector(norm if norm is not None else venv, pol, T,
                                                use_cuda_graph=arm == "graph")
        arms[arm] = col.collect
    for fn in arms.values():   # warm-up: module load, cuBLAS heuristics, allocator, graph capture
        fn()
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    rows = []
    for k, ts in times.items():
        ts = sorted(ts)
        med = ts[len(ts) // 2]
        rate = n * T / med
        tflops = rate * FLOP_PER_ENV_STEP / 1e12
        rows.append({"kind": kind, "n": n, "T": T, "arm": k, "seconds_median": med, "seconds_all": ts,
                     "env_steps_per_s": rate, "mlp_tflops": tflops, "ffma_peak_tflops": fma_peak,
                     "mlp_share_of_ffma_peak": tflops / fma_peak, **info})
    for venv in venvs:
        venv.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="collect_rate.jsonl")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cases", default="all", help="comma-separated kind:n:T, or 'all'")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("collect_rate needs a CUDA device")
    cases = CASES if args.cases == "all" else \
        [(c.split(":")[0], int(c.split(":")[1]), int(c.split(":")[2])) for c in args.cases.split(",")]
    info = gpu_info()
    fma_peak = measure_fma_peak(0, dtype_bytes=4)
    with open(args.out, "w") as f:
        for kind, n, T in cases:
            for row in run_case(kind, n, T, args.reps, fma_peak, info):
                print(json.dumps(row), flush=True)
                f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
