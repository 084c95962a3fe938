#!/usr/bin/env python
"""Rate of PPO / A2C rollout collection behind a VecNormalize in TRAINING mode (code/lorenz_pmsm/train.py's
A2C pipeline: the running statistics are updated every step) on hr_sync and pmsm_sync.  Four arms, each on
its own batch with the same weights and the same start statistics, warmed up, then alternated REPS times and
timed with CUDA events (median reported):
  fused_train  -- FusedRolloutCollector(update_normalize=True): one cl_policy_collect_norm launch + GAE;
  fused_frozen -- FusedRolloutCollector with the normaliser frozen (training=False): cl_policy_collect;
  graph        -- DeviceRolloutCollector over DeviceVecNormalize(training=True), n_steps loop as one CUDA graph;
  eager        -- the same collector without the graph.
Cases: both kinds at 4,096 and 65,536 envs with n_steps = 256, hr_sync at 65,536 x 2048 (code/train.py's
PPO n_steps), and 262,144 x 256 -- more envs than the fused training-mode grid holds co-resident, so its
threads own several envs each -- with the two fused arms only.  pmsm_sync starts from the statistics of
tests/golden/sb3_artefacts.json.  Reports env-steps/s and the MLP's algorithmic rate (collect_rate.py's
18,304 flop per env-step) as a share of the FFMA peak measured in the same run.  One JSON line per case
(all arms) to --out; the GPU name and power limit are read in the same run."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

from collect_rate import FLOP_PER_ENV_STEP, ActorCritic, gpu_info, timed  # noqa: E402
from gym_lorenz_b200 import rl_ops  # noqa: E402
from gym_lorenz_b200.core import measure_fma_peak  # noqa: E402
from gym_lorenz_b200.vec_env import BatchedChaosVecEnv  # noqa: E402

CASES = [("hr_sync", 4096, 256), ("pmsm_sync", 4096, 256), ("hr_sync", 65536, 256), ("pmsm_sync", 65536, 256),
         ("hr_sync", 65536, 2048), ("hr_sync", 262144, 256)]
FUSED_ONLY = 100_000   # above this many envs only the fused arms run


def normalizer(venv, kind, training):
    art = json.load(open(os.path.join(ROOT, "tests", "golden", "sb3_artefacts.json")))["runs"]["0.50"]
    vn = rl_ops.DeviceVecNormalize(venv, training=training, norm_reward=False, clip_obs=art["clip_obs"],
                                   epsilon=art["epsilon"], gamma=art["gamma"])
    if kind == "pmsm_sync":
        vn.obs_rms.mean.copy_(torch.tensor(art["obs_mean"], dtype=torch.float64))
        vn.obs_rms.var.copy_(torch.tensor(art["obs_var"], dtype=torch.float64))
        vn.obs_rms.count = float.fromhex(art["obs_count"])
        vn.ret_rms.mean.fill_(art["ret_mean"])
        vn.ret_rms.var.fill_(art["ret_var"])
        vn.ret_rms.count = float.fromhex(art["ret_count"])
    return vn


def run_case(kind, n, T, reps, fma_peak, info):
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    pol = ActorCritic().to(dev)
    names = ("fused_train", "fused_frozen") if n > FUSED_ONLY else ("fused_train", "fused_frozen", "graph", "eager")
    venvs, arms = [], {}
    for arm in names:
        venv = BatchedChaosVecEnv(kind, n, seed=1)
        venvs.append(venv)
        vn = normalizer(venv, kind, training=arm != "fused_frozen")
        if arm.startswith("fused"):
            col = rl_ops.FusedRolloutCollector(vn, pol, T, normalize=vn, update_normalize=arm == "fused_train")
        else:
            col = rl_ops.DeviceRolloutCollector(vn, pol, T, use_cuda_graph=arm == "graph")
        arms[arm] = col.collect
    for fn in arms.values():   # warm-up: module load, cuBLAS heuristics, allocator, graph capture
        fn()
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    row = {"kind": kind, "n": n, "T": T, **info, "ffma_peak_tflops": fma_peak, "arms": {}}
    for k, ts in times.items():
        ts = sorted(ts)
        med = ts[len(ts) // 2]
        rate = n * T / med
        tflops = rate * FLOP_PER_ENV_STEP / 1e12
        row["arms"][k] = {"seconds_median": med, "seconds_all": ts, "env_steps_per_s": rate, "mlp_tflops": tflops,
                          "mlp_share_of_ffma_peak": tflops / fma_peak}
    a = row["arms"]
    row["train_over_frozen"] = a["fused_train"]["env_steps_per_s"] / a["fused_frozen"]["env_steps_per_s"]
    if "graph" in a:
        row["train_over_graph"] = a["fused_train"]["env_steps_per_s"] / a["graph"]["env_steps_per_s"]
    for venv in venvs:
        venv.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="collect_train_rate.jsonl")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="all", help="comma-separated kind:n:T, or 'all'")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("collect_train_rate needs a CUDA device")
    cases = CASES if args.cases == "all" else \
        [(c.split(":")[0], int(c.split(":")[1]), int(c.split(":")[2])) for c in args.cases.split(",")]
    info = gpu_info()
    fma_peak = measure_fma_peak(0, dtype_bytes=4)
    with open(args.out, "w") as f:
        for kind, n, T in cases:
            row = run_case(kind, n, T, args.reps, fma_peak, info)
            print(json.dumps(row), flush=True)
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
