"""bench.py's JSON contract (the driver parses these lines): the reference arm is run here on a tiny
sample (CPU only), the B200 arm is checked on the committed line of the last measurement pass."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
             "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "gpu_launches"}


def _check_common(d):
    assert BASE_KEYS <= set(d), sorted(BASE_KEYS - set(d))
    assert d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["data"] == "synthetic" and d["dtype"] in ("f64", "f32")
    assert isinstance(d["config"].get("workload"), str) and "model" not in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e) and e["unit"] == d["unit"]
    c = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] in ("port", "reference") and c["cores"] >= 1


def test_reference_arm_line():
    env = dict(os.environ, OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                          "--warmup", "1", "--envs-per-gpu", "2048"], capture_output=True, text=True, env=env,
                         timeout=300, check=True).stdout.strip().splitlines()
    assert len(out) == 1, out                      # exactly ONE JSON line
    d = json.loads(out[0])
    _check_common(d)
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["steps"] == 2 and d["warmup"] == 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "1"], capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_committed_b200_line_has_the_contract_keys():
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r01*_bench_1gpu.json")))
    assert files, "no committed bench line under profiles/"
    d = json.load(open(files[-1]))
    _check_common(d)
    assert d["n_gpus"] == 1 and d["gpu_launches"] == d["steps"] > 0 and d["warmup"] >= 3
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
    assert r["traffic"] is None or isinstance(r["traffic"], (int, float))
    assert d["config"]["envs_per_gpu"] == 65536 and d["config"]["substeps"] == 16       # BASELINE configs[1]
    c = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(c)
    assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"]))
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["e2e"]["value"] < d["value"]          # the host-buffer path cannot repeat the device-timed number


@pytest.mark.gpu
def test_dump_outputs_are_repeatable_and_follow_steps(tmp_path):
    """--dump-outputs at the bench shape: float32/float64 arrays of at most 64 MB in all, identical for identical
    arguments.  Every warm-up and timed step is one rollout of the same envs, so the last timed step of 4 warm-up + 3
    timed steps computes what that of 3 + 4 does: equal dumps pin both --steps and the moment the dump is taken."""
    def run(warmup, steps, d):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                              "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, check=True).stdout.strip().splitlines()
        line = json.loads(out[-1])
        assert line["steps"] == line["gpu_launches"] == steps and line["warmup"] == warmup
        assert sum(f.stat().st_size for f in d.iterdir()) <= 64_000_000
        return {f.stem: np.load(f) for f in d.iterdir() if f.suffix == ".npy"}

    a, b, c = run(4, 3, tmp_path / "a"), run(4, 3, tmp_path / "b"), run(3, 4, tmp_path / "c")
    assert sorted(a) == ["done", "obs", "reward", "state"]
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    T, k = a["reward"].shape
    assert T == 256 and 0 < k <= 65536 and a["obs"].shape == (T, 6, k) and a["state"].shape[1] == k
    assert np.isin(a["done"], (0, 1, 2, 3)).all()
    # the state is the one the dumped step left: its last observation holds the positions (f32) of that state
    live = a["done"][-1] == 0
    assert live.any()
    assert np.array_equal(a["obs"][-1, :3, live], a["state"][:3, live].astype(np.float32).T, equal_nan=True)
    for name in a:
        assert np.array_equal(a[name], b[name], equal_nan=True), name
        assert np.array_equal(a[name], c[name], equal_nan=True), name
