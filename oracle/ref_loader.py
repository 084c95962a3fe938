"""TEST INFRASTRUCTURE ONLY -- loads the *unmodified* reference env files.

The reference (a checkout of gym-lorenz named by ``GYM_LORENZ_REFERENCE``) is pure Python but imports ``gym`` / ``gymnasium`` /
``stable_baselines3`` / ``matplotlib`` at module top, none of which is installed in this
image.  The env classes only use ``gym.Env`` as a base class, ``spaces.Box`` and (PMSM)
``Env.reset(seed) -> self.np_random``.  This module injects minimal stub modules into
``sys.modules`` and then executes the reference files *by path*, unchanged, so the
arithmetic that runs is the reference's own.

The reference is not part of this repository: this module works only where
``GYM_LORENZ_REFERENCE`` points at a checkout of it.  It is used by
``tests/golden/make_golden.py`` to generate the committed fixtures and by the CPU test
suite to pin ``oracle/chaos_oracle.c``.  Nothing in the product package imports it, and
nothing on the GPU side of the suite depends on it.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

import numpy as np

REF_ROOT = os.environ.get("GYM_LORENZ_REFERENCE", "")
ENV_DIR = os.path.join(REF_ROOT, "code", "gym-lorenz", "gym_lorenz", "envs")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isdir(ENV_DIR)


class _Box:
    def __init__(self, low, high, shape=None, dtype=np.float32):
        self.low, self.high, self.shape, self.dtype = low, high, shape, dtype


class _Env:
    """Stand-in for gym.Env / gymnasium.Env: only what the reference touches."""

    metadata: dict = {}
    np_random = None

    def reset(self, seed=None, options=None):
        # gymnasium.Env.reset: (re)seed self.np_random with PCG64 when a seed is given
        # or when no generator exists yet.
        if seed is not None or self.np_random is None:
            self.np_random = np.random.default_rng(seed)


def _module(name: str, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    return m


_STUBBED = False


def _install_stubs() -> None:
    global _STUBBED
    if _STUBBED:
        return
    spaces = _module("spaces", Box=_Box)
    for root in ("gym", "gymnasium"):
        if root in sys.modules:
            continue
        sp = _module(root + ".spaces", Box=_Box)
        utils = _module(root + ".utils")
        seeding = _module(root + ".utils.seeding")
        utils.seeding = seeding
        err = _module(root + ".error")
        mod = _module(root, Env=_Env, spaces=sp, utils=utils, error=err)
        sys.modules[root] = mod
        sys.modules[root + ".spaces"] = sp
        sys.modules[root + ".utils"] = utils
        sys.modules[root + ".utils.seeding"] = seeding
        sys.modules[root + ".error"] = err
    del spaces
    if "stable_baselines3" not in sys.modules:
        sys.modules["stable_baselines3"] = _module("stable_baselines3", PPO=object)
    if "matplotlib" not in sys.modules:
        plt = _module("matplotlib.pyplot")
        mpl = _module("matplotlib", pyplot=plt)
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt
    if "mpl_toolkits" not in sys.modules:
        m3 = _module("mpl_toolkits.mplot3d", Axes3D=object)
        mt = _module("mpl_toolkits", mplot3d=m3)
        sys.modules["mpl_toolkits"] = mt
        sys.modules["mpl_toolkits.mplot3d"] = m3
    _STUBBED = True


_CACHE: dict = {}


def load(filename: str) -> types.ModuleType:
    """Execute ``envs/<filename>`` from the reference tree, unmodified."""
    if filename in _CACHE:
        return _CACHE[filename]
    if not available():
        raise FileNotFoundError(f"reference tree not found at {ENV_DIR}")
    _install_stubs()
    path = os.path.join(ENV_DIR, filename)
    spec = importlib.util.spec_from_file_location("_ref_" + filename[:-3], path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    _CACHE[filename] = mod
    return mod


# Convenience constructors, named after the reference classes they return -------------

def lorenz3():
    """dynamic.py outer class (3-D Lorenz driven to the origin), dynamic.py:5-93."""
    return load("dynamic.py").lorenzEnv_transient()


def lorenz3_pair():
    """dynamic.py nested class (frozen second Lorenz as target), dynamic.py:109-233."""
    return load("dynamic.py").lorenzEnv_transient.lorenzEnv_transient()


def lorenz4_pair():
    """lorenz_env_transient.py live class (4-D pair), :247-376."""
    return load("lorenz_env_transient.py").lorenzEnv_transient()


def hr_sync(**kw):
    """lorenz_env_try.py::HRSyncEnv."""
    return load("lorenz_env_try.py").HRSyncEnv(**kw)


def pmsm_sync(**kw):
    """lorenz_env_try_pmsm.py::PMSM_Sync_Env."""
    return load("lorenz_env_try_pmsm.py").PMSM_Sync_Env(**kw)


def pmsm_classic():
    """lorenz_env_transient_pmsm.py::lorenzEnv_transient."""
    return load("lorenz_env_transient_pmsm.py").lorenzEnv_transient()


def pmsm_single():
    """lorenz_env_transient1.py::lorenzEnv_transient (single PMSM to the origin)."""
    return load("lorenz_env_transient1.py").lorenzEnv_transient()


def memristive4_pair():
    """lorenz_env_transient2.py::lorenzEnv_transient (4-D memristive pair, u*100 control)."""
    return load("lorenz_env_transient2.py").lorenzEnv_transient()


def pmsm_free():
    """lorenz_singlecontrol.py::lorenzEnv_transient (uncontrolled noisy PMSM; step() has no action)."""
    return load("lorenz_singlecontrol.py").lorenzEnv_transient()


# ---- the reference's evaluation metrics (code/lorenz_pmsm/test_evaluate.py) -------------------

EVAL_SCRIPT = os.path.join(REF_ROOT, "code", "lorenz_pmsm", "test_evaluate.py")


def load_eval_script() -> types.ModuleType:
    """Execute code/lorenz_pmsm/test_evaluate.py unmodified (module level only: imports, rcParams,
    function definitions; its __main__ block does not run).  Needs stubs for the SB3 / matplotlib /
    env_utils / gym_lorenz imports at its top; pandas is real."""
    key = "lorenz_pmsm/test_evaluate.py"
    if key in _CACHE:
        return _CACHE[key]
    if not os.path.exists(EVAL_SCRIPT):
        raise FileNotFoundError(EVAL_SCRIPT)
    _install_stubs()
    sys.modules["matplotlib.pyplot"].rcParams = {}
    sb3 = sys.modules["stable_baselines3"]
    sb3.A2C = object
    for name, attrs in (("stable_baselines3.common", {}),
                        ("stable_baselines3.common.vec_env", {"DummyVecEnv": object, "VecNormalize": object}),
                        ("stable_baselines3.common.monitor", {"Monitor": object})):
        sys.modules.setdefault(name, _module(name, **attrs))
    sys.modules.setdefault("env_utils", _module("env_utils", make_env=None))
    sys.modules.setdefault("gym_lorenz", _module("gym_lorenz"))
    path_before = list(sys.path)
    try:
        spec = importlib.util.spec_from_file_location("_ref_lorenz_pmsm_test_evaluate", EVAL_SCRIPT)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.path[:] = path_before        # the script appends its gym-lorenz directory
    _CACHE[key] = mod
    return mod


def eval_steady_block():
    """The steady-state MAE / RMSE / settling-time block of test_evaluate.py (:239-250 -- inline code
    of the evaluation loop, not a function) compiled from the reference file's own lines.  Returns
    f(arr_e1, arr_e2, arr_e3, arr_u1, arr_u2, dt) -> (mae, rmse, max_ts, energy)."""
    import textwrap
    mod = load_eval_script()
    lines = open(EVAL_SCRIPT, encoding="utf-8").read().splitlines()
    first = next(k for k, ln in enumerate(lines) if "actual_steady_start = min(1000" in ln)
    last = next(k for k, ln in enumerate(lines) if "max_ts = np.nanmax([ts1, ts2, ts3])" in ln)
    assert 0 < last - first < 20
    code = compile(textwrap.dedent("\n".join(lines[first:last + 1])), EVAL_SCRIPT + f":{first + 1}-{last + 1}", "exec")

    def run(arr_e1, arr_e2, arr_e3, arr_u1, arr_u2, dt):
        ns = {"np": np, "calculate_advanced_metrics": mod.calculate_advanced_metrics, "arr_e1": arr_e1,
              "arr_e2": arr_e2, "arr_e3": arr_e3, "arr_u1": arr_u1, "arr_u2": arr_u2, "dt": dt}
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")          # np.nanmax of all-NaN settling times warns
            exec(code, ns)
        return ns["mae"], ns["rmse"], ns["max_ts"], ns["energy"]

    return run
