"""The C-ABI library loads and exports every symbol include/chaos_b200.h declares; no compute
is attempted without a GPU, and the product fails loudly instead of falling back."""
import ctypes as C
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    src = open(os.path.join(ROOT, "include", "chaos_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?[a-z_0-9]+\s*\*?\s*(cl_[a-z0-9_]+)\s*\(", src, flags=re.M)
    return sorted(set(names))


def test_header_declares_the_expected_surface():
    names = declared_functions()
    for must in ("cl_create", "cl_destroy", "cl_reset", "cl_step", "cl_rollout", "cl_stats",
                 "cl_step_host_async", "cl_step_host_wait", "cl_last_error", "cl_derivatives"):
        assert must in names


def test_library_exports_every_declared_symbol(chaos_lib):
    raw = C.CDLL(os.path.join(ROOT, "gym_lorenz_b200", "libchaos_b200.so"))
    missing = [n for n in declared_functions() if not hasattr(raw, n)]
    assert not missing, missing


def test_binding_covers_every_declared_symbol():
    from gym_lorenz_b200 import _lib
    bound = {s[0] for s in _lib.SYMBOLS}
    assert set(declared_functions()) <= bound


def test_layouts(chaos_lib):
    from gym_lorenz_b200 import _lib as L
    expect = {  # kind: (real_bytes, n_state, obs_dim, act_dim, act_low, act_high)
        "lorenz3": (8, 4, 6, 3, -500.0, 500.0),       # dynamic.py:18-19
        "lorenz3_pair": (8, 10, 6, 3, -500.0, 500.0),  # dynamic.py:122-123
        "lorenz4_pair": (8, 9, 8, 3, -2.0, 2.0),       # lorenz_env_transient.py:255-260
        "hr_sync": (8, 9, 6, 2, -1.0, 1.0),            # lorenz_env_try.py:27,31
        "pmsm_sync": (4, 9, 6, 2, -1.0, 1.0),          # lorenz_env_try_pmsm.py:40,43
        "pmsm_classic": (8, 7, 6, 2, -2.0, 2.0),
        "pmsm_single": (8, 4, 6, 2, -10.0, 10.0),
    }
    for name, (rb, ns, od, ad, lo, hi) in expect.items():
        lay = L.layout(L.KIND_NAMES[name])
        assert (lay.real_bytes, lay.n_state, lay.obs_dim, lay.act_dim, lay.act_low, lay.act_high) == \
            (rb, ns, od, ad, lo, hi), name
    assert L.layout(L.HR_SYNC).default_max_episode_steps == 5000    # gym_lorenz/__init__.py:12
    assert L.layout(L.PMSM_SYNC).default_max_episode_steps == 2000  # gym_lorenz/__init__.py:20


def test_create_validates_arguments(chaos_lib):
    from gym_lorenz_b200 import _lib as L
    ctx = C.c_void_p()
    bad = L.Config(abi_version=L.CL_ABI_VERSION, kind=99, num_envs=1, n_pad=128)
    assert chaos_lib.cl_create(C.byref(bad), C.byref(ctx)) == -1
    bad = L.Config(abi_version=L.CL_ABI_VERSION, kind=0, num_envs=100, n_pad=100)
    assert chaos_lib.cl_create(C.byref(bad), C.byref(ctx)) == -1
    assert b"n_pad" in chaos_lib.cl_last_error(None)
    bad = L.Config(abi_version=7, kind=0, num_envs=1, n_pad=128)
    assert chaos_lib.cl_create(C.byref(bad), C.byref(ctx)) == -1


def test_no_cpu_fallback_without_gpu():
    """Runs in a child process that sees no GPU (CUDA_VISIBLE_DEVICES empty), so it also runs where a GPU is present."""
    code = ("import sys\n"
            f"sys.path.insert(0, {ROOT!r})\n"
            "from gym_lorenz_b200 import ChaosLibError\n"
            "from gym_lorenz_b200.vec_env import BatchedChaosVecEnv\n"
            "try:\n"
            "    BatchedChaosVecEnv('hr_sync', 4)\n"
            "except ChaosLibError as e:\n"
            "    print('raised:', e)\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.startswith("raised:"), r.stdout


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gym_lorenz_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "chaos_oracle" not in text, f
                assert "ref_loader" not in text, f


def test_compat_package_has_the_reference_import_names():
    """`import gym_lorenz` / `from gym_lorenz.envs import HRSyncEnv, PMSM_Sync_Env` resolve to the
    GPU facades (reference: gym_lorenz/__init__.py:4-23, envs/__init__.py:2-3)."""
    import importlib
    import sys
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    try:
        for m in [k for k in sys.modules if k == "gym_lorenz" or k.startswith("gym_lorenz.")]:
            del sys.modules[m]
        pkg = importlib.import_module("gym_lorenz")
        envs = importlib.import_module("gym_lorenz.envs")
        assert hasattr(envs, "HRSyncEnv") and hasattr(envs, "PMSM_Sync_Env")
        assert envs.HRSyncEnv.__module__ == "gym_lorenz_b200.envs"
        assert pkg.REGISTERED in (True, False)
        import inspect
        assert list(inspect.signature(envs.HRSyncEnv.__init__).parameters)[1:4] == ["add_noise", "eval_mode", "add_filter"]
        assert list(inspect.signature(envs.PMSM_Sync_Env.__init__).parameters)[1:3] == ["alpha", "add_noise"]
    finally:
        sys.path.remove(os.path.join(ROOT, "compat"))
        for m in [k for k in sys.modules if k == "gym_lorenz" or k.startswith("gym_lorenz.")]:
            del sys.modules[m]


def test_lazy_infos_behaves_like_the_eager_list():
    """SB3 reads `infos` by index, by iteration and by slicing (VecMonitor: `list(infos[:])`)."""
    import numpy as np
    from gym_lorenz_b200.vec_env import _LazyInfos
    inf = _LazyInfos(5)
    inf._begin_step(([1, 3], np.arange(12, dtype=np.float32).reshape(2, 6), [True, False], [1.5, 2.5], [10, 20], 0.1))
    assert isinstance(inf, list) and len(inf) == 5
    assert inf[0] == {} and inf[1]["episode"] == {"r": 1.5, "l": 10, "t": 0.1}
    assert inf[3]["TimeLimit.truncated"] is False and inf[1]["terminal_observation"].tolist() == [0, 1, 2, 3, 4, 5]
    assert [bool(d) for d in inf] == [False, True, False, True, False]
    inf[1]["extra"] = 7                                  # wrappers may add keys to a done env's dict
    assert list(inf[:])[1]["extra"] == 7
    inf._begin_step(None)                                # next step: nothing finished
    assert all(d == {} for d in inf)
    inf._begin_step(([2], np.zeros((1, 6), np.float32), [True], None, None, 0.2))   # monitor off
    assert "episode" not in inf[2] and inf[2]["TimeLimit.truncated"] is True
