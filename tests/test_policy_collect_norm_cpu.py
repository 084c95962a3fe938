"""FusedRolloutCollector(update_normalize=True) and cl_policy_collect_norm argument handling without a GPU:
the Python refusals, the frozen refusals unchanged, the C-ABI refusals reachable without a context, and the
scratch size."""
import ctypes as C
import types

import pytest
from gym_lorenz_b200 import rl_ops
from test_policy_collect_cpu import SB3Policy, _fake_env

CL_EINVAL = -1


def _vn(env, **kw):
    d = dict(training=True, norm_obs=True, norm_reward=False, num_envs=env.batch.num_envs, venv=env)
    d.update(kw)
    return types.SimpleNamespace(**d)


def test_update_normalize_refusals(chaos_lib):
    m = SB3Policy()
    env = _fake_env()
    with pytest.raises(ValueError, match="needs a DeviceVecNormalize"):
        rl_ops.FusedRolloutCollector(env, m, 8, update_normalize=True)
    with pytest.raises(ValueError, match="training mode"):
        rl_ops.FusedRolloutCollector(env, m, 8, normalize=_vn(env, training=False), update_normalize=True)
    with pytest.raises(ValueError, match="this collector's batch"):
        rl_ops.FusedRolloutCollector(env, m, 8, normalize=_vn(_fake_env()), update_normalize=True)
    with pytest.raises(ValueError, match="this collector's batch"):
        rl_ops.FusedRolloutCollector(env, m, 8, normalize=_vn(env, num_envs=5), update_normalize=True)
    with pytest.raises(ValueError, match="float32"):
        e64 = _fake_env(obs_f64=True)
        rl_ops.FusedRolloutCollector(e64, m, 8, normalize=_vn(e64), update_normalize=True)
    for kind in ("lorenz3", "pmsm_classic", "lorenz_rk4"):
        ek = _fake_env(kind)
        with pytest.raises(ValueError, match="hr_sync and pmsm_sync"):
            rl_ops.FusedRolloutCollector(ek, m, 8, normalize=_vn(ek), update_normalize=True)


def test_frozen_refusals_unchanged_and_name_the_new_keyword(chaos_lib):
    m = SB3Policy()
    env = _fake_env()
    frozen = dict(training=False, norm_obs=True, norm_reward=False)
    with pytest.raises(ValueError, match="normalize must be frozen \\(training=False\\); DeviceRolloutCollector "
                                         "updates the statistics every step") as e:
        rl_ops.FusedRolloutCollector(env, m, 8, normalize=types.SimpleNamespace(**{**frozen, "training": True}))
    assert "update_normalize=True" in str(e.value)
    with pytest.raises(ValueError, match="reward normalisation is not fused \\(norm_reward=False\\); use "
                                         "DeviceRolloutCollector") as e:
        rl_ops.FusedRolloutCollector(env, m, 8, normalize=types.SimpleNamespace(**{**frozen, "norm_reward": True}))
    assert "update_normalize=True" in str(e.value)


def test_c_abi_refusals_without_a_context(chaos_lib):
    from gym_lorenz_b200 import _lib as L
    args = [C.byref(x) for x in (L.Buffers(), L.IO(), L.RolloutDesc(T=4), L.Policy(), L.Collect(), L.VecNormUpdate())]
    assert chaos_lib.cl_policy_collect_norm(None, None, *args) == CL_EINVAL
    assert b"null ctx" in chaos_lib.cl_last_error(None)
    out = C.c_int64(-1)
    for kind in (L.LORENZ3, L.PMSM_CLASSIC, L.LORENZ_RK4, 99, -1):
        assert chaos_lib.cl_policy_collect_norm_scratch_bytes(kind, 1000, C.byref(out)) == CL_EINVAL
        assert b"hr_sync and pmsm_sync" in chaos_lib.cl_last_error(None)
    for n in (0, -5):
        assert chaos_lib.cl_policy_collect_norm_scratch_bytes(L.HR_SYNC, n, C.byref(out)) == CL_EINVAL
    assert chaos_lib.cl_policy_collect_norm_scratch_bytes(L.HR_SYNC, 10, None) == CL_EINVAL
    assert out.value == -1


def _scratch_bytes(n, obs_dim=6):
    up = lambda b: (b + 255) // 256 * 256
    slots = up(2 * ((n + 31) // 32) * (2 * obs_dim + 2) * 8)     # per-block partial sums, two parities
    return slots + up(8 * n) + up(4 * n) + up(4 * obs_dim * n)  # raw reward, done flags, pre-reset obs


@pytest.mark.parametrize("n", [1, 33, 1000, 65536, 262144, 1 << 22])
def test_scratch_bytes(chaos_lib, n):
    from gym_lorenz_b200 import _lib as L
    for kind in (L.HR_SYNC, L.PMSM_SYNC):
        out = C.c_int64(-1)
        assert chaos_lib.cl_policy_collect_norm_scratch_bytes(kind, n, C.byref(out)) == 0
        assert out.value == _scratch_bytes(n) and out.value % 256 == 0
