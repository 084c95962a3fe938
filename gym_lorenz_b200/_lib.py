"""ctypes binding of libchaos_b200.so (include/chaos_b200.h).

There is deliberately NO fallback: if the shared library is missing or fails to load, every
entry point of the package raises.  The CPU oracle under oracle/ is test infrastructure and is
never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# CHAOS_B200_LIB: tuning override (A/B runs of differently compiled builds, tools/ab_variants.sh)
LIB_PATH = os.environ.get("CHAOS_B200_LIB") or os.path.join(HERE, "libchaos_b200.so")

CL_ABI_VERSION = 1

# env kinds (cl_env_kind)
LORENZ3, LORENZ3_PAIR, LORENZ4_PAIR, HR_SYNC, PMSM_SYNC, PMSM_CLASSIC, PMSM_SINGLE = range(7)
LORENZ_RK4, LORENZ_RK4_F32, PMSM_RK4 = 7, 8, 9
MEMRISTIVE4_PAIR, PMSM_FREE = 10, 11
KIND_NAMES = {
    "lorenz3": LORENZ3, "lorenz3_pair": LORENZ3_PAIR, "lorenz4_pair": LORENZ4_PAIR,
    "hr_sync": HR_SYNC, "pmsm_sync": PMSM_SYNC, "pmsm_classic": PMSM_CLASSIC,
    "pmsm_single": PMSM_SINGLE, "lorenz_rk4": LORENZ_RK4, "lorenz_rk4_f32": LORENZ_RK4_F32,
    "pmsm_rk4": PMSM_RK4, "memristive4_pair": MEMRISTIVE4_PAIR, "pmsm_free": PMSM_FREE,
}

F_ADD_NOISE, F_EVAL_MODE, F_ADD_FILTER, F_AUTORESET, F_OBS_F64 = 0x01, 0x02, 0x04, 0x08, 0x10
DONE_TERMINATED, DONE_TRUNCATED = 0x1, 0x2
HOST_DMA, HOST_ZEROCOPY, HOST_PIPELINED, HOST_STREAMED = 0, 1, 2, 3
NSTATS = 8
STAT_NAMES = ("episodes", "return_sum", "return_sq_sum", "length_sum", "nonfinite_events",
              "terminated", "truncated", "reserved")


class ChaosLibError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("kind", C.c_int32), ("device", C.c_int32), ("flags", C.c_int32),
        ("num_envs", C.c_int64), ("n_pad", C.c_int64), ("env_id_base", C.c_int64),
        ("seed", C.c_uint64), ("max_episode_steps", C.c_int32), ("substeps", C.c_int32),
        ("dt", C.c_double), ("alpha", C.c_double), ("act_limit", C.c_double),
        ("act_gain", C.c_double), ("param_jitter", C.c_double),
    ]


class Layout(C.Structure):
    _fields_ = [
        ("real_bytes", C.c_int32), ("n_state", C.c_int32), ("n_int", C.c_int32),
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("noise_dim", C.c_int32),
        ("act_low", C.c_double), ("act_high", C.c_double),
        ("obs_low", C.c_double), ("obs_high", C.c_double),
        ("default_max_episode_steps", C.c_int32), ("reserved", C.c_int32),
    ]


class Buffers(C.Structure):
    _fields_ = [
        ("state", C.c_void_p), ("aux_int", C.c_void_p), ("ep_len", C.c_void_p),
        ("ep_return", C.c_void_p), ("stats", C.c_void_p),
    ]


class IO(C.Structure):
    _fields_ = [
        ("action", C.c_void_p), ("act_es", C.c_int64), ("act_cs", C.c_int64),
        ("noise", C.c_void_p),
        ("obs", C.c_void_p), ("obs_es", C.c_int64), ("obs_cs", C.c_int64),
        ("reward", C.c_void_p), ("done", C.c_void_p), ("term_obs", C.c_void_p),
        ("last_ep_ret", C.c_void_p), ("last_ep_len", C.c_void_p), ("mask", C.c_void_p),
    ]


class RolloutDesc(C.Structure):
    _fields_ = [
        ("T", C.c_int32), ("reserved", C.c_int32), ("act_ts", C.c_int64), ("obs_ts", C.c_int64),
        ("rew_ts", C.c_int64), ("done_ts", C.c_int64), ("synth_amp", C.c_double),
    ]


POLICY_HIDDEN = 64   # CL_POLICY_HIDDEN


class Policy(C.Structure):
    _fields_ = [
        ("params", C.c_void_p), ("obs_mean", C.c_void_p), ("obs_var", C.c_void_p),
        ("epsilon", C.c_double), ("clip_obs", C.c_double),
        ("obs0", C.c_void_p), ("obs0_es", C.c_int64), ("obs0_cs", C.c_int64),
        ("obs_last", C.c_void_p), ("act_out", C.c_void_p), ("metrics", C.c_void_p),
        ("steady_start", C.c_int32), ("dt", C.c_double), ("error_band", C.c_double),
    ]


class Collect(C.Structure):
    _fields_ = [
        ("gamma", C.c_double), ("starts", C.c_void_p), ("obs", C.c_void_p), ("actions", C.c_void_p),
        ("rewards", C.c_void_p), ("values", C.c_void_p), ("log_probs", C.c_void_p),
        ("episode_starts", C.c_void_p), ("last_values", C.c_void_p),
    ]


class VecNormUpdate(C.Structure):
    _fields_ = [
        ("obs_mean", C.c_void_p), ("obs_var", C.c_void_p), ("obs_count", C.c_void_p),
        ("ret_mean", C.c_void_p), ("ret_var", C.c_void_p), ("ret_count", C.c_void_p), ("returns", C.c_void_p),
        ("gamma", C.c_double), ("epsilon", C.c_double), ("clip_obs", C.c_double), ("clip_reward", C.c_double),
        ("norm_obs", C.c_int32), ("norm_reward", C.c_int32),
        ("scratch", C.c_void_p), ("scratch_bytes", C.c_int64),
    ]


class HostView(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
        ("term_obs", C.c_void_p), ("last_ep_ret", C.c_void_p), ("last_ep_len", C.c_void_p),
        ("n_done", C.c_int64),
    ]


# every symbol include/chaos_b200.h declares: (name, restype, argtypes)
_VP = C.c_void_p
SYMBOLS = [
    ("cl_abi_version", C.c_int, []),
    ("cl_env_layout", C.c_int, [C.c_int32, C.POINTER(Layout)]),
    ("cl_create", C.c_int, [C.POINTER(Config), C.POINTER(_VP)]),
    ("cl_destroy", C.c_int, [_VP]),
    ("cl_last_error", C.c_char_p, [_VP]),
    ("cl_reset", C.c_int, [_VP, _VP, C.POINTER(Buffers), C.POINTER(IO)]),
    ("cl_init_persistent", C.c_int, [_VP, _VP, C.POINTER(Buffers)]),
    ("cl_step", C.c_int, [_VP, _VP, C.POINTER(Buffers), C.POINTER(IO)]),
    ("cl_rollout", C.c_int, [_VP, _VP, C.POINTER(Buffers), C.POINTER(IO), C.POINTER(RolloutDesc)]),
    ("cl_policy_rollout", C.c_int, [_VP, _VP, C.POINTER(Buffers), C.POINTER(IO), C.POINTER(RolloutDesc),
                                    C.POINTER(Policy)]),
    ("cl_policy_collect", C.c_int, [_VP, _VP, C.POINTER(Buffers), C.POINTER(IO), C.POINTER(RolloutDesc),
                                    C.POINTER(Policy), C.POINTER(Collect)]),
    ("cl_policy_collect_norm", C.c_int, [_VP, _VP, C.POINTER(Buffers), C.POINTER(IO), C.POINTER(RolloutDesc),
                                         C.POINTER(Policy), C.POINTER(Collect), C.POINTER(VecNormUpdate)]),
    ("cl_policy_collect_norm_scratch_bytes", C.c_int, [C.c_int32, C.c_int64, C.POINTER(C.c_int64)]),
    ("cl_derivatives", C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int64]),
    ("cl_stats", C.c_int, [_VP, _VP, C.POINTER(Buffers), _VP, C.c_int]),
    ("cl_get_step_index", C.c_int, [_VP, C.POINTER(C.c_uint64)]),
    ("cl_set_step_index", C.c_int, [_VP, C.c_uint64]),
    ("cl_set_graph_mode", C.c_int, [_VP, C.c_int]),
    ("cl_host_action_staging", C.c_int, [_VP, C.POINTER(_VP)]),
    ("cl_host_set_zero_copy", C.c_int, [_VP, C.c_int]),
    ("cl_host_set_mode", C.c_int, [_VP, C.c_int, C.c_int]),
    ("cl_step_host_async", C.c_int, [_VP, _VP, C.POINTER(Buffers), _VP]),
    ("cl_step_host_wait", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, C.POINTER(C.c_int64)]),
    ("cl_step_host_wait_view", C.c_int, [_VP, _VP, C.POINTER(HostView)]),
    ("cl_reset_host", C.c_int, [_VP, _VP, C.POINTER(Buffers), _VP]),
    ("cl_host_streamed_fallbacks", C.c_int64, [_VP]),
    ("cl_host_h2d_bytes", C.c_int64, [_VP]),
    ("cl_host_d2h_bytes", C.c_int64, [_VP]),
    ("cl_measure_fma_peak", C.c_int, [C.c_int32, C.c_int32, C.c_double, C.POINTER(C.c_double)]),
    ("cl_launch_count", C.c_int64, [_VP]),
    ("cl_block_size", C.c_int, [_VP]),
    ("cl_dyn_launch_count", C.c_int64, [_VP]),
    ("cl_plain_launch_count", C.c_int64, [_VP]),
    ("cl_sm_launch_count", C.c_int64, [_VP]),
    ("cl_gae", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_double, C.c_double, C.c_int32, C.c_int64, C.c_int64, _VP, _VP]),
    ("cl_obs_moments", C.c_int, [_VP, _VP, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _VP, _VP]),
    ("cl_rms_update", C.c_int, [_VP, _VP, C.c_int64, C.c_int32, _VP, _VP, _VP]),
    ("cl_moments_f64", C.c_int, [_VP, _VP, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _VP, _VP]),
    ("cl_obs_normalize", C.c_int, [_VP, _VP, C.c_int64, C.c_int64, _VP, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                   _VP, _VP, C.c_double, C.c_double]),
    ("cl_frame_stack", C.c_int, [_VP, _VP, _VP, C.c_int64, C.c_int64, _VP, C.c_int64, C.c_int32, C.c_int32]),
    ("cl_frame_stack_term", C.c_int, [_VP, _VP, _VP, C.c_int64, C.c_int64, _VP, _VP, C.c_int64, C.c_int64, _VP,
                                      C.c_int64, C.c_int32, C.c_int32]),
    ("cl_eval_metrics", C.c_int, [_VP, _VP, _VP, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int32,
                                  C.c_double, C.c_double, _VP]),
    ("cl_philox4x32_10", None, [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    ("cl_uniform53", C.c_double, [C.c_uint32, C.c_uint32, C.c_double, C.c_double]),
]

_lib = None


def load():
    """Load libchaos_b200.so; raises ChaosLibError (never falls back) if that fails."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ChaosLibError(
            f"{LIB_PATH} is missing: build it with `python -m gym_lorenz_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback.")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise ChaosLibError(f"cannot load {LIB_PATH}: {e}") from e
    for name, res, args in SYMBOLS:
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise ChaosLibError(f"{LIB_PATH} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    v = lib.cl_abi_version()
    if v != CL_ABI_VERSION:
        raise ChaosLibError(f"ABI mismatch: library {v}, binding {CL_ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, ctx=None, what: str = "") -> None:
    if rc != 0:
        msg = load().cl_last_error(ctx)
        raise ChaosLibError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")


def layout(kind: int) -> Layout:
    lay = Layout()
    check(load().cl_env_layout(kind, C.byref(lay)), None, "cl_env_layout")
    return lay
