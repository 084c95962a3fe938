"""Device-resident counterparts of the SB3 pieces that wrap the env step in the reference's
pipelines (SURVEY 8f ranks 1-3).  Everything stays in HBM as torch tensors; the arithmetic is
in csrc/tu_rl_ops.cu.

  gae(...)               SB3 RolloutBuffer.compute_returns_and_advantage   (code/train.py:112-120)
  DeviceVecNormalize     SB3 VecNormalize(norm_obs, norm_reward, clip_obs) (code/lorenz_pmsm/train.py:118,170)
  DeviceVecFrameStack    SB3 VecFrameStack(n_stack)                        (code/lorenz_filter/train.py:115)
  eval_metrics(...)      calculate_advanced_metrics + steady-state MAE/RMSE (code/lorenz_pmsm/test_evaluate.py:25-59,239-250)
  evaluate_policy(...)   the predict loop of those scripts + eval_metrics, one launch (csrc/tu_policy.cu)
  DeviceRolloutCollector SB3 OnPolicyAlgorithm.collect_rollouts without NumPy / host round trips
  FusedRolloutCollector  the same for an SB3 ActorCriticPolicy, the n_steps loop in one launch (csrc/tu_policy.cu)
"""
from __future__ import annotations

import ctypes as C
import os
import zipfile
from io import BytesIO
from typing import Callable, Dict, Optional, Tuple

import torch

from . import _lib as L
from .core import ChaosBatch


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)   # absent in CPU-only builds


def _stream(dev: torch.device):
    """torch's current stream on `dev` as a raw cudaStream_t (see ChaosBatch._stream)."""
    if _RAW_STREAM is not None and dev.index is not None:
        return _RAW_STREAM(dev.index)
    return torch.cuda.current_stream(dev).cuda_stream


def gae(rewards: torch.Tensor, values: torch.Tensor, episode_starts: torch.Tensor, last_values: torch.Tensor,
        last_dones: torch.Tensor, gamma: float, gae_lambda: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """advantages, returns (float32 [T, N]) exactly as SB3 computes them (float32 recurrence)."""
    lib = L.load()
    T, N = rewards.shape
    dev = rewards.device
    args = [x.to(dev, torch.float32).contiguous() for x in (rewards, values, episode_starts)]
    lv = last_values.to(dev, torch.float32).contiguous().view(-1)
    ld = last_dones.to(dev, torch.float32).contiguous().view(-1)
    adv, ret = torch.empty_like(args[0]), torch.empty_like(args[0])
    with torch.cuda.device(dev):
        L.check(lib.cl_gae(_stream(dev), _p(args[0]), _p(args[1]), _p(args[2]), _p(lv), _p(ld), float(gamma),
                           float(gae_lambda), T, N, N, _p(adv), _p(ret)), None, "cl_gae")
    return adv, ret


def eval_metrics(err: torch.Tensor, ctrl: torch.Tensor, dt: float, error_band: float = 0.05,
                 steady_start: Optional[int] = None) -> Dict[str, torch.Tensor]:
    """err f64 [T, n_err, N], ctrl f64 [T, n_ctrl, N] -> per-trajectory mae/rmse/settling_time/energy."""
    lib = L.load()
    T, ne, N = err.shape
    nc = ctrl.shape[1]
    dev = err.device
    err = err.to(dev, torch.float64).contiguous()
    ctrl = ctrl.to(dev, torch.float64).contiguous()
    if steady_start is None:
        steady_start = min(1000, T // 2)          # test_evaluate.py:239
    out = torch.empty((N, 4), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        L.check(lib.cl_eval_metrics(_stream(dev), _p(err), _p(ctrl), T, ne, nc, N, N, int(steady_start), float(dt),
                                    float(error_band), _p(out)), None, "cl_eval_metrics")
    return {"mae": out[:, 0], "rmse": out[:, 1], "settling_time": out[:, 2], "energy": out[:, 3]}


# kinds cl_policy_rollout serves (the reference trains policies on these two) -> control interval (s)
_POLICY_DT = {L.HR_SYNC: 0.001, L.PMSM_SYNC: 0.001}
_SB3_KEYS = ("mlp_extractor.policy_net.0.weight", "mlp_extractor.policy_net.0.bias",
             "mlp_extractor.policy_net.2.weight", "mlp_extractor.policy_net.2.bias",
             "action_net.weight", "action_net.bias")
_RECORDABLE = ("obs", "action", "reward", "done")


def _policy_kind(kind) -> int:
    k = L.KIND_NAMES.get(kind, -1) if isinstance(kind, str) else int(kind)
    if k not in _POLICY_DT:
        raise ValueError(f"policy evaluation supports hr_sync and pmsm_sync only, got {kind!r}")
    return k


_SB3_CRITIC_KEYS = ("mlp_extractor.value_net.0.weight", "mlp_extractor.value_net.0.bias",
                    "mlp_extractor.value_net.2.weight", "mlp_extractor.value_net.2.bias",
                    "value_net.weight", "value_net.bias", "log_std")


def _shapes(k: int, critic: bool):
    """Parameter shapes of the [64, 64] MlpPolicy for kind k, in packing order."""
    lay = L.layout(k)
    obs_dim, act_dim, h = lay.obs_dim, lay.act_dim, L.POLICY_HIDDEN
    actor = [(h, obs_dim), (h,), (h, h), (h,), (act_dim, h), (act_dim,)]
    return actor + ([(h, obs_dim), (h,), (h, h), (h,), (1, h), (1,), (act_dim,)] if critic else [])


def _read_model_zip(src):
    """The policy state dict of an SB3 model zip (its `policy.pth` member, read with zipfile and
    torch.load(weights_only=True): SB3 itself is not needed); any other `src` is returned as is."""
    if isinstance(src, (str, os.PathLike)):
        with zipfile.ZipFile(src) as z:
            if "policy.pth" not in z.namelist():
                raise ValueError(f"{src}: no policy.pth member (not an SB3 model zip)")
            return torch.load(BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
    return src


def _sb3_tensors(sd, keys):
    """The tensors of `keys` from an SB3 policy state dict, refusing missing keys and deeper nets."""
    missing = [key for key in keys if key not in sd]
    if missing:
        raise ValueError(f"not an SB3 MlpPolicy state dict: missing {missing}")
    for net in ("policy_net", "value_net"):
        prefix = f"mlp_extractor.{net}."
        if any(key.startswith(prefix) for key in keys):
            extra = sorted(key for key in sd if key.startswith(prefix) and key not in keys)
            if extra:
                raise ValueError(f"{net} is not [64, 64]: unexpected {extra}")
    return [sd[key] for key in keys]


def _check_shapes(keys, tensors, shapes) -> None:
    for key, t, shape in zip(keys, tensors, shapes):
        if t is None or tuple(t.shape) != shape:
            got = None if t is None else tuple(t.shape)
            raise ValueError(f"{key}: expected shape {shape}, got {got}")


def pack_policy(src, device, kind="hr_sync") -> torch.Tensor:
    """The float32 parameter block `cl_policy_rollout` reads, in torch Linear layout:
    W1[64][obs_dim] b1[64] W2[64][64] b2[64] W3[act_dim][64] b3[act_dim].

    `src` is one of
      * a stable-baselines3 `ActorCriticPolicy` state dict (`mlp_extractor.policy_net.{0,2}.{weight,bias}`,
        `action_net.{weight,bias}`; the value head and `log_std` are ignored);
      * the path of an SB3 model zip: its `policy.pth` member is read with `zipfile` and
        `torch.load(weights_only=True)`, SB3 itself is not needed.  The key names follow SB3 2.7.1's
        source; they have not been checked against the reference's own saved models;
      * a `(policy_net, action_net)` pair of torch modules: Linear-Tanh-Linear-Tanh and a Linear.

    Every shape is checked against `kind`'s observation / action dimensions and the [64, 64] MlpPolicy
    architecture; a mismatch raises ValueError before anything reaches the device.
    """
    k = _policy_kind(kind)
    src = _read_model_zip(src)
    if isinstance(src, (tuple, list)):
        if len(src) != 2 or not all(isinstance(m, torch.nn.Module) for m in src):
            raise ValueError("expected a (policy_net, action_net) pair of torch modules")
        pnet, anet = src
        leaves = [m for m in pnet.modules() if len(list(m.children())) == 0]
        if [type(m) for m in leaves] != [torch.nn.Linear, torch.nn.Tanh, torch.nn.Linear, torch.nn.Tanh] or \
                not isinstance(anet, torch.nn.Linear):
            raise ValueError("policy_net must be Linear-Tanh-Linear-Tanh and action_net a Linear "
                             "(SB3 MlpPolicy, pi=[64, 64], activation_fn=Tanh)")
        tensors = [leaves[0].weight, leaves[0].bias, leaves[2].weight, leaves[2].bias, anet.weight, anet.bias]
    elif isinstance(src, dict):
        tensors = _sb3_tensors(src, _SB3_KEYS)
    else:
        raise ValueError(f"cannot pack a policy from {type(src).__name__}")
    _check_shapes(_SB3_KEYS, tensors, _shapes(k, critic=False))
    with torch.no_grad():
        return torch.cat([t.detach().reshape(-1).to(torch.float32).cpu() for t in tensors]).to(device)


def _n_params(obs_dim: int, act_dim: int, critic: bool) -> int:
    h = L.POLICY_HIDDEN
    n = h * (obs_dim + 1 + h + 1 + act_dim) + act_dim
    return n + (h * (obs_dim + 1 + h + 1 + 1) + 1 + act_dim if critic else 0)


def pack_actor_critic(src, device, kind="hr_sync", out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The float32 parameter block `cl_policy_collect` reads: `pack_policy`'s actor block first, then
    V1[64][obs_dim] c1[64] V2[64][64] c2[64] Wv[1][64] bv[1] (SB3's `mlp_extractor.value_net` and
    `value_net`), then log_std[act_dim].  `block[:n_actor]` is a valid `evaluate_policy` block.

    `src` is an SB3 `ActorCriticPolicy` state dict (`pack_policy`'s keys plus
    `mlp_extractor.value_net.{0,2}.{weight,bias}`, `value_net.{weight,bias}` and `log_std`), the path of
    an SB3 model zip, or any torch.nn.Module whose `state_dict()` carries those names.  Shapes are
    checked as in `pack_policy`.  With `out` (a contiguous f32 tensor of the block's size) the block is
    written in place by device-side copies: no host synchronisation, so a training loop can refresh it
    after every optimiser step and a captured CUDA graph keeps reading the same storage.
    """
    k = _policy_kind(kind)
    src = _read_model_zip(src)
    if isinstance(src, torch.nn.Module):
        src = src.state_dict()
    if not isinstance(src, dict):
        raise ValueError(f"cannot pack an actor-critic from {type(src).__name__}")
    keys = _SB3_KEYS + _SB3_CRITIC_KEYS
    tensors = _sb3_tensors(src, keys)
    _check_shapes(keys, tensors, _shapes(k, critic=True))
    if out is None:
        with torch.no_grad():
            return torch.cat([t.detach().reshape(-1).to(torch.float32).cpu() for t in tensors]).to(device)
    n = sum(t.numel() for t in tensors)
    if not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or out.numel() != n or \
            not out.is_contiguous():
        raise ValueError(f"out must be a contiguous f32 tensor of {n} values")
    with torch.no_grad():
        o = 0
        for t in tensors:
            out[o:o + t.numel()].view(t.shape).copy_(t.detach(), non_blocking=True)
            o += t.numel()
    return out


def evaluate_policy(env, policy, T: int, *, normalize=None, dt: Optional[float] = None, error_band: float = 0.05,
                    steady_start: Optional[int] = None, record=(), obs0: Optional[torch.Tensor] = None
                    ) -> Dict[str, torch.Tensor]:
    """Roll a trained policy deterministically for T control intervals in ONE launch and return the
    evaluation metrics of `eval_metrics` without storing the trajectories: the reference's
    `model.predict(obs, deterministic=True)` loops (code/test_evaluate.py, code/lorenz_pmsm/test_evaluate.py).

    env: a BatchedChaosVecEnv (or device wrapper around one) or a ChaosBatch of kind hr_sync / pmsm_sync.
    policy: what `pack_policy` accepts, or its packed tensor.  normalize: a DeviceVecNormalize whose
    `obs_rms`, `epsilon` and `clip_obs` are used frozen, or None.  dt defaults to the control interval,
    steady_start to min(1000, T // 2).  obs0 (f32 [N, obs_dim]) is the observation interval 0 acts on;
    by default the batch's observation planes, which hold it after `reset()` / `step()` -- after
    `set_attr(...)` or `rollout()` pass it explicitly.  The last observation is written back to the
    observation planes, so a following `step()` or `evaluate_policy` continues from there.

    Returns {"mae", "rmse", "settling_time", "energy"} (f64 [N] device tensors) plus the streams named in
    `record`: "obs" f32 [T, obs_dim, n_pad], "reward" [T, n_pad], "done" u8 [T, n_pad] (as `rollout`) and
    "action" f32 [T, N, act_dim] (the clipped actions applied).

    For an evaluation like the reference's use a ChaosBatch(autoreset=False) with max_episode_steps >= T:
    with auto-reset on, the window contains the reset observations, as the recorded streams show.
    The metrics are in observation units.  For hr_sync the error components are err / 50 (the env's
    scale_factor): for state units pass error_band=0.05 / 50 and multiply MAE / RMSE by 50.
    """
    b = env if isinstance(env, ChaosBatch) else base_batch(env)
    kind = _policy_kind(b.kind)
    if b.obs_f64:
        raise ValueError("evaluate_policy needs float32 observations (obs_f64=False)")
    T = int(T)
    if T < 1:
        raise ValueError("T must be >= 1")
    if steady_start is None:
        steady_start = min(1000, T // 2)          # test_evaluate.py:239, as eval_metrics
    if not 0 <= int(steady_start) < T:
        raise ValueError(f"steady_start must lie in [0, {T}), got {steady_start}")
    unknown = [r for r in record if r not in _RECORDABLE]
    if unknown:
        raise ValueError(f"record: unknown streams {unknown}; choose from {_RECORDABLE}")
    params = policy if isinstance(policy, torch.Tensor) else pack_policy(policy, b.device, kind)
    npar = _n_params(b.obs_dim, b.act_dim, critic=False)
    if params.dtype != torch.float32 or params.device != b.device or params.numel() != npar or \
            not params.is_contiguous():
        raise ValueError(f"packed policy must be a contiguous f32 tensor of {npar} values on {b.device}")
    dev, N, NP = b.device, b.num_envs, b.n_pad
    planes = b._view(b.obs_planes)
    if obs0 is not None:
        if not isinstance(obs0, torch.Tensor) or obs0.dtype != torch.float32 or obs0.device != dev or \
                tuple(obs0.shape) != (N, b.obs_dim):
            raise ValueError(f"obs0 must be f32 [{N}, {b.obs_dim}] on {dev}")
        planes.copy_(obs0)
    out = {}
    io = L.IO()
    desc = L.RolloutDesc(T=T)
    if "obs" in record:
        out["obs"] = torch.empty((T, b.obs_dim, NP), dtype=torch.float32, device=dev)
        io.obs, io.obs_es, io.obs_cs, desc.obs_ts = _p(out["obs"]), 1, NP, b.obs_dim * NP
    if "reward" in record:
        out["reward"] = torch.empty((T, NP), dtype=b.real, device=dev)
        io.reward, desc.rew_ts = _p(out["reward"]), NP
    if "done" in record:
        out["done"] = torch.empty((T, NP), dtype=torch.uint8, device=dev)
        io.done, desc.done_ts = _p(out["done"]), NP
    if "action" in record:
        out["action"] = torch.empty((T, N, b.act_dim), dtype=torch.float32, device=dev)
    io.last_ep_ret, io.last_ep_len = _p(b.last_ep_ret), _p(b.last_ep_len)
    metrics = torch.empty((N, 4), dtype=torch.float64, device=dev)
    pol = L.Policy(params=_p(params), obs0=_p(b.obs_planes), obs0_es=1, obs0_cs=NP, obs_last=_p(b.obs_planes),
                   act_out=_p(out.get("action")), metrics=_p(metrics), steady_start=int(steady_start),
                   dt=float(_POLICY_DT[kind] if dt is None else dt), error_band=float(error_band))
    if normalize is not None and normalize.norm_obs:
        pol.obs_mean, pol.obs_var = _p(normalize.obs_rms.mean), _p(normalize.obs_rms.var)
        pol.epsilon, pol.clip_obs = float(normalize.epsilon), float(normalize.clip_obs)
    L.check(b.lib.cl_policy_rollout(b.ctx, b._stream(), C.byref(b._bufs), C.byref(io), C.byref(desc), C.byref(pol)),
            b.ctx, "cl_policy_rollout")
    b._keep_policy = (params, metrics, out)
    out.update(mae=metrics[:, 0], rmse=metrics[:, 1], settling_time=metrics[:, 2], energy=metrics[:, 3])
    return out


def base_batch(env):
    """The ChaosBatch under any stack of device wrappers (walks `.venv` until `.batch` is found)."""
    e = env
    while not hasattr(e, "batch"):
        if not hasattr(e, "venv"):
            raise AttributeError(f"{type(env).__name__} wraps no BatchedChaosVecEnv")
        e = e.venv
    return e.batch


class RunningMeanStd:
    """SB3 RunningMeanStd (float64 mean/var/count, Chan et al. parallel update).  Batch moments and
    the merge both run on the device and update `mean` / `var` / `count_t` in place: no host
    synchronisation, and an `update` can be captured in a CUDA graph and replayed."""

    def __init__(self, shape, device, epsilon: float = 1e-4):
        self.mean = torch.zeros(shape, dtype=torch.float64, device=device)
        self.var = torch.ones(shape, dtype=torch.float64, device=device)
        self.count_t = torch.full((1,), float(epsilon), dtype=torch.float64, device=device)
        self._acc = torch.zeros((2,) + tuple(shape), dtype=torch.float64, device=device)

    @property
    def count(self) -> float:
        """Host copy of the running count (synchronises; for inspection / checkpoints)."""
        return float(self.count_t.item())

    @count.setter
    def count(self, v: float) -> None:
        self.count_t.fill_(float(v))

    def update(self, x: torch.Tensor) -> None:
        """x: f32 or f64 [N, dim] (any strides)."""
        lib = L.load()
        n, dim = x.shape
        dev = x.device
        if x.dtype not in (torch.float32, torch.float64):
            raise ValueError("RunningMeanStd.update expects float32 or float64")
        with torch.cuda.device(dev):
            st = _stream(dev)
            fn, name = (lib.cl_obs_moments, "cl_obs_moments") if x.dtype == torch.float32 else \
                (lib.cl_moments_f64, "cl_moments_f64")
            L.check(fn(st, _p(x), x.stride(0), x.stride(1), n, dim, _p(self.mean), _p(self._acc)), None, name)
            L.check(lib.cl_rms_update(st, _p(self._acc), n, dim, _p(self.mean), _p(self.var), _p(self.count_t)),
                    None, "cl_rms_update")


class DeviceVecNormalize:
    """VecNormalize on device tensors: `reset_tensor()` / `step_tensor(actions)` of the wrapped
    env, observations normalised with running statistics (updated while `training`), rewards
    optionally normalised by the running std of the discounted return."""

    def __init__(self, venv, training: bool = True, norm_obs: bool = True, norm_reward: bool = True,
                 clip_obs: float = 10.0, clip_reward: float = 10.0, gamma: float = 0.99, epsilon: float = 1e-8):
        self.venv, self.training = venv, training
        self.norm_obs, self.norm_reward = norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.num_envs = venv.num_envs
        b = base_batch(venv)
        self.device = b.device
        self.obs_rms = RunningMeanStd((b.obs_dim,), self.device)
        self.ret_rms = RunningMeanStd((1,), self.device)
        self.returns = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)
        self._out = torch.empty((self.num_envs, b.obs_dim), dtype=torch.float32, device=self.device)
        self._term = torch.empty_like(self._out)
        self.old_obs = None
        self.old_reward = None

    def normalize_obs(self, obs: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if not self.norm_obs:
            return obs
        lib = L.load()
        out = torch.empty(obs.shape, dtype=torch.float32, device=obs.device) if out is None else out
        n, dim = obs.shape
        with torch.cuda.device(obs.device):
            L.check(lib.cl_obs_normalize(_stream(obs.device), _p(obs), obs.stride(0), obs.stride(1), _p(out),
                                         out.stride(0), out.stride(1), n, dim, _p(self.obs_rms.mean),
                                         _p(self.obs_rms.var), float(self.epsilon), float(self.clip_obs)),
                    None, "cl_obs_normalize")
        return out

    def normalize_reward(self, reward: torch.Tensor) -> torch.Tensor:
        if not self.norm_reward:
            return reward
        r = reward.double() / torch.sqrt(self.ret_rms.var[0] + self.epsilon)
        return torch.clamp(r, -self.clip_reward, self.clip_reward).float()

    def reset_tensor(self) -> torch.Tensor:
        obs = self.venv.reset_tensor()
        self.old_obs = obs
        self.returns.zero_()
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs, self._out)

    def step_tensor(self, actions: torch.Tensor):
        obs, rew, done = self.venv.step_tensor(actions)
        self.old_obs, self.old_reward = obs, rew
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        nobs = self.normalize_obs(obs, self._out)
        if self.training:
            # SB3 VecNormalize.step_wait -> _update_reward: whenever `training`, float64 returns
            self.returns.mul_(self.gamma).add_(rew)      # in place: replayable as a captured graph
            self.ret_rms.update(self.returns.view(-1, 1))
        nrew = self.normalize_reward(rew)
        self.returns.masked_fill_(done != 0, 0.0)
        return nobs, nrew, done

    def terminal_obs(self) -> torch.Tensor:
        inner = self.venv.terminal_obs() if hasattr(self.venv, "terminal_obs") else base_batch(self.venv).terminal_obs()
        return self.normalize_obs(inner, self._term)

    def get_original_obs(self) -> torch.Tensor:
        return self.old_obs

    def state_dict(self):
        return {"obs_mean": self.obs_rms.mean.clone(), "obs_var": self.obs_rms.var.clone(),
                "obs_count": self.obs_rms.count, "ret_mean": self.ret_rms.mean.clone(),
                "ret_var": self.ret_rms.var.clone(), "ret_count": self.ret_rms.count}

    def load_state_dict(self, sd):
        for rms, k in ((self.obs_rms, "obs"), (self.ret_rms, "ret")):   # in place: captured graphs keep pointing here
            rms.mean.copy_(sd[k + "_mean"]); rms.var.copy_(sd[k + "_var"]); rms.count = sd[k + "_count"]


class DeviceVecFrameStack:
    """VecFrameStack(n_stack) for 1-D observations, stacked along the last axis, on device.
    Wraps a BatchedChaosVecEnv or a DeviceVecNormalize (code/lorenz_filter/train.py:109-115)."""

    def __init__(self, venv, n_stack: int):
        self.venv, self.n_stack = venv, int(n_stack)
        self.num_envs = venv.num_envs
        src = base_batch(venv)
        self.dim = src.obs_dim
        self.device = src.device
        self.stacked = torch.zeros((self.num_envs, self.dim * self.n_stack), dtype=torch.float32, device=self.device)
        self._term = torch.zeros_like(self.stacked)

    def _inner_terminal_obs(self) -> torch.Tensor:
        return self.venv.terminal_obs() if hasattr(self.venv, "terminal_obs") else base_batch(self.venv).terminal_obs()

    def _push(self, obs: torch.Tensor, done: Optional[torch.Tensor], term: Optional[torch.Tensor] = None) -> torch.Tensor:
        lib = L.load()
        with torch.cuda.device(self.device):
            if term is None or done is None:
                L.check(lib.cl_frame_stack(_stream(self.device), _p(self.stacked), _p(obs), obs.stride(0), obs.stride(1),
                                           _p(done), self.num_envs, self.dim, self.n_stack), None, "cl_frame_stack")
            else:
                L.check(lib.cl_frame_stack_term(_stream(self.device), _p(self.stacked), _p(obs), obs.stride(0),
                                                obs.stride(1), _p(done), _p(term), term.stride(0), term.stride(1),
                                                _p(self._term), self.num_envs, self.dim, self.n_stack), None,
                        "cl_frame_stack_term")
        return self.stacked

    def reset_tensor(self) -> torch.Tensor:
        obs = self.venv.reset_tensor()
        self.stacked.zero_()
        return self._push(obs, None)

    def step_tensor(self, actions: torch.Tensor):
        obs, rew, done = self.venv.step_tensor(actions)
        return self._push(obs, done, self._inner_terminal_obs()), rew, done

    def terminal_obs(self) -> torch.Tensor:
        """[N, dim * n_stack]: for envs that finished an episode in the last step, the stacked terminal
        observation of SB3's StackedObservations.update (previous stack rolled by one frame + the inner
        env's -- normalised, if wrapped -- terminal observation).  Other rows are undefined."""
        return self._term


class DeviceRolloutCollector:
    """SB3 `OnPolicyAlgorithm.collect_rollouts` on device tensors: policy forward -> env step ->
    buffer write, then GAE, with no NumPy and no host round trip inside the loop.

    `policy(obs) -> (actions, values, log_probs)` is any torch callable (the learner's network);
    time-limit truncations bootstrap with the value of the terminal observation like SB3
    (`rewards[idx] += gamma * V(terminal_obs)`).

    `use_cuda_graph=True` captures the whole n_steps loop (policy kernels, env step kernels,
    buffer writes, GAE) into ONE CUDA graph and replays it per rollout: at a few thousand envs the
    loop is launch-latency bound (~30 small kernels per step), which is exactly what graphs remove.
    The env is switched to graph mode (device-resident Philox step index), so replays keep
    advancing the random streams.
    """

    def __init__(self, env, policy: Callable, n_steps: int, gamma: float = 0.99, gae_lambda: float = 0.95,
                 use_cuda_graph: bool = False):
        self.env, self.policy, self.n_steps = env, policy, int(n_steps)
        self.gamma, self.gae_lambda = gamma, gae_lambda
        b = base_batch(env)
        self.batch, dev, N, T = b, b.device, b.num_envs, self.n_steps
        self.obs_dim = env.stacked.shape[1] if hasattr(env, "stacked") else b.obs_dim
        self.buf = {
            "obs": torch.empty((T, N, self.obs_dim), dtype=torch.float32, device=dev),
            "actions": torch.empty((T, N, b.act_dim), dtype=torch.float32, device=dev),
            "rewards": torch.empty((T, N), dtype=torch.float32, device=dev),
            "values": torch.empty((T, N), dtype=torch.float32, device=dev),
            "log_probs": torch.empty((T, N), dtype=torch.float32, device=dev),
            "episode_starts": torch.empty((T, N), dtype=torch.float32, device=dev),
        }
        self._last_obs = None
        self._last_starts = torch.ones(N, dtype=torch.float32, device=dev)
        self._lo = float(b.layout.act_low)
        self._hi = float(b.layout.act_high)
        self.use_cuda_graph = bool(use_cuda_graph)
        self._graph = None
        self._graph_out = None
        self._warm = False

    def _terminal_obs(self):
        return self.env.terminal_obs() if hasattr(self.env, "terminal_obs") else self.batch.terminal_obs()

    def _loop(self, sync_free: bool) -> Dict[str, torch.Tensor]:
        buf = self.buf
        for t in range(self.n_steps):
            obs = self._last_obs
            actions, values, log_probs = self.policy(obs)
            buf["obs"][t].copy_(obs)
            buf["actions"][t].copy_(actions)
            buf["values"][t].copy_(values.view(-1))
            buf["log_probs"][t].copy_(log_probs.view(-1))
            buf["episode_starts"][t].copy_(self._last_starts)
            new_obs, rew, done = self.env.step_tensor(torch.clamp(actions, self._lo, self._hi))
            rew = rew.float().clone()
            trunc = (done & L.DONE_TRUNCATED).bool() & ~(done & L.DONE_TERMINATED).bool()
            if sync_free or bool(trunc.any()):   # TimeLimit bootstrap (SB3 collect_rollouts)
                _, tv, _ = self.policy(self._terminal_obs())
                rew = torch.where(trunc, rew + self.gamma * tv.view(-1), rew)
            buf["rewards"][t].copy_(rew)
            self._last_starts.copy_((done != 0).float())
            self._last_obs.copy_(new_obs)
        _, last_values, _ = self.policy(self._last_obs)
        adv, ret = gae(buf["rewards"], buf["values"], buf["episode_starts"], last_values.view(-1), self._last_starts,
                       self.gamma, self.gae_lambda)
        out = dict(buf)
        out["advantages"], out["returns"] = adv, ret
        return out

    @torch.no_grad()
    def collect(self) -> Dict[str, torch.Tensor]:
        if self._last_obs is None:
            self._last_obs = self.env.reset_tensor().clone()
        if not self.use_cuda_graph:
            return self._loop(sync_free=False)
        if self._graph is None:
            dev = self.batch.device
            if not self._warm:
                # first rollout: eager, sync-free -- it is a real rollout AND the warm-up that
                # CUDA-graph capture needs (lazy initialisation, allocator, occupancy queries)
                self.batch.set_graph_mode(True)
                self._warm = True
                return self._loop(sync_free=True)
            torch.cuda.synchronize(dev)
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):            # capture executes nothing
                self._graph_out = self._loop(sync_free=True)
        self._graph.replay()
        return self._graph_out


class FusedRolloutCollector:
    """SB3 `OnPolicyAlgorithm.collect_rollouts` for an `ActorCriticPolicy` (pi = vf = [64, 64], Tanh,
    Gaussian actions with a state-independent log_std) in ONE launch per rollout (`cl_policy_collect`):
    per control interval the kernel normalises the observation, runs actor and critic, samples the action
    from the env's Philox stream (purpose TAG_POLICY), steps the env with the clipped action, bootstraps
    TimeLimit truncations with the critic on the terminal observation and writes one buffer row.  GAE is
    `rl_ops.gae` on the result.

    env: a BatchedChaosVecEnv (or device wrapper around one) or a ChaosBatch of kind hr_sync / pmsm_sync.
    policy: a torch.nn.Module with SB3's parameter names, an SB3 state dict or model zip (see
    `pack_actor_critic`), or an already packed block.  normalize: a DeviceVecNormalize used frozen (its
    `obs_rms`, `epsilon`, `clip_obs`); one in training mode or with `norm_reward` is refused unless
    `update_normalize=True`.

    update_normalize=True (`cl_policy_collect_norm`): `normalize` is a DeviceVecNormalize in training mode
    over this batch, with `norm_obs` / `norm_reward` in any combination, and the kernel does what SB3's
    VecNormalize.step_wait does every step: obs_rms.update on the raw observations, the discounted
    `returns` (the normaliser's `gamma`) and ret_rms.update, reward normalisation with the updated
    ret_rms, observations normalised with the updated obs_rms.  `vn.obs_rms`, `vn.ret_rms` and
    `vn.returns` are updated in place on the device, so a training loop can switch between this collector
    and `DeviceRolloutCollector` or checkpoint `vn.state_dict()` with continuous statistics.  The first
    `collect()` starts with `vn.reset_tensor()` (SB3's reset in training mode: obs_rms sees the reset
    observation, returns are zeroed); `vn.old_obs` is the raw last observation.  The statistics cover the
    envs of this collector, i.e. one GPU; each interval's batch statistics are summed in a fixed order, so
    they are bit-reproducible run to run.

    `collect()` returns the dict of `DeviceRolloutCollector.collect()` (same keys, shapes, dtypes).  The
    first call resets the env and starts every episode; later calls continue from the batch's observation
    planes and the carried `starts`.  `last_values` holds V of the last observation.  `collect()` never
    synchronises with the host: with the env in graph mode it can be captured in a CUDA graph.
    `sync_params()` repacks the module's current weights into the same storage (capturable as well).
    """

    def __init__(self, env, policy, n_steps: int, gamma: float = 0.99, gae_lambda: float = 0.95,
                 normalize=None, update_normalize: bool = False):
        b = env if isinstance(env, ChaosBatch) else base_batch(env)
        kind = _policy_kind(b.kind)
        if b.obs_f64:
            raise ValueError("FusedRolloutCollector needs float32 observations (obs_f64=False)")
        if int(n_steps) < 1:
            raise ValueError("n_steps must be >= 1")
        self.update_normalize = bool(update_normalize)
        if self.update_normalize:
            if normalize is None:
                raise ValueError("update_normalize=True needs a DeviceVecNormalize (normalize=...)")
            if not normalize.training:
                raise ValueError("update_normalize=True needs a normaliser in training mode (training=True)")
            if base_batch(normalize) is not b or normalize.num_envs != b.num_envs:
                raise ValueError("update_normalize=True needs a normaliser over this collector's batch")
        else:
            if normalize is not None and normalize.training:
                raise ValueError("normalize must be frozen (training=False); DeviceRolloutCollector updates the "
                                 "statistics every step, or pass update_normalize=True")
            if normalize is not None and normalize.norm_reward:
                raise ValueError("reward normalisation is not fused (norm_reward=False); use DeviceRolloutCollector "
                                 "or update_normalize=True")
        self.env, self.policy, self.n_steps = env, policy, int(n_steps)
        self.gamma, self.gae_lambda, self.normalize = gamma, gae_lambda, normalize
        self.batch, self.kind = b, kind
        dev, N, T = b.device, b.num_envs, self.n_steps
        npar = _n_params(b.obs_dim, b.act_dim, critic=True)
        self.n_actor = _n_params(b.obs_dim, b.act_dim, critic=False)
        self.params = policy if isinstance(policy, torch.Tensor) else pack_actor_critic(policy, dev, kind)
        if self.params.dtype != torch.float32 or self.params.device != dev or self.params.numel() != npar or \
                not self.params.is_contiguous():
            raise ValueError(f"packed actor-critic must be a contiguous f32 tensor of {npar} values on {dev}")
        f32 = dict(dtype=torch.float32, device=dev)
        self.buf = {
            "obs": torch.empty((T, N, b.obs_dim), **f32),
            "actions": torch.empty((T, N, b.act_dim), **f32),
            "rewards": torch.empty((T, N), **f32),
            "values": torch.empty((T, N), **f32),
            "log_probs": torch.empty((T, N), **f32),
            "episode_starts": torch.empty((T, N), **f32),
        }
        self.last_values = torch.empty(N, **f32)
        self.starts = torch.ones(N, **f32)
        self._started = False
        self._io = L.IO(last_ep_ret=_p(b.last_ep_ret), last_ep_len=_p(b.last_ep_len))
        self._desc = L.RolloutDesc(T=T)
        self._pol = L.Policy(params=_p(self.params), obs0=_p(b.obs_planes), obs0_es=1, obs0_cs=b.n_pad,
                             obs_last=_p(b.obs_planes))
        if normalize is not None and normalize.norm_obs and not self.update_normalize:
            self._pol.obs_mean, self._pol.obs_var = _p(normalize.obs_rms.mean), _p(normalize.obs_rms.var)
            self._pol.epsilon, self._pol.clip_obs = float(normalize.epsilon), float(normalize.clip_obs)
        buf = self.buf
        self._col = L.Collect(gamma=float(gamma), starts=_p(self.starts), obs=_p(buf["obs"]),
                              actions=_p(buf["actions"]), rewards=_p(buf["rewards"]), values=_p(buf["values"]),
                              log_probs=_p(buf["log_probs"]), episode_starts=_p(buf["episode_starts"]),
                              last_values=_p(self.last_values))
        self._vn = None
        if self.update_normalize:
            vn = normalize
            nb = C.c_int64()
            L.check(b.lib.cl_policy_collect_norm_scratch_bytes(kind, N, C.byref(nb)), None,
                    "cl_policy_collect_norm_scratch_bytes")
            self._scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
            self._vn = L.VecNormUpdate(
                obs_mean=_p(vn.obs_rms.mean), obs_var=_p(vn.obs_rms.var), obs_count=_p(vn.obs_rms.count_t),
                ret_mean=_p(vn.ret_rms.mean), ret_var=_p(vn.ret_rms.var), ret_count=_p(vn.ret_rms.count_t),
                returns=_p(vn.returns), gamma=float(vn.gamma), epsilon=float(vn.epsilon),
                clip_obs=float(vn.clip_obs), clip_reward=float(vn.clip_reward), norm_obs=int(bool(vn.norm_obs)),
                norm_reward=int(bool(vn.norm_reward)), scratch=_p(self._scratch), scratch_bytes=nb.value)

    def sync_params(self) -> None:
        """Repack the policy module's current weights into `self.params` (device copies only)."""
        if isinstance(self.policy, torch.Tensor):
            raise ValueError("the collector was given a packed block: there is no module to repack from")
        pack_actor_critic(self.policy, self.batch.device, self.kind, out=self.params)

    @torch.no_grad()
    def collect(self) -> Dict[str, torch.Tensor]:
        b = self.batch
        if not self._started:
            if self._vn is not None:
                self.normalize.reset_tensor()
            else:
                b.reset()
            self.starts.fill_(1.0)
            self._started = True
        if self._vn is not None:
            L.check(b.lib.cl_policy_collect_norm(b.ctx, b._stream(), C.byref(b._bufs), C.byref(self._io),
                                                 C.byref(self._desc), C.byref(self._pol), C.byref(self._col),
                                                 C.byref(self._vn)), b.ctx, "cl_policy_collect_norm")
            self.normalize.old_obs = b._view(b.obs_planes)
        else:
            L.check(b.lib.cl_policy_collect(b.ctx, b._stream(), C.byref(b._bufs), C.byref(self._io),
                                            C.byref(self._desc), C.byref(self._pol), C.byref(self._col)),
                    b.ctx, "cl_policy_collect")
        buf = self.buf
        adv, ret = gae(buf["rewards"], buf["values"], buf["episode_starts"], self.last_values, self.starts,
                       self.gamma, self.gae_lambda)
        out = dict(buf)
        out["advantages"], out["returns"] = adv, ret
        return out
