"""cl_policy_collect_norm on the B200: the fused PPO / A2C collector behind a VecNormalize in training mode
replays through DeviceRolloutCollector(DeviceVecNormalize(training=True)) from the same snapshot and the same
start statistics, its raw io streams fed to the SB3 VecNormalize restatement reproduce its buffer and
statistics, and windows are bit-reproducible, chain, replay as a CUDA graph and take new weights."""
import json
import os

import numpy as np
import pytest
import torch

from test_gpu_policy_collect import (KEYS, SEED, _actor, _assert_same_final, _assert_stats_close, _critic, _policy,
                                     _Replay, _restore, _snapshot, _venv)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VN_KEYS = ("obs_mean", "obs_var", "obs_count", "ret_mean", "ret_var", "ret_count", "returns")


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _vn_tensors(vn):
    return dict(zip(VN_KEYS, (vn.obs_rms.mean, vn.obs_rms.var, vn.obs_rms.count_t, vn.ret_rms.mean,
                              vn.ret_rms.var, vn.ret_rms.count_t, vn.returns)))


def _vn_snap(vn):
    return {k: v.clone() for k, v in _vn_tensors(vn).items()}


def _vn_restore(vn, snap):
    for k, v in _vn_tensors(vn).items():
        v.copy_(snap[k])


def _normalizer(venv, kind, norm_obs=True, norm_reward=False):
    """DeviceVecNormalize in training mode; pmsm_sync starts from the statistics of the SB3 artefacts."""
    from gym_lorenz_b200.rl_ops import DeviceVecNormalize
    art = json.load(open(os.path.join(ROOT, "tests", "golden", "sb3_artefacts.json")))["runs"]["0.50"]
    vn = DeviceVecNormalize(venv, training=True, norm_obs=norm_obs, norm_reward=norm_reward,
                            clip_obs=art["clip_obs"], clip_reward=art["clip_reward"], gamma=art["gamma"],
                            epsilon=art["epsilon"])
    if kind == "pmsm_sync":
        vn.obs_rms.mean.copy_(torch.tensor(art["obs_mean"], dtype=torch.float64))
        vn.obs_rms.var.copy_(torch.tensor(art["obs_var"], dtype=torch.float64))
        vn.obs_rms.count = float.fromhex(art["obs_count"])
        vn.ret_rms.mean.fill_(art["ret_mean"])
        vn.ret_rms.var.fill_(art["ret_var"])
        vn.ret_rms.count = float.fromhex(art["ret_count"])
    return vn


def _collector(kind, n, T, max_steps=9, norm_obs=True, norm_reward=False, seed=11):
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector
    venv = _venv(kind, n, max_steps)
    vn = _normalizer(venv, kind, norm_obs, norm_reward)
    m = _policy(seed)
    return venv, vn, m, FusedRolloutCollector(vn, m, T, normalize=vn, update_normalize=True)


def _ulps(a, b):
    """|a - b| in units of the float32 spacing at b."""
    spacing = torch.nextafter(b.abs(), torch.full_like(b, float("inf"))) - b.abs()
    return ((a - b).abs() / spacing).max().item()


def _assert_vn_close(got, want):
    for k in ("obs_count", "ret_count", "returns"):                 # per-env arithmetic / one addition per step
        assert torch.equal(got[k], want[k]), k
    for rms in ("obs", "ret"):                                     # the reductions differ in summation order
        sd = want[rms + "_var"].sqrt()
        assert bool(((got[rms + "_mean"] - want[rms + "_mean"]).abs() <= 1e-12 * sd).all()), rms
        assert bool(((got[rms + "_var"] - want[rms + "_var"]).abs() <= 1e-12 * want[rms + "_var"]).all()), rms


# (kind, n, T, norm_obs, norm_reward); pmsm_sync starts from the artefact statistics
CASES = [("hr_sync", 33, 64, True, False), ("pmsm_sync", 33, 64, True, False),
         ("hr_sync", 1000, 64, True, False), ("pmsm_sync", 1000, 64, True, False),
         ("hr_sync", 65536, 64, True, False), ("pmsm_sync", 65536, 64, True, False),
         ("hr_sync", 1000, 1, True, False), ("pmsm_sync", 65536, 1, True, False),
         ("hr_sync", 1000, 64, True, True), ("pmsm_sync", 1000, 64, False, False),
         ("hr_sync", 262144, 16, True, False), ("pmsm_sync", 262144, 16, True, True)]


@pytest.mark.parametrize("kind,n,T,norm_obs,norm_reward", CASES)
def test_replay_through_device_vecnormalize(kind, n, T, norm_obs, norm_reward):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import DeviceRolloutCollector
    if n > 100_000:
        # 128 registers per thread: at most 512 threads per SM are co-resident, so threads own several envs
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        assert n >= 2 * 512 * sms
    venv, vn, m, fused = _collector(kind, n, T, norm_obs=norm_obs, norm_reward=norm_reward)
    b = venv.batch
    for _ in range(max(1, 12 // T)):
        fused.collect()              # episodes running, some truncated already; statistics moved
    if kind == "hr_sync":
        # error m0 - s0 beyond the env's +-70 bound on every 7th env: they terminate in the window's first step
        b.state[0, 3:n:7] = b.state[3, 3:n:7] + 75.0
    start, vstart = _snapshot(b, fused), _vn_snap(vn)
    got = {k: v.clone() for k, v in fused.collect().items()}
    end, vend = _snapshot(b, fused), _vn_snap(vn)
    assert torch.equal(vn.get_original_obs(), end["obs"])
    _restore(b, fused, start)
    _vn_restore(vn, vstart)
    replay = _Replay(m, got["actions"])
    ref = DeviceRolloutCollector(vn, replay, T, gamma=fused.gamma)
    replay.col = ref
    ref._last_obs = vn.normalize_obs(start["obs"]).clone()
    ref._last_starts.copy_(start["starts"])
    want = ref.collect()
    replayed, vwant = _snapshot(b, fused), _vn_snap(vn)
    replayed["starts"] = ref._last_starts.clone()
    _assert_same_final(end, replayed)
    _assert_stats_close(end["stats"], replayed["stats"])
    assert torch.equal(end["starts"], replayed["starts"])
    assert torch.equal(got["episode_starts"], want["episode_starts"])
    assert end["step_index"] == start["step_index"] + T
    _assert_vn_close(vend, vwant)
    assert _ulps(got["obs"], want["obs"]) <= 1.0
    # rewards: where an episode ended the critic may have bootstrapped a truncation (its MLP rounding and the
    # 1-ulp observations differ: 1e-5, relative where |reward| >= 1, as test_gpu_policy_collect)
    done = torch.cat([got["episode_starts"][1:], end["starts"][None]]) != 0
    err = (got["rewards"] - want["rewards"]).abs() / want["rewards"].abs().clamp(min=1.0)
    if norm_reward:
        rel = (got["rewards"] - want["rewards"]).abs() / want["rewards"].abs().clamp(min=1e-30)
        assert float(rel[~done].max()) <= 1e-6
    else:
        assert bool((got["rewards"] == want["rewards"])[~done].all())
    assert float(torch.cat([err[done], err.new_zeros(1)]).max()) <= 1e-5
    if T > 1:
        assert float(end["stats"][6] - start["stats"][6]) > 0, "the window should contain truncations"
    if kind == "hr_sync" and n > 3:
        assert float(end["stats"][5] - start["stats"][5]) > 0, "the window should contain terminations"
    if not norm_obs:
        assert torch.equal(vend["obs_mean"], vstart["obs_mean"]) and torch.equal(vend["obs_count"], vstart["obs_count"])
    venv.close()


def test_raw_streams_through_the_sb3_restatement():
    """1,000 pmsm_sync envs x 64 steps: the raw obs / reward / done streams of a fused window, fed to
    oracle/sb3_ref's VecNormalize restatement, give the buffer observations, rewards and statistics."""
    _need_gpu()
    from gym_lorenz_b200 import rl_ops
    from oracle import sb3_ref as S
    n, T = 1000, 64
    venv, vn, m, col = _collector("pmsm_sync", n, T, max_steps=9)
    b = venv.batch
    NP = b.n_pad
    col.collect()
    streams = {"obs": torch.empty((T, b.obs_dim, NP), dtype=torch.float32, device=b.device),
               "reward": torch.empty((T, NP), dtype=b.real, device=b.device),
               "done": torch.empty((T, NP), dtype=torch.uint8, device=b.device)}
    col._io.obs, col._io.obs_es, col._io.obs_cs = rl_ops._p(streams["obs"]), 1, NP
    col._io.reward, col._io.done = rl_ops._p(streams["reward"]), rl_ops._p(streams["done"])
    col._desc.obs_ts, col._desc.rew_ts, col._desc.done_ts = b.obs_dim * NP, NP, NP
    s0 = _vn_snap(vn)
    obs0 = b._view(b.obs_planes).cpu().numpy().copy()
    out = {k: v.cpu().numpy() for k, v in col.collect().items()}
    raw = {k: v.cpu().numpy() for k, v in streams.items()}
    ref = S.VecNormalizeRef(None, None, n, b.obs_dim, norm_obs=True, norm_reward=False, clip_obs=vn.clip_obs,
                            clip_reward=vn.clip_reward, gamma=vn.gamma, epsilon=vn.epsilon)
    ref.obs_rms.mean, ref.obs_rms.var = s0["obs_mean"].cpu().numpy(), s0["obs_var"].cpu().numpy()
    ref.obs_rms.count = float(s0["obs_count"].item())
    ref.ret_rms.mean, ref.ret_rms.var = s0["ret_mean"].cpu().numpy()[0], s0["ret_var"].cpu().numpy()[0]
    ref.ret_rms.count = float(s0["ret_count"].item())
    ref.returns = s0["returns"].cpu().numpy().copy()
    assert np.allclose(out["obs"][0], ref.normalize_obs(obs0), rtol=2e-5, atol=2e-5)
    t_idx = {"t": 0}

    def step_fn(_):
        t = t_idx["t"]
        return raw["obs"][t, :, :n].T, raw["reward"][t, :n].astype(np.float64), raw["done"][t, :n]
    ref.step_fn = step_fn
    for t in range(T):
        nobs, nrew, done = ref.step(None)
        t_idx["t"] += 1
        if t + 1 < T:
            assert np.allclose(out["obs"][t + 1], nobs, rtol=2e-5, atol=2e-5), t
        plain = done == 0
        assert np.array_equal(out["rewards"][t][plain], nrew[plain].astype(np.float32)), t
    assert np.array_equal(b._view(b.obs_planes).cpu().numpy(), raw["obs"][T - 1, :, :n].T)
    assert np.allclose(vn.obs_rms.mean.cpu().numpy(), ref.obs_rms.mean, rtol=1e-5, atol=1e-5)
    assert np.allclose(vn.obs_rms.var.cpu().numpy(), ref.obs_rms.var, rtol=2e-5)
    assert np.isclose(vn.ret_rms.mean.item(), ref.ret_rms.mean, rtol=1e-12)
    assert np.isclose(vn.ret_rms.var.item(), ref.ret_rms.var, rtol=1e-11)
    assert vn.obs_rms.count == pytest.approx(ref.obs_rms.count, rel=1e-15)
    assert vn.ret_rms.count == pytest.approx(ref.ret_rms.count, rel=1e-15)
    assert np.allclose(vn.returns.cpu().numpy(), ref.returns, rtol=1e-12, atol=1e-9)
    venv.close()


def _window(col, vn, b):
    out = {k: v.clone() for k, v in col.collect().items()}
    out["last_values"] = col.last_values.clone()
    return out, _snapshot(b, col), _vn_snap(vn)


@pytest.mark.parametrize("kind,n", [("hr_sync", 1000), ("pmsm_sync", 262144)])
def test_windows_are_bit_reproducible_and_chain(kind, n):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector
    T = 16
    venv, vn, m, one = _collector(kind, n, T // 2, norm_reward=True)
    b = venv.batch
    two = FusedRolloutCollector(vn, m, T, normalize=vn, update_normalize=True)
    one.collect()
    start, vstart = _snapshot(b, one), _vn_snap(vn)
    w1, end1, v1 = _window(one, vn, b)
    w2, end2, v2 = _window(one, vn, b)
    # the same two windows again from the same snapshot: bit for bit, statistics included
    _restore(b, one, start)
    _vn_restore(vn, vstart)
    w1b, _, v1b = _window(one, vn, b)
    w2b, end2b, v2b = _window(one, vn, b)
    for a, c in ((w1, w1b), (w2, w2b), (v1, v1b), (v2, v2b)):
        for k in a:
            assert torch.equal(a[k], c[k]), k
    _assert_same_final(end2, end2b)
    # two windows of T/2 == one window of T
    two._started = True
    _restore(b, two, start)
    _vn_restore(vn, vstart)
    big, end_big, vbig = _window(two, vn, b)
    for k in KEYS[:6]:
        assert torch.equal(torch.cat([w1[k], w2[k]]), big[k]), k
    assert torch.equal(w2["last_values"], big["last_values"])
    for k in VN_KEYS:
        assert torch.equal(v2[k], vbig[k]), k
    _assert_same_final(end2, end_big)
    assert torch.equal(end2["starts"], end_big["starts"])
    venv.close()


def test_graph_replays_equal_eager_calls():
    _need_gpu()
    n, T = 1000, 16
    venv, vn, m, col = _collector("hr_sync", n, T, max_steps=10, norm_reward=True)
    b = venv.batch
    col.collect()
    start, vstart = _snapshot(b, col), _vn_snap(vn)
    eager = [_window(col, vn, b) for _ in range(3)]
    _restore(b, col, start)
    _vn_restore(vn, vstart)
    b.set_graph_mode(True)
    col.collect()                                  # warm-up = eager window 1
    torch.cuda.synchronize(b.device)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = col.collect()
    for w in (1, 2):
        g.replay()
        for k in KEYS:
            assert torch.equal(out[k], eager[w][0][k]), (w, k)
        for k, v in _vn_tensors(vn).items():
            assert torch.equal(v, eager[w][2][k]), (w, k)
    b.set_graph_mode(False)
    _assert_same_final(eager[2][1], _snapshot(b, col))
    venv.close()


def test_sync_params_takes_new_weights():
    _need_gpu()
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector, pack_actor_critic
    n, T = 1000, 16
    venv, vn, m, col = _collector("pmsm_sync", n, T, max_steps=10, seed=4)
    b = venv.batch
    col.collect()
    start, vstart = _snapshot(b, col), _vn_snap(vn)
    with torch.no_grad():
        for q in m.parameters():
            q.mul_(1.5)
    col.sync_params()
    got, _, vgot = _window(col, vn, b)
    fresh = FusedRolloutCollector(vn, pack_actor_critic(m, b.device, "pmsm_sync"), T, normalize=vn,
                                  update_normalize=True)
    fresh._started = True
    _restore(b, fresh, start)
    _vn_restore(vn, vstart)
    want, _, vwant = _window(fresh, vn, b)
    for k in KEYS:
        assert torch.equal(got[k], want[k]), k
    for k in VN_KEYS:
        assert torch.equal(vgot[k], vwant[k]), k
    venv.close()


def test_network_outputs_match_torch_on_the_buffer_observations():
    _need_gpu()
    from gym_lorenz_b200 import _lib as L
    from test_policy_collect_cpu import policy_noise
    n, T = 1000, 48
    venv, vn, m, col = _collector("hr_sync", n, T, max_steps=20, seed=7)
    b = venv.batch
    col.collect()
    s0 = b.step_index
    out = col.collect()
    z = out["obs"]
    eps = torch.tensor(policy_noise(L.load(), SEED, range(n), range(s0, s0 + T)), dtype=torch.float32, device=b.device)
    mu, std = _actor(m, z), m.log_std.detach().exp()
    dist = torch.distributions.Normal(mu, std)
    checks = {"actions": (out["actions"], mu + std * eps),
              "values": (out["values"], _critic(m, z)),
              "log_probs": (out["log_probs"], dist.log_prob(out["actions"]).sum(-1)),
              "last_values": (col.last_values, _critic(m, vn.normalize_obs(b._view(b.obs_planes))))}
    for k, (g, w) in checks.items():
        assert float((g - w).abs().max()) <= 1e-5, k
    venv.close()
