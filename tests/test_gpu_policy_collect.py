"""cl_policy_collect on the B200: the fused PPO / A2C rollout collector replays bit for bit through
DeviceRolloutCollector, its network outputs are the torch float32 actor-critic's on the restated policy
noise, the noise is keyed by global env id and step, GAE, window chaining, CUDA-graph replay and weight
refresh behave as in the unfused path, and the shared actor still serves evaluate_policy."""
import json
import os

import numpy as np
import pytest
import torch

from test_policy_collect_cpu import SB3Policy, policy_noise

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 5
KEYS = ("obs", "actions", "rewards", "values", "log_probs", "episode_starts", "advantages", "returns")


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _venv(kind, n, max_steps, env_id_base=0):
    from gym_lorenz_b200.vec_env import BatchedChaosVecEnv
    kw = {"eval_mode": True, "add_noise": True} if kind == "hr_sync" else {}
    return BatchedChaosVecEnv(kind, n, seed=SEED, max_episode_steps=max_steps, env_id_base=env_id_base, **kw)


def _normalizer(venv, kind):
    if kind != "pmsm_sync":
        return None
    from gym_lorenz_b200.rl_ops import DeviceVecNormalize
    art = json.load(open(os.path.join(ROOT, "tests", "golden", "sb3_artefacts.json")))["runs"]["0.50"]
    vn = DeviceVecNormalize(venv, training=False, norm_reward=False, clip_obs=art["clip_obs"], epsilon=art["epsilon"])
    vn.obs_rms.mean.copy_(torch.tensor(art["obs_mean"], dtype=torch.float64))
    vn.obs_rms.var.copy_(torch.tensor(art["obs_var"], dtype=torch.float64))
    return vn


def _policy(seed=11):
    return SB3Policy(seed=seed).cuda()


def _snapshot(b, col):
    torch.cuda.synchronize(b.device)
    return {"state": b.state.clone(), "aux_int": b.aux_int.clone(), "ep_len": b.ep_len.clone(),
            "ep_return": b.ep_return.clone(), "step_index": b.step_index, "stats": b.stats_buf.clone(),
            "obs": b._view(b.obs_planes).clone(), "starts": col.starts.clone()}


def _restore(b, col, snap):
    b.load_state_dict({"kind": b.kind_name, "num_envs": b.num_envs,
                       **{k: v for k, v in snap.items() if k not in ("obs", "starts")}})
    b._view(b.obs_planes).copy_(snap["obs"])
    col.starts.copy_(snap["starts"])


def _assert_same_final(a, c):
    for k in ("state", "aux_int", "ep_len", "ep_return", "obs"):
        assert torch.equal(a[k], c[k]), k
    assert a["step_index"] == c["step_index"]


def _assert_stats_close(s, r):
    s, r = s.cpu(), r.cpu()
    for k in (0, 3, 4, 5, 6):      # counts: exact
        assert s[k] == r[k], (k, s[k], r[k])
    for k in (1, 2):               # sums over f64 atomics in a different order
        assert abs(s[k] - r[k]) <= 1e-12 * max(abs(r[k]), 1e-300), (k, s[k], r[k])


def _no_tf32(fn):
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            return fn()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32


def _critic(m, z):
    return _no_tf32(lambda: m.value_net(m.mlp_extractor.value_net(z)).squeeze(-1))


def _actor(m, z):
    return _no_tf32(lambda: m.action_net(m.mlp_extractor.policy_net(z)))


class _Replay:
    """A DeviceRolloutCollector policy that returns the recorded actions for step t and the torch critic's
    values (the TimeLimit bootstrap reads them)."""

    def __init__(self, m, actions):
        self.m, self.actions, self.t, self.col = m, actions, 0, None

    def __call__(self, obs):
        main = obs.data_ptr() == self.col._last_obs.data_ptr()
        if main and self.t < self.actions.shape[0]:
            a = self.actions[self.t]
            self.t += 1
        else:
            a = torch.zeros_like(self.actions[0])
        return a, _critic(self.m, obs), torch.zeros(obs.shape[0], device=obs.device)


CASES = [("hr_sync", 33, 64), ("pmsm_sync", 33, 64), ("hr_sync", 1000, 64), ("pmsm_sync", 1000, 64),
         ("hr_sync", 65536, 64), ("pmsm_sync", 65536, 64), ("hr_sync", 1000, 1), ("pmsm_sync", 65536, 1)]


@pytest.mark.parametrize("kind,n,T", CASES)
def test_replay_through_device_rollout_collector(kind, n, T):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import DeviceRolloutCollector, FusedRolloutCollector
    venv = _venv(kind, n, max_steps=9)
    b, norm, m = venv.batch, _normalizer(venv, kind), _policy()
    fused = FusedRolloutCollector(venv, m, T, normalize=norm)
    for _ in range(max(1, 12 // T)):
        fused.collect()              # episodes running, some truncated already
    start = _snapshot(b, fused)
    got = {k: v.clone() for k, v in fused.collect().items()}
    end = _snapshot(b, fused)
    _restore(b, fused, start)
    replay = _Replay(m, got["actions"])
    ref = DeviceRolloutCollector(norm if norm is not None else venv, replay, T, gamma=fused.gamma)
    replay.col = ref
    ref._last_obs = (norm.normalize_obs(start["obs"]) if norm is not None else start["obs"]).clone()
    ref._last_starts.copy_(start["starts"])
    want = ref.collect()
    replayed = _snapshot(b, fused)
    replayed["starts"] = ref._last_starts.clone()
    assert torch.equal(got["obs"], want["obs"])
    assert torch.equal(got["episode_starts"], want["episode_starts"])
    assert torch.equal(end["starts"], replayed["starts"])
    _assert_same_final(end, replayed)
    _assert_stats_close(end["stats"], replayed["stats"])
    # rewards: equal except where the critic bootstrapped a truncation (only its MLP rounding differs: 1e-5,
    # or relative 1e-5 where |reward| >= 1, since at |reward| >= 128 one float32 step is already 1.5e-5)
    done = torch.cat([got["episode_starts"][1:], end["starts"][None]]) != 0
    same = got["rewards"] == want["rewards"]
    assert bool(same[~done].all())
    err = (got["rewards"] - want["rewards"]).abs() / want["rewards"].abs().clamp(min=1.0)
    assert float(torch.cat([err[done], err.new_zeros(1)]).max()) <= 1e-5
    if T > 1:
        assert float(end["stats"][6] - start["stats"][6]) > 0, "the window should contain truncations"
    assert end["step_index"] == start["step_index"] + T
    venv.close()


def _mlp64(block, z, off, nout):
    """float64 MLP read from the packed block at `off` (torch Linear layout, [64, 64], Tanh)."""
    d, h = z.shape[-1], 64
    take = lambda k, shape: (block[k:k + int(np.prod(shape))].reshape(shape), k + int(np.prod(shape)))
    W1, k = take(off, (h, d)); b1, k = take(k, (h,)); W2, k = take(k, (h, h)); b2, k = take(k, (h,))
    W3, k = take(k, (nout, h)); b3, k = take(k, (nout,))
    return np.tanh(np.tanh(z @ W1.T + b1) @ W2.T + b2) @ W3.T + b3, k


@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
def test_network_outputs_match_torch_and_float64(kind):
    _need_gpu()
    from gym_lorenz_b200 import _lib as L
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector
    n, T = 1000, 48
    venv = _venv(kind, n, max_steps=20)
    b, norm, m = venv.batch, _normalizer(venv, kind), _policy(7)
    col = FusedRolloutCollector(venv, m, T, normalize=norm)
    col.collect()
    s0 = b.step_index
    out = col.collect()
    z = out["obs"]
    eps = torch.tensor(policy_noise(L.load(), SEED, range(n), range(s0, s0 + T)), dtype=torch.float32, device=b.device)
    mu, std = _actor(m, z), m.log_std.detach().exp()
    dist = torch.distributions.Normal(mu, std)
    last_z = norm.normalize_obs(b._view(b.obs_planes)) if norm is not None else b._view(b.obs_planes)
    checks = {"actions": (out["actions"], mu + std * eps),
              "values": (out["values"], _critic(m, z)),
              "log_probs": (out["log_probs"], dist.log_prob(out["actions"]).sum(-1)),
              "last_values": (col.last_values, _critic(m, last_z))}
    for k, (g, w) in checks.items():
        assert float((g - w).abs().max()) <= 1e-5, k
    assert float(mu.abs().max()) > 0.1 and float(out["values"].abs().max()) > 0.01
    # the same outputs from a float64 MLP read at the documented offsets of the packed block
    blk = col.params.double().cpu().numpy()
    z64 = z.double().cpu().numpy()
    mu64, k = _mlp64(blk, z64, 0, 2)
    v64, k = _mlp64(blk, z64, k, 1)
    log_std = blk[k:k + 2]
    sd = np.exp(log_std)
    a64 = mu64 + sd * eps.double().cpu().numpy()
    assert np.abs(out["actions"].cpu().numpy() - a64).max() <= 1e-5
    assert np.abs(out["values"].cpu().numpy() - v64[..., 0]).max() <= 1e-5
    lp64 = (-(out["actions"].double().cpu().numpy() - mu64) ** 2 / (2 * sd ** 2) - log_std
            - 0.5 * np.log(2 * np.pi)).sum(-1)
    assert np.abs(out["log_probs"].cpu().numpy() - lp64).max() <= 1e-4 * max(1.0, np.abs(lp64).max())
    venv.close()


def test_noise_is_keyed_by_global_env_id_and_step():
    _need_gpu()
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector
    n1, n2, T = 600, 400, 16
    m = _policy(3)
    parts = []
    for base, n in ((0, n1), (n1, n2)):
        venv = _venv("hr_sync", n, 50, env_id_base=base)
        parts.append(FusedRolloutCollector(venv, m, T).collect()["actions"].clone())
        venv.close()
    venv = _venv("hr_sync", n1 + n2, 50)
    col = FusedRolloutCollector(venv, m, T)
    first = col.collect()["actions"].clone()
    assert torch.equal(torch.cat(parts, dim=1), first)
    second = col.collect()["actions"]
    assert not bool((first == second).any())
    venv.close()


@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
def test_gae_and_chaining(kind):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector, gae
    n, T = 1000, 24
    venv = _venv(kind, n, max_steps=10)
    b, norm, m = venv.batch, _normalizer(venv, kind), _policy(5)
    one = FusedRolloutCollector(venv, m, T, normalize=norm)
    two = FusedRolloutCollector(venv, m, 2 * T, normalize=norm)
    one.collect()
    out = one.collect()
    adv, ret = gae(out["rewards"], out["values"], out["episode_starts"], one.last_values, one.starts, 0.99, 0.95)
    assert torch.equal(adv, out["advantages"]) and torch.equal(ret, out["returns"])
    # two windows of T == one window of 2T, bit for bit
    start = _snapshot(b, one)
    r1 = {k: v.clone() for k, v in one.collect().items()}
    r2 = {k: v.clone() for k, v in one.collect().items()}
    end_two = _snapshot(b, one)
    two._started = True
    _restore(b, two, start)
    big = two.collect()
    end_one = _snapshot(b, two)
    for k in KEYS[:6]:
        assert torch.equal(torch.cat([r1[k], r2[k]]), big[k]), k
    assert torch.equal(one.last_values, two.last_values)
    _assert_same_final(end_two, end_one)
    assert torch.equal(end_two["starts"], end_one["starts"])
    venv.close()


def test_graph_replays_equal_eager_calls():
    _need_gpu()
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector
    n, T = 1000, 16
    venv = _venv("hr_sync", n, max_steps=10)
    b, m = venv.batch, _policy(2)
    col = FusedRolloutCollector(venv, m, T)
    col.collect()
    start = _snapshot(b, col)
    eager = [{k: v.clone() for k, v in col.collect().items()} for _ in range(3)]
    end_eager = _snapshot(b, col)
    _restore(b, col, start)
    b.set_graph_mode(True)
    col.collect()                                  # warm-up = eager window 1
    torch.cuda.synchronize(b.device)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = col.collect()
    for w in (1, 2):
        g.replay()
        for k in KEYS:
            assert torch.equal(out[k], eager[w][k]), (w, k)
    b.set_graph_mode(False)
    end = _snapshot(b, col)
    _assert_same_final(end_eager, end)
    assert torch.equal(end_eager["starts"], end["starts"])
    venv.close()


def test_sync_params_takes_new_weights_and_is_capturable():
    _need_gpu()
    from gym_lorenz_b200.rl_ops import FusedRolloutCollector, pack_actor_critic
    n, T = 1000, 16
    venv = _venv("pmsm_sync", n, max_steps=10)
    b, m = venv.batch, _policy(4)
    col = FusedRolloutCollector(venv, m, T)
    col.collect()
    start = _snapshot(b, col)
    with torch.no_grad():
        for q in m.parameters():
            q.mul_(1.5)
    col.sync_params()
    got = {k: v.clone() for k, v in col.collect().items()}
    fresh = FusedRolloutCollector(venv, pack_actor_critic(m, b.device, "pmsm_sync"), T)
    fresh._started = True
    _restore(b, fresh, start)
    want = fresh.collect()
    for k in KEYS:
        assert torch.equal(got[k], want[k]), k
    # captured: a replay copies whatever the module holds then, with no host copy in between
    torch.cuda.synchronize(b.device)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        col.sync_params()
    with torch.no_grad():
        for q in m.parameters():
            q.add_(0.125)
    g.replay()
    assert torch.equal(col.params, pack_actor_critic(m, b.device, "pmsm_sync"))
    venv.close()


@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
def test_evaluate_policy_runs_on_the_actor_prefix(kind):
    _need_gpu()
    from gym_lorenz_b200.core import ChaosBatch
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_actor_critic, pack_policy
    n, T = 1000, 40
    m = _policy(9)
    blk = pack_actor_critic(m, "cuda", kind)
    n_actor = pack_policy(m.state_dict(), "cpu", kind).numel()
    res = []
    for params in (blk[:n_actor], pack_policy(m.state_dict(), "cuda", kind)):
        b = ChaosBatch(kind, n, seed=1, autoreset=True, max_episode_steps=25)
        b.reset()
        res.append(evaluate_policy(b, params, T, record=("obs", "action")))
        b.close()
    assert torch.equal(res[0]["obs"][..., :n], res[1]["obs"][..., :n])   # padding columns are never written
    for k in ("action", "mae", "rmse", "energy"):
        assert torch.equal(res[0][k], res[1][k]), k
