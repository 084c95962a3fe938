"""cl_policy_rollout on the B200: the fused policy evaluation replays bit for bit through cl_rollout,
its actions are the torch float32 MlpPolicy's, its streamed metrics are eval_metrics' on the recorded
trajectories, and windows chain."""
import json
import os
import types

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STREAMS = ("obs", "action", "reward", "done")


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def _modules(seed, scale=1.0):
    torch.manual_seed(seed)
    pnet = torch.nn.Sequential(torch.nn.Linear(6, 64), torch.nn.Tanh(), torch.nn.Linear(64, 64), torch.nn.Tanh())
    anet = torch.nn.Linear(64, 2)
    with torch.no_grad():
        for p in list(pnet.parameters()) + list(anet.parameters()):
            p.mul_(scale)
    return pnet, anet


def _batch(kind, n, autoreset=False, max_episode_steps=None, seed=5, add_noise=True):
    from gym_lorenz_b200.core import ChaosBatch
    kw = {"eval_mode": True} if kind == "hr_sync" and add_noise else {}
    b = ChaosBatch(kind, n, seed=seed, autoreset=autoreset, max_episode_steps=max_episode_steps,
                   add_noise=add_noise, **kw)
    b.reset()
    b.step(torch.zeros((n, b.act_dim), device=b.device))   # a step index > 0, episode counters running
    return b


def _normalizer(b, run="0.50"):
    from gym_lorenz_b200.rl_ops import DeviceVecNormalize
    art = json.load(open(os.path.join(ROOT, "tests", "golden", "sb3_artefacts.json")))["runs"][run]
    vn = DeviceVecNormalize(types.SimpleNamespace(batch=b, num_envs=b.num_envs), training=False,
                            clip_obs=art["clip_obs"], epsilon=art["epsilon"])
    vn.obs_rms.mean.copy_(torch.tensor(art["obs_mean"], dtype=torch.float64))
    vn.obs_rms.var.copy_(torch.tensor(art["obs_var"], dtype=torch.float64))
    return vn


def _snapshot(b):
    torch.cuda.synchronize(b.device)
    return {"state": b.state.clone(), "aux_int": b.aux_int.clone(), "ep_len": b.ep_len.clone(),
            "ep_return": b.ep_return.clone(), "step_index": b.step_index, "stats": b.stats_buf.clone(),
            "obs": b._view(b.obs_planes).clone()}


def _restore(b, snap):
    b.load_state_dict({"kind": b.kind_name, "num_envs": b.num_envs, **{k: v for k, v in snap.items() if k != "obs"}})


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


CASES = [("hr_sync", 1000, False, None), ("pmsm_sync", 1000, False, None),
         ("hr_sync", 65536, False, None), ("pmsm_sync", 65536, False, None),
         ("hr_sync", 1000, True, 24), ("pmsm_sync", 1000, True, 24)]


@pytest.mark.parametrize("kind,n,autoreset,max_steps", CASES)
def test_replay_through_rollout_is_bit_identical(kind, n, autoreset, max_steps):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_policy
    b = _batch(kind, n, autoreset, max_steps)
    T = 64
    params = pack_policy(_modules(11), b.device, kind)
    norm = _normalizer(b) if kind == "pmsm_sync" else None
    start = _snapshot(b)
    res = evaluate_policy(b, params, T, normalize=norm, record=STREAMS)
    end = _snapshot(b)
    _restore(b, start)
    ref = b.rollout(T, actions=res["action"])
    torch.cuda.synchronize(b.device)
    for k in ("obs", "reward", "done"):
        assert torch.equal(res[k][..., :n], ref[k][..., :n]), k
    replayed = _snapshot(b)
    replayed["obs"] = ref["obs"][-1, :, :n].t().contiguous()
    _assert_same_final(end, replayed)
    _assert_stats_close(end["stats"], replayed["stats"])
    if autoreset:
        assert bool((res["done"][:, :n] != 0).any()), "the window should contain auto-resets"
    assert end["step_index"] == start["step_index"] + T
    b.close()


@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
def test_actions_match_the_torch_policy(kind):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_policy
    n, T = 1000, 48
    b = _batch(kind, n, autoreset=True, max_episode_steps=20)
    pnet, anet = _modules(7)
    norm = _normalizer(b) if kind == "pmsm_sync" else None
    obs0 = b._view(b.obs_planes).clone()
    res = evaluate_policy(b, pack_policy((pnet, anet), b.device, kind), T, normalize=norm, record=("obs", "action"))
    seen = torch.cat([obs0[None], res["obs"][:-1, :, :n].permute(0, 2, 1)])     # [T, N, 6]: what each interval acted on
    x = seen.reshape(T * n, 6).contiguous()
    if norm is not None:
        x = norm.normalize_obs(x)
    pnet, anet = pnet.to(b.device), anet.to(b.device)
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            want = torch.clamp(anet(pnet(x)), -1.0, 1.0).view(T, n, 2)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    assert float((res["action"] - want).abs().max()) <= 1e-5
    assert float(want.abs().max()) > 0.1          # the policy is not trivially zero
    b.close()


def _metrics_vs_eval(b, res, n, dt, band, steady):
    from gym_lorenz_b200.rl_ops import eval_metrics
    err = res["obs"][:, :3, :n].double()
    ctrl = res["action"].permute(0, 2, 1).double()
    ref = eval_metrics(err, ctrl, dt=dt, error_band=band, steady_start=steady)
    for k in ("mae", "rmse", "energy"):
        got, want = res[k].cpu(), ref[k].cpu()
        assert torch.all((got - want).abs() <= 1e-12 * want.abs()), k
    assert torch.equal(res["settling_time"].isnan(), ref["settling_time"].isnan())
    ok = ~ref["settling_time"].isnan()
    assert torch.equal(res["settling_time"][ok], ref["settling_time"][ok])
    return ref


@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
def test_streamed_metrics_equal_eval_metrics(kind):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_policy
    n, T = 1000, 300
    b = _batch(kind, n)
    norm = _normalizer(b) if kind == "pmsm_sync" else None
    band = 0.05
    res = evaluate_policy(b, pack_policy(_modules(3), b.device, kind), T, normalize=norm, error_band=band,
                          record=("obs", "action"))
    _metrics_vs_eval(b, res, n, 0.001, band, min(1000, T // 2))
    b.close()


def test_metrics_special_cases_never_settles_and_never_leaves_the_band():
    _need_gpu()
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_policy
    n, T, k = 1000, 200, 100
    b = _batch("hr_sync", n, add_noise=False)
    # envs 0..k-1: slave = master, no noise, zero policy -> the error is exactly 0 at every step
    b.state[3:6, :k] = b.state[0:3, :k]
    obs0 = b._view(b.obs_planes).clone()
    obs0[:k, :3] = 0.0
    zero = pack_policy(_modules(0, scale=0.0), b.device)
    band = 1e-9   # the unsynchronised chaotic pairs are never within it
    res = evaluate_policy(b, zero, T, error_band=band, steady_start=50, obs0=obs0, record=("obs", "action"))
    ref = _metrics_vs_eval(b, res, n, 0.001, band, 50)
    st = ref["settling_time"].cpu()
    assert torch.all(st[:k] == 0.0) and torch.all(res["mae"][:k] == 0.0)
    assert bool(st[k:].isnan().all())
    assert float(res["energy"].abs().max()) == 0.0
    b.close()


@pytest.mark.parametrize("kind", ["hr_sync", "pmsm_sync"])
def test_windows_chain_and_repeat(kind):
    _need_gpu()
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_policy
    n, T1, T2 = 1000, 40, 25
    b = _batch(kind, n, autoreset=True, max_episode_steps=30)
    params = pack_policy(_modules(5), b.device, kind)
    norm = _normalizer(b) if kind == "pmsm_sync" else None
    start = _snapshot(b)
    one = evaluate_policy(b, params, T1 + T2, normalize=norm, record=STREAMS)
    end_one = _snapshot(b)
    _restore(b, start)
    r1 = evaluate_policy(b, params, T1, normalize=norm, record=STREAMS, obs0=start["obs"])
    r2 = evaluate_policy(b, params, T2, normalize=norm, record=STREAMS)     # continues from the obs planes
    end_two = _snapshot(b)
    for k in STREAMS:   # obs / reward / done are [T, ..., n_pad]: the padding columns are never written
        assert torch.equal(torch.cat([r1[k], r2[k]])[..., :n], one[k][..., :n]), k
    _assert_same_final(end_one, end_two)
    # determinism: the same call twice
    _restore(b, start)
    again = evaluate_policy(b, params, T1 + T2, normalize=norm, record=STREAMS, obs0=start["obs"])
    for k in STREAMS:
        assert torch.equal(again[k][..., :n], one[k][..., :n]), k
    for k in ("mae", "rmse", "settling_time", "energy"):
        assert torch.equal(again[k].nan_to_num(-1.0), one[k].nan_to_num(-1.0)), k
    _assert_same_final(end_one, _snapshot(b))
    b.close()


def test_graph_mode_replays_advance_like_eager_calls():
    _need_gpu()
    from gym_lorenz_b200.rl_ops import evaluate_policy, pack_policy
    n, T = 1000, 16
    b = _batch("hr_sync", n, autoreset=True, max_episode_steps=10)
    params = pack_policy(_modules(2), b.device)
    start = _snapshot(b)
    eager = [evaluate_policy(b, params, T, record=("obs",))["obs"].clone() for _ in range(3)]
    end_eager = _snapshot(b)
    _restore(b, start)
    b._view(b.obs_planes).copy_(start["obs"])
    b.set_graph_mode(True)
    evaluate_policy(b, params, T, record=("obs",))          # warm-up = eager window 1
    torch.cuda.synchronize(b.device)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = evaluate_policy(b, params, T, record=("obs",))
    got = []
    for _ in range(2):
        g.replay()
        got.append(out["obs"].clone())
    b.set_graph_mode(False)
    assert torch.equal(got[0][..., :n], eager[1][..., :n]) and torch.equal(got[1][..., :n], eager[2][..., :n])
    _assert_same_final(end_eager, _snapshot(b))
    b.close()
