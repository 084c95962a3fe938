"""pack_actor_critic / FusedRolloutCollector argument handling and the policy-noise stream: layout of the
packed actor-critic block, SB3 zip reading, in-place repacking, every refusal, and a restatement of the
Gaussian policy noise (Philox purpose TAG_POLICY + Box-Muller) -- all without a GPU."""
import ctypes as C
import io
import math
import types
import zipfile

import numpy as np
import pytest
import torch

from gym_lorenz_b200 import rl_ops

TAG_POLICY = 0x40000000
H = 64


class SB3Policy(torch.nn.Module):
    """The parameter names of a stable-baselines3 ActorCriticPolicy with net_arch [64, 64] and Tanh."""

    def __init__(self, seed=0, obs_dim=6, act_dim=2, hidden=H):
        super().__init__()
        torch.manual_seed(seed)
        mlp = lambda: torch.nn.Sequential(torch.nn.Linear(obs_dim, hidden), torch.nn.Tanh(),
                                          torch.nn.Linear(hidden, hidden), torch.nn.Tanh())
        self.mlp_extractor = torch.nn.Module()
        self.mlp_extractor.policy_net, self.mlp_extractor.value_net = mlp(), mlp()
        self.action_net, self.value_net = torch.nn.Linear(hidden, act_dim), torch.nn.Linear(hidden, 1)
        self.log_std = torch.nn.Parameter(torch.linspace(-0.7, 0.2, act_dim))


def _ordered(m):
    e = m.mlp_extractor
    return [e.policy_net[0].weight, e.policy_net[0].bias, e.policy_net[2].weight, e.policy_net[2].bias,
            m.action_net.weight, m.action_net.bias,
            e.value_net[0].weight, e.value_net[0].bias, e.value_net[2].weight, e.value_net[2].bias,
            m.value_net.weight, m.value_net.bias, m.log_std]


def test_packed_layout_at_the_documented_offsets(chaos_lib):
    m = SB3Policy(seed=3)
    p = rl_ops.pack_actor_critic(m, "cpu")
    n_actor = H * 6 + H + H * H + H + 2 * H + 2
    n_critic = H * 6 + H + H * H + H + H + 1
    assert p.dtype == torch.float32 and p.numel() == n_actor + n_critic + 2
    assert 4 * n_actor == 18952 and 4 * n_critic == 18692 and 4 * p.numel() == 37652
    o = 0
    for t in _ordered(m):
        assert torch.equal(p[o:o + t.numel()].view(t.shape), t.detach())
        o += t.numel()
    assert o == p.numel()
    # the actor prefix is pack_policy's block, bit for bit: evaluate_policy runs on block[:n_actor]
    actor = rl_ops.pack_policy(m.state_dict(), "cpu")
    assert actor.numel() == n_actor and torch.equal(p[:n_actor], actor)


def test_state_dict_module_and_zip_round_trip(chaos_lib, tmp_path):
    m = SB3Policy(seed=1)
    ref = rl_ops.pack_actor_critic(m, "cpu", "pmsm_sync")
    sd = m.state_dict()
    assert torch.equal(rl_ops.pack_actor_critic(sd, "cpu", "pmsm_sync"), ref)
    buf = io.BytesIO()
    torch.save(sd, buf)
    path = tmp_path / "a2c_model.zip"
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", "{}")
        z.writestr("policy.pth", buf.getvalue())
    assert torch.equal(rl_ops.pack_actor_critic(str(path), "cpu", "pmsm_sync"), ref)
    assert torch.equal(rl_ops.pack_actor_critic(path, "cpu"), ref)


def test_out_packs_in_place(chaos_lib):
    m = SB3Policy(seed=2)
    out = torch.full((rl_ops.pack_actor_critic(m, "cpu").numel(),), float("nan"))
    ptr = out.data_ptr()
    with torch.no_grad():
        for q in m.parameters():
            q.add_(0.25)
    got = rl_ops.pack_actor_critic(m, "cpu", out=out)
    assert got is out and out.data_ptr() == ptr
    assert torch.equal(out, rl_ops.pack_actor_critic(m, "cpu"))
    for bad in (torch.zeros(out.numel() + 1), torch.zeros(out.numel(), dtype=torch.float64),
                torch.zeros(2 * out.numel())[::2]):
        with pytest.raises(ValueError, match="out must be"):
            rl_ops.pack_actor_critic(m, "cpu", out=bad)


@pytest.mark.parametrize("case", ["v1_obs_dim", "wv_rows", "c2_len", "log_std_len", "three_layers",
                                  "no_value_net", "no_value_head", "no_log_std", "actor_w1"])
def test_wrong_shapes_and_missing_parts_raise(chaos_lib, case):
    sd = dict(SB3Policy().state_dict())
    if case == "v1_obs_dim":
        sd["mlp_extractor.value_net.0.weight"] = torch.zeros(H, 8)
    elif case == "wv_rows":
        sd["value_net.weight"], sd["value_net.bias"] = torch.zeros(2, H), torch.zeros(2)
    elif case == "c2_len":
        sd["mlp_extractor.value_net.2.bias"] = torch.zeros(32)
    elif case == "log_std_len":
        sd["log_std"] = torch.zeros(3)
    elif case == "three_layers":
        sd["mlp_extractor.value_net.4.weight"], sd["mlp_extractor.value_net.4.bias"] = torch.zeros(H, H), torch.zeros(H)
    elif case == "no_value_net":
        for k in [k for k in sd if k.startswith("mlp_extractor.value_net.")]:
            del sd[k]
    elif case == "no_value_head":
        del sd["value_net.weight"]
    elif case == "no_log_std":
        del sd["log_std"]
    else:
        sd["mlp_extractor.policy_net.0.weight"] = torch.zeros(H, 8)
    with pytest.raises(ValueError):
        rl_ops.pack_actor_critic(sd, "cpu")


def _fake_env(kind="hr_sync", obs_f64=False, n=4):
    # no library context, no device buffers: reaching a launch would fail with something else than ValueError
    from gym_lorenz_b200 import _lib as L
    b = types.SimpleNamespace(kind=L.KIND_NAMES[kind], kind_name=kind, obs_f64=obs_f64, num_envs=n, n_pad=128,
                              obs_dim=6, act_dim=2, device=torch.device("cpu"))
    return types.SimpleNamespace(batch=b)


def test_collector_refusals_before_launch(chaos_lib):
    m = SB3Policy()
    for kind in ("lorenz3", "pmsm_classic", "lorenz_rk4"):
        with pytest.raises(ValueError, match="hr_sync and pmsm_sync"):
            rl_ops.pack_actor_critic(m, "cpu", kind)
        with pytest.raises(ValueError, match="hr_sync and pmsm_sync"):
            rl_ops.FusedRolloutCollector(_fake_env(kind), m, 8)
    with pytest.raises(ValueError, match="float32"):
        rl_ops.FusedRolloutCollector(_fake_env(obs_f64=True), m, 8)
    for n_steps in (0, -3):
        with pytest.raises(ValueError, match="n_steps"):
            rl_ops.FusedRolloutCollector(_fake_env(), m, n_steps)
    frozen = dict(training=False, norm_obs=True, norm_reward=False)
    with pytest.raises(ValueError, match="training"):
        rl_ops.FusedRolloutCollector(_fake_env(), m, 8, normalize=types.SimpleNamespace(**{**frozen, "training": True}))
    with pytest.raises(ValueError, match="norm_reward"):
        rl_ops.FusedRolloutCollector(_fake_env(), m, 8, normalize=types.SimpleNamespace(**{**frozen, "norm_reward": True}))
    with pytest.raises(ValueError, match="packed actor-critic"):
        rl_ops.FusedRolloutCollector(_fake_env(), torch.zeros(7), 8)


def policy_noise(lib, seed, gids, steps):
    """eps [len(steps), len(gids), 2] of the collector: Philox4x32-10 with key (seed lo, seed hi ^ step >> 32)
    and counter (global env id lo, hi, step lo, TAG_POLICY), then Box-Muller on two 53-bit uniforms."""
    ctr, key, out = (C.c_uint32 * 4)(), (C.c_uint32 * 2)(), (C.c_uint32 * 4)()
    words = np.empty((len(steps), len(gids), 4), np.uint64)
    for a, step in enumerate(steps):
        key[0], key[1] = seed & 0xFFFFFFFF, ((seed >> 32) ^ ((step >> 32) & 0xFFFFFF)) & 0xFFFFFFFF
        for b, g in enumerate(gids):
            ctr[0], ctr[1], ctr[2], ctr[3] = g & 0xFFFFFFFF, g >> 32, step & 0xFFFFFFFF, TAG_POLICY
            lib.cl_philox4x32_10(ctr, key, out)
            words[a, b] = out[0], out[1], out[2], out[3]
    u = lambda hi, lo: ((hi >> np.uint64(5)) * np.uint64(1 << 26) + (lo >> np.uint64(6))).astype(np.float64) / 2.0 ** 53
    u1, u2 = 1.0 - u(words[..., 0], words[..., 1]), u(words[..., 2], words[..., 3])
    rad = np.sqrt(-2.0 * np.log(u1))
    return np.stack([rad * np.cos(2.0 * np.pi * u2), rad * np.sin(2.0 * np.pi * u2)], axis=-1)


def test_policy_noise_stream_is_standard_normal(chaos_lib):
    from scipy import stats
    eps = policy_noise(chaos_lib, 0x1234_5678_9ABC, list(range(5000)) + [2 ** 33 + 7], list(range(100))).reshape(-1)
    assert eps.size >= 10 ** 6
    assert abs(eps.mean()) < 5.0 / math.sqrt(eps.size)
    assert abs(eps.var() - 1.0) < 5.0 * math.sqrt(2.0 / eps.size)
    assert abs(stats.skew(eps)) < 0.01 and abs(stats.kurtosis(eps)) < 0.02
    assert stats.kstest(eps, "norm").pvalue > 1e-3
    # the two components of a draw are independent, and so are neighbouring envs and steps
    e = policy_noise(chaos_lib, 7, range(64), range(64))
    for x, y in ((e[..., 0], e[..., 1]), (e[:, :-1, 0], e[:, 1:, 0]), (e[:-1, :, 0], e[1:, :, 0])):
        assert abs(np.corrcoef(x.reshape(-1), y.reshape(-1))[0, 1]) < 0.05
