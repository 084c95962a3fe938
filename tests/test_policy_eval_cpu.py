"""pack_policy / evaluate_policy argument handling: layout of the packed parameter block, SB3 zip
reading, and every refusal -- all before anything reaches a GPU."""
import io
import types
import zipfile

import pytest
import torch

from gym_lorenz_b200 import rl_ops


def _modules(seed=0, obs_dim=6, act_dim=2, hidden=64, act=torch.nn.Tanh):
    torch.manual_seed(seed)
    pnet = torch.nn.Sequential(torch.nn.Linear(obs_dim, hidden), act(), torch.nn.Linear(hidden, hidden), act())
    return pnet, torch.nn.Linear(hidden, act_dim)


def _sb3_state_dict(pnet, anet):
    sd = {"mlp_extractor.policy_net." + k: v for k, v in pnet.state_dict().items()}
    sd.update({"mlp_extractor.value_net.0.weight": torch.zeros(64, 6), "value_net.weight": torch.zeros(1, 64),
               "log_std": torch.zeros(2)})
    sd.update({"action_net." + k: v for k, v in anet.state_dict().items()})
    return sd


def test_pack_layout_offsets(chaos_lib):
    pnet, anet = _modules()
    p = rl_ops.pack_policy((pnet, anet), "cpu")
    assert p.dtype == torch.float32 and p.shape == (64 * 6 + 64 + 64 * 64 + 64 + 2 * 64 + 2,)
    o = 0
    for t in (pnet[0].weight, pnet[0].bias, pnet[2].weight, pnet[2].bias, anet.weight, anet.bias):
        n = t.numel()
        assert torch.equal(p[o:o + n].view(t.shape), t.detach())
        o += n
    assert o == p.numel()
    # W2 starts on a 16-byte boundary (the kernel reads its rows as float4)
    assert (64 * 6 + 64) % 4 == 0


def test_state_dict_and_zip_round_trip(chaos_lib, tmp_path):
    pnet, anet = _modules(seed=1)
    ref = rl_ops.pack_policy((pnet, anet), "cpu", "pmsm_sync")
    sd = _sb3_state_dict(pnet, anet)
    assert torch.equal(rl_ops.pack_policy(sd, "cpu", "pmsm_sync"), ref)
    buf = io.BytesIO()
    torch.save(sd, buf)
    path = tmp_path / "ppo_model.zip"
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", "{}")
        z.writestr("policy.pth", buf.getvalue())
        z.writestr("_stable_baselines3_version", "2.7.1")
    assert torch.equal(rl_ops.pack_policy(str(path), "cpu", "pmsm_sync"), ref)
    assert torch.equal(rl_ops.pack_policy(path, "cpu"), ref)
    bad = tmp_path / "not_a_model.zip"
    with zipfile.ZipFile(bad, "w") as z:
        z.writestr("data", "{}")
    with pytest.raises(ValueError, match="policy.pth"):
        rl_ops.pack_policy(bad, "cpu")


@pytest.mark.parametrize("case", ["w1_obs_dim", "w3_act_dim", "b2_len", "missing_key", "three_layers"])
def test_wrong_shapes_and_architecture_raise(chaos_lib, case):
    pnet, anet = _modules()
    sd = _sb3_state_dict(pnet, anet)
    if case == "w1_obs_dim":
        sd["mlp_extractor.policy_net.0.weight"] = torch.zeros(64, 8)
    elif case == "w3_act_dim":
        sd["action_net.weight"], sd["action_net.bias"] = torch.zeros(3, 64), torch.zeros(3)
    elif case == "b2_len":
        sd["mlp_extractor.policy_net.2.bias"] = torch.zeros(32)
    elif case == "missing_key":
        del sd["action_net.bias"]
    else:
        sd["mlp_extractor.policy_net.4.weight"], sd["mlp_extractor.policy_net.4.bias"] = torch.zeros(64, 64), torch.zeros(64)
    with pytest.raises(ValueError):
        rl_ops.pack_policy(sd, "cpu")


def test_wrong_modules_raise(chaos_lib):
    with pytest.raises(ValueError, match="Linear-Tanh"):
        rl_ops.pack_policy(_modules(act=torch.nn.ReLU), "cpu")
    with pytest.raises(ValueError):
        rl_ops.pack_policy(_modules(hidden=32), "cpu")
    with pytest.raises(ValueError):
        rl_ops.pack_policy(_modules(obs_dim=8, act_dim=3), "cpu")      # lorenz4_pair's dims
    with pytest.raises(ValueError):
        rl_ops.pack_policy(torch.nn.Linear(6, 2), "cpu")


def _fake_env(kind="hr_sync", obs_f64=False, n=4):
    # no library context, no device buffers: reaching the launch would fail with something else than ValueError
    from gym_lorenz_b200 import _lib as L
    b = types.SimpleNamespace(kind=L.KIND_NAMES[kind], kind_name=kind, obs_f64=obs_f64, num_envs=n, n_pad=128,
                              obs_dim=6, act_dim=2, device=torch.device("cpu"))
    return types.SimpleNamespace(batch=b)


def test_unsupported_kind_and_f64_obs_raise_before_launch(chaos_lib):
    sd = _sb3_state_dict(*_modules())
    for kind in ("lorenz3", "pmsm_classic", "lorenz_rk4"):
        with pytest.raises(ValueError, match="hr_sync and pmsm_sync"):
            rl_ops.pack_policy(sd, "cpu", kind)
    with pytest.raises(ValueError, match="hr_sync and pmsm_sync"):
        rl_ops.evaluate_policy(_fake_env("pmsm_classic"), sd, 10)
    with pytest.raises(ValueError, match="float32"):
        rl_ops.evaluate_policy(_fake_env(obs_f64=True), sd, 10)


def test_bad_window_arguments_raise_before_launch(chaos_lib):
    sd = _sb3_state_dict(*_modules())
    env = _fake_env()
    with pytest.raises(ValueError, match="T must be"):
        rl_ops.evaluate_policy(env, sd, 0)
    for ss in (-1, 10, 11):
        with pytest.raises(ValueError, match="steady_start"):
            rl_ops.evaluate_policy(env, sd, 10, steady_start=ss)
    with pytest.raises(ValueError, match="record"):
        rl_ops.evaluate_policy(env, sd, 10, record=("err",))
    with pytest.raises(ValueError, match="packed policy"):
        rl_ops.evaluate_policy(env, torch.zeros(7), 10)
