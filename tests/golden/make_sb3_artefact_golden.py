"""Extracts what the reference's own SB3 artefacts hold about the wrappers around the env (needs its sources).

    GYM_LORENZ_REFERENCE=<gym-lorenz checkout> python tests/golden/make_sb3_artefact_golden.py

The reference ships eight finished training runs of code/lorenz_pmsm/train.py:152-190
(`DummyVecEnv([Monitor(make_env(alpha))])` -> `VecNormalize(norm_obs=True, norm_reward=False,
clip_obs=10.0)` -> `A2C.learn(1_000_000)`): `pmsm_a2c_alpha_<a>_clean_model` (SB3 2.7.1 zip) and
`pmsm_a2c_alpha_<a>_clean_vecnorm.pkl` (pickled VecNormalize).  stable_baselines3 / gymnasium are not
installed, so the pickles are opened with attribute-bag stand-ins for their classes; only numbers are read.

Output tests/golden/sb3_artefacts.json, per alpha:
  obs_count / ret_count   RunningMeanStd.count of obs_rms / ret_rms (float.hex)
  obs_mean / obs_var, ret_mean / ret_var
  clip_obs, clip_reward, gamma, epsilon, norm_obs, norm_reward, training
  old_obs, old_reward     VecNormalize's last unnormalised observation / reward (float32)
  num_timesteps, n_envs, last_episode_starts, last_original_obs, last_obs     from the model zip
  ep_l, ep_r, ep_t        Monitor records of the last 100 episodes (model.ep_info_buffer)
(The zip and the pkl of one alpha are not from the same process -- their last observations differ -- so
`last_obs` cannot be replayed from the pkl statistics; each file pins what it holds on its own.)
"""
from __future__ import annotations

import base64
import glob
import io
import json
import os
import pickle
import warnings
import zipfile

import numpy as np

REF = os.environ["GYM_LORENZ_REFERENCE"]
HERE = os.path.dirname(os.path.abspath(__file__))


class _Bag:
    def __init__(self, *a, **k):
        pass

    def __setstate__(self, st):
        self.__dict__.update(st)


class _Unpickler(pickle.Unpickler):
    def find_class(self, mod, name):
        if mod.split(".")[0] in ("stable_baselines3", "gym", "gymnasium"):
            return type(name, (_Bag,), {"__module__": mod})
        return super().find_class(mod, name)


def _b64(field):
    return _Unpickler(io.BytesIO(base64.b64decode(field[":serialized:"]))).load()


def main():
    warnings.simplefilter("ignore")
    out = {}
    for zpath in sorted(glob.glob(os.path.join(REF, "pmsm_a2c_alpha_*_clean_model"))):
        alpha = os.path.basename(zpath).split("alpha_")[1][:4]
        with open(os.path.join(REF, f"pmsm_a2c_alpha_{alpha}_clean_vecnorm.pkl"), "rb") as f:
            vn = _Unpickler(f).load()
        data = json.loads(zipfile.ZipFile(zpath).read("data"))
        ep = list(_b64(data["ep_info_buffer"]))
        out[alpha] = {
            "obs_count": float(vn.obs_rms.count).hex(), "ret_count": float(vn.ret_rms.count).hex(),
            "obs_mean": np.asarray(vn.obs_rms.mean).tolist(), "obs_var": np.asarray(vn.obs_rms.var).tolist(),
            "ret_mean": float(vn.ret_rms.mean), "ret_var": float(vn.ret_rms.var),
            "clip_obs": vn.clip_obs, "clip_reward": vn.clip_reward, "gamma": vn.gamma, "epsilon": vn.epsilon,
            "norm_obs": vn.norm_obs, "norm_reward": vn.norm_reward, "training": vn.training,
            "num_envs": vn.num_envs,
            "old_obs": np.asarray(vn.old_obs, np.float32).reshape(-1).tolist(),
            "old_reward": np.asarray(vn.old_reward, np.float32).reshape(-1).tolist(),
            "num_timesteps": data["num_timesteps"], "n_envs": data["n_envs"], "n_steps": data["n_steps"],
            "stats_window_size": data["_stats_window_size"],
            "last_episode_starts": np.asarray(_b64(data["_last_episode_starts"])).astype(bool).tolist(),
            "last_original_obs": np.asarray(_b64(data["_last_original_obs"]), np.float32).reshape(-1).tolist(),
            "last_obs": np.asarray(_b64(data["_last_obs"]), np.float32).reshape(-1).tolist(),
            "ep_l": [int(e["l"]) for e in ep], "ep_r": [float(e["r"]) for e in ep], "ep_t": [float(e["t"]) for e in ep],
        }
    with open(os.path.join(REF, "_stable_baselines3_version")) as f:
        ver = f.read().strip()
    with open(os.path.join(HERE, "sb3_artefacts.json"), "w") as f:
        json.dump({"stable_baselines3": ver, "runs": out}, f, indent=0, sort_keys=True)
    print("wrote sb3_artefacts.json:", sorted(out), "SB3", ver)


if __name__ == "__main__":
    main()
