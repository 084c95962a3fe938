#!/usr/bin/env python
"""PPO on the Hindmarsh-Rose synchronisation task (the reference's `train.py` setting:
`lorenz_try-v0`, lr 3e-4, gae_lambda 0.95, MlpPolicy-shaped actor-critic) with everything on the
GPU: 4,096 envs, DeviceRolloutCollector (CUDA-graph captured), GAE kernel, torch PPO update.
With --fused the rollouts come from FusedRolloutCollector instead (actor-critic, sampling, env step and
buffer writes in one kernel launch), whose weights are refreshed from the module after every update.
With --normalize the env is wrapped in DeviceVecNormalize(norm_reward=False) in training mode, the
reference's A2C pipeline; with --fused as well the kernel updates the running statistics itself
(FusedRolloutCollector(update_normalize=True)).

This is a usage example / end-to-end sanity check of the env semantics (episode return must
improve), not part of the measured hot path.   python examples/ppo_hr_device.py --updates 30
"""
import argparse, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT)
import torch
from gym_lorenz_b200 import rl_ops
from gym_lorenz_b200.distributed import summarize
from gym_lorenz_b200.vec_env import BatchedChaosVecEnv


class ActorCritic(torch.nn.Module):
    """SB3 ActorCriticPolicy's parameter names (mlp_extractor.policy_net / value_net, action_net, value_net,
    log_std), so rl_ops.pack_actor_critic reads the module directly."""

    def __init__(self, obs_dim=6, act_dim=2, hidden=64):
        super().__init__()
        mlp = lambda: torch.nn.Sequential(torch.nn.Linear(obs_dim, hidden), torch.nn.Tanh(),
                                          torch.nn.Linear(hidden, hidden), torch.nn.Tanh())
        self.mlp_extractor = torch.nn.Module()
        self.mlp_extractor.policy_net, self.mlp_extractor.value_net = mlp(), mlp()
        self.action_net, self.value_net = torch.nn.Linear(hidden, act_dim), torch.nn.Linear(hidden, 1)
        self.log_std = torch.nn.Parameter(torch.full((act_dim,), -0.5))

    def pi(self, obs):
        return self.action_net(self.mlp_extractor.policy_net(obs))

    def v(self, obs):
        return self.value_net(self.mlp_extractor.value_net(obs)).squeeze(-1)

    def dist(self, obs):
        return torch.distributions.Normal(self.pi(obs), self.log_std.exp())

    def forward(self, obs):                       # collector interface: actions, values, log_probs
        mu, std = self.pi(obs), self.log_std.exp()
        a = mu + std * torch.randn_like(mu)
        logp = (-0.5 * ((a - mu) / std) ** 2 - self.log_std - 0.9189385).sum(-1)
        return a, self.v(obs), logp


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--n-steps", type=int, default=128)
    ap.add_argument("--updates", type=int, default=30)
    ap.add_argument("--epochs", type=int, default=4)
    ap.add_argument("--minibatches", type=int, default=8)
    ap.add_argument("--fused", action="store_true", help="collect with FusedRolloutCollector (one launch per rollout)")
    ap.add_argument("--normalize", action="store_true",
                    help="VecNormalize(norm_reward=False) in training mode around the env")
    args = ap.parse_args()
    torch.manual_seed(0)
    env = BatchedChaosVecEnv("hr_sync", args.envs, seed=0, max_episode_steps=1000)
    pol = ActorCritic().to("cuda:0")
    opt = torch.optim.Adam(pol.parameters(), lr=3e-4)
    vn = rl_ops.DeviceVecNormalize(env, training=True, norm_reward=False) if args.normalize else None
    if args.fused:
        col = rl_ops.FusedRolloutCollector(env, pol, n_steps=args.n_steps, gamma=0.99, gae_lambda=0.95,
                                           normalize=vn, update_normalize=vn is not None)
    else:
        col = rl_ops.DeviceRolloutCollector(vn if vn is not None else env, pol, n_steps=args.n_steps, gamma=0.99,
                                            gae_lambda=0.95, use_cuda_graph=True)
    t0, steps = time.time(), 0
    for it in range(args.updates):
        with torch.no_grad():
            ro = col.collect()
        steps += args.envs * args.n_steps
        obs = ro["obs"].reshape(-1, 6); act = ro["actions"].reshape(-1, 2)
        adv = ro["advantages"].reshape(-1); ret = ro["returns"].reshape(-1); old = ro["log_probs"].reshape(-1)
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
        n = obs.shape[0]
        for _ in range(args.epochs):
            perm = torch.randperm(n, device=obs.device)
            for mb in perm.chunk(args.minibatches):
                d = pol.dist(obs[mb])
                logp = d.log_prob(act[mb]).sum(-1)
                ratio = (logp - old[mb]).exp()
                pg = -torch.min(ratio * adv[mb], ratio.clamp(0.8, 1.2) * adv[mb]).mean()
                vloss = 0.5 * (pol.v(obs[mb]) - ret[mb]).pow(2).mean()
                loss = pg + 0.5 * vloss
                opt.zero_grad(set_to_none=True); loss.backward()
                torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.5); opt.step()
        if args.fused:
            col.sync_params()
        st = summarize(env.batch.stats_tensor(clear=True).cpu())
        print(f"update {it + 1:3d}  env-steps {steps:>10d}  step-reward mean {ro['rewards'].mean().item():9.4f}  "
              f"episodes {int(st['episodes']):6d}  ep_rew_mean {st['ep_rew_mean']:10.2f}  ep_len_mean {st['ep_len_mean']:7.1f}  "
              f"terminated {int(st['terminated']):5d}  {steps / (time.time() - t0):.3g} steps/s", flush=True)
    env.close()


if __name__ == "__main__":
    main()
