"""Step-based use: a random-action loop over 4096 HoleReacher envs, one control step per call (what PPO / SAC do).

    python examples/step_based.py

make_vec on a step-based id keeps everything on the device with tensors=True; sub-envs that terminate (collision) or are
truncated (200 steps) start their next episode automatically, and their last observation is in infos["final_observation"].
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import fancy_gym_b200 as fancy_gym  # noqa: E402

N = 4096
vec = fancy_gym.make_vec("fancy/HoleReacher-v0", N, device="cuda:0", tensors=True)
obs, _ = vec.reset(seed=0)
gen = torch.Generator(device="cuda:0").manual_seed(0)
episodes = torch.zeros((), dtype=torch.int64, device="cuda:0")
returns = torch.zeros(N, dtype=torch.float64, device="cuda:0")
finished_return = torch.zeros((), dtype=torch.float64, device="cuda:0")
for t in range(1000):
    action = 0.5 * torch.randn(N, 5, generator=gen, device="cuda:0")      # float32 joint velocities
    obs, reward, terminated, truncated, infos = vec.step(action)
    returns += reward
    done = infos["_final_observation"]
    episodes += done.sum()
    finished_return += torch.where(done, returns, 0.0).sum()
    returns = torch.where(done, 0.0, returns)
n = int(episodes)
print(f"{N * 1000} env steps, {n} finished episodes, mean return {float(finished_return) / max(n, 1):.3f}")
vec.close()
