"""gymnasium.vector.VectorEnv-shaped adapters over the batched black-box env (SURVEY.md §8f rank 4) and over the batched
step-based env.

RL libraries drive vector envs through  reset(seed=, options=) -> (obs[N, O], infos)  and
step(actions[N, P]) -> (obs, rewards, terminations, truncations, infos)  on numpy arrays, with finished
sub-envs reset automatically (gymnasium <= 0.29 semantics: the returned observation of a finished sub-env is the first
one of its NEXT episode and the last one of the finished episode goes to infos["final_observation"]).  A black-box
step is a whole episode, so every sub-env finishes on every step and the auto-reset is one extra fg_reset launch.  A step-based
step is one control step (fg_env_step); only the sub-envs that finished on it are reset, in one masked fg_reset launch.

gymnasium itself is not a dependency; the attribute names follow its VectorEnv (num_envs, single_action_space,
single_observation_space, action_space, observation_space, closed).
"""
from __future__ import annotations

from typing import Any, Dict, Optional

import numpy as np
import torch

from .utils.gym_compat import Box, make, registry


class BlackBoxVectorEnv:
    def __init__(self, env_id: str, num_envs: int, device="cuda:0", tensors: bool = False, **make_kwargs):
        """tensors=True keeps everything on the device (torch tensors in, torch tensors out: no host round trip)."""
        self.env = make(env_id, num_envs=num_envs, device=device, **make_kwargs)
        if self.env.do_replanning or self.env.learn_sub_trajectories:
            raise NotImplementedError("BlackBoxVectorEnv auto-resets after every black-box step; replanning / "
                                      "sub-trajectory envs keep one clock per batch and are driven through reset()/step()")
        self.num_envs = int(num_envs)
        self.tensors = bool(tensors)
        self.single_action_space = Box(self.env.action_space.low, self.env.action_space.high, dtype=self.env.action_space.dtype)
        self.single_observation_space = Box(self.env.observation_space.low, self.env.observation_space.high,
                                            dtype=self.env.observation_space.dtype)
        self.action_space = Box(self.single_action_space.low, self.single_action_space.high,
                                dtype=self.single_action_space.dtype, batch=self.num_envs)
        self.observation_space = Box(self.single_observation_space.low, self.single_observation_space.high,
                                     dtype=self.single_observation_space.dtype, batch=self.num_envs)
        self.closed = False
        self.spec = self.env.spec

    def _out(self, x):
        return x if self.tensors or not torch.is_tensor(x) else x.cpu().numpy()

    def reset(self, *, seed: Optional[int] = None, options: Optional[Dict[str, Any]] = None):
        opts = dict(options or {})
        opts["as_numpy"] = False
        obs, info = self.env.reset(seed=seed, options=opts)
        return self._out(obs if self.num_envs > 1 or obs.dim() == 2 else obs[None]), info

    def step(self, actions):
        a = actions if torch.is_tensor(actions) else torch.as_tensor(np.asarray(actions))
        if a.dim() == 1:
            a = a[None]
        obs, ret, terminated, truncated, infos = self.env.step(a.to(self.env.device))
        done = terminated | truncated
        infos = dict(infos)
        infos["final_observation"] = obs
        infos["_final_observation"] = done
        next_obs = self.env.reset_done()           # every finished sub-env starts its next episode (its own context stream)
        return (self._out(next_obs), self._out(ret), self._out(terminated), self._out(truncated),
                {k: self._out(v) for k, v in infos.items()})

    def close(self):
        if not self.closed:
            self.env.close()
            self.closed = True


class StepVectorEnv:
    """The same adapter over a step-based env (`fancy/HoleReacher-v0`, ...): one step() is one control step of every
    sub-env (fg_env_step).  Sub-envs that terminated or were truncated on a step are reset in one masked fg_reset launch,
    each continuing its own context stream; their returned observation is the first one of the next episode and the last
    one of the finished episode goes to infos["final_observation"] (gymnasium <= 0.29 auto-reset)."""

    def __init__(self, env_id: str, num_envs: int, device="cuda:0", tensors: bool = False, **make_kwargs):
        """tensors=True keeps everything on the device (torch tensors in, torch tensors out: no host round trip)."""
        self.env = make(env_id, num_envs=num_envs, device=device, **make_kwargs)
        if getattr(self.env, "context_sampler", None) != "device":
            raise NotImplementedError("StepVectorEnv auto-resets through the device-side sampler (context_sampler='device')")
        self.num_envs = int(num_envs)
        self.tensors = bool(tensors)
        self.single_action_space = Box(self.env.action_space.low, self.env.action_space.high, dtype=self.env.action_space.dtype)
        self.single_observation_space = Box(self.env.observation_space.low, self.env.observation_space.high,
                                            dtype=self.env.observation_space.dtype)
        self.action_space = Box(self.single_action_space.low, self.single_action_space.high,
                                dtype=self.single_action_space.dtype, batch=self.num_envs)
        self.observation_space = Box(self.single_observation_space.low, self.single_observation_space.high,
                                     dtype=self.single_observation_space.dtype, batch=self.num_envs)
        self.closed = False
        self.spec = self.env.spec

    def _out(self, x):
        return x if self.tensors or not torch.is_tensor(x) else x.cpu().numpy()

    def reset(self, *, seed: Optional[int] = None, options: Optional[Dict[str, Any]] = None):
        obs, info = self.env.reset(seed=seed, options=options)
        return self._out(obs), info

    def step(self, actions):
        """actions [num_envs, n_links], float32 or float64 (numpy or torch) -> (obs, rewards, terminations, truncations,
        infos)"""
        a = actions if torch.is_tensor(actions) else torch.as_tensor(np.ascontiguousarray(actions))
        if a.dim() == 1:
            a = a[None]
        obs, rew, terminated, truncated, infos = self.env.step(a)
        infos = dict(infos)
        infos["final_observation"] = obs
        infos["_final_observation"] = terminated | truncated
        # the kernel has set done = terminated | truncated: exactly the envs to reset, the others keep their rows
        next_obs = obs.clone()
        self.env.device_reset(None, out=next_obs, mask=self.env.done)
        return (self._out(next_obs), self._out(rew), self._out(terminated), self._out(truncated),
                {k: self._out(v) for k, v in infos.items()})

    def close(self):
        if not self.closed:
            self.env.close()
            self.closed = True


def make_vec(env_id: str, num_envs: int, **kwargs):
    """BlackBoxVectorEnv for a black-box id (`fancy_ProMP/HoleReacher-v0`), StepVectorEnv for a step-based one
    (`fancy/HoleReacher-v0`)."""
    from .envs.registry import bb_env_constructor
    spec = registry.get(env_id)
    if spec is not None and spec.entry_point is not bb_env_constructor:
        return StepVectorEnv(env_id, num_envs, **kwargs)
    return BlackBoxVectorEnv(env_id, num_envs, **kwargs)
