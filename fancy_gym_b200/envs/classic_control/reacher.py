"""Batched step-env state holders for the classic_control reachers.

The dynamics themselves run on the device: inside the fused rollout kernel for the black-box ids
(fancy_gym_b200/csrc/fg_rollout.cuh), one control step per step() call for the step-based ids
(fancy_gym_b200/csrc/fg_env_step.cu).  These classes own the per-env device state (joint angles /
velocities / step counters / task context), the spaces, the constructor kwargs of the reference envs
and the reset-time context sampling:
  HoleReacherEnv      fancy_gym/envs/classic_control/hole_reacher/hole_reacher.py
  ViaPointReacherEnv  fancy_gym/envs/classic_control/viapoint_reacher/viapoint_reacher.py
  SimpleReacherEnv    fancy_gym/envs/classic_control/simple_reacher/simple_reacher.py
  (base: base_reacher/base_reacher.py, base_reacher_direct.py, base_reacher_torque.py)

reset(seed=s) seeds env i with s + i (gymnasium's vector-env convention); env i then is the reference
env reset with seed s + i: its context comes from Generator(PCG64(SeedSequence(seed_i))) in the
reference's draw order.  context_sampler='device' (default) runs that sampler as ONE CUDA kernel
(fg_reset: PCG64 / SeedSequence restated in integer arithmetic, per-env stream state kept in HBM for
unseeded resets); context_sampler='numpy' is the same sampling done with numpy on the host (a cross-check
for tests, O(num_envs) Python).
"""
from __future__ import annotations

from typing import Any, Dict, Iterable, Optional, Union

import numpy as np
import torch

from ... import _lib
from ...utils.gym_compat import Box, Env


def _np_rng(seed):
    return np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed)))


class BaseReacherEnv(Env):
    env_kind = -1
    torque = False
    n_ctx_obs = 0            # task-specific obs entries between velocity and step counter

    def __init__(self, n_links: int, random_start: bool = True, allow_self_collision: bool = False,
                 num_envs: int = 1, device: Union[str, torch.device, None] = None, context_sampler: str = "device",
                 render_mode: Optional[str] = None, **kwargs):
        if kwargs:
            raise TypeError(f"unexpected keyword arguments {sorted(kwargs)}")
        if not 1 <= n_links <= _lib.FG_MAX_DOF:
            raise ValueError(f"n_links must be in 1..{_lib.FG_MAX_DOF}")
        if context_sampler not in ("numpy", "device"):
            raise ValueError("context_sampler must be 'numpy' or 'device'")
        self.n_links = int(n_links)
        self.num_envs = int(num_envs)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.random_start = random_start
        self.allow_self_collision = allow_self_collision
        self.context_sampler = context_sampler
        self.render_mode = render_mode
        self._dt = 0.01                                   # base_reacher.py:21
        self._start_pos = np.hstack([[np.pi / 2], np.zeros(self.n_links - 1)])   # base_reacher.py:34
        bound = 1000.0 if self.torque else 2 * np.pi      # base_reacher_torque.py:16 / base_reacher_direct.py:16
        ab = np.ones(self.n_links) * bound
        self.action_space = Box(low=-ab, high=ab, shape=ab.shape, batch=self._batch_or_none())
        self.observation_space = self._make_observation_space()
        B, n = self.num_envs, self.n_links
        dev = self.device
        self.q = torch.zeros(B, n, dtype=torch.float64, device=dev)
        self.v = torch.zeros(B, n, dtype=torch.float64, device=dev)
        self.steps = torch.zeros(B, dtype=torch.int32, device=dev)
        self.done = torch.zeros(B, dtype=torch.uint8, device=dev)
        self.ctx = torch.zeros(B, 4, dtype=torch.float64, device=dev)
        self._seed_rngs = None
        self._rng_state = None            # [B, 5] uint64 PCG64 stream state of the device sampler
        self._was_reset = False
        self._step_sets = None            # output ring of step()
        self._latch = None                # [B, 2] end effector latched by rew_fct "unbounded" (step())
        self._last_action_dtype = None    # dtype of the last step() action since the last full reset

    def _batch_or_none(self):
        return self.num_envs if self.num_envs > 1 else None

    # ---- spaces --------------------------------------------------------------------------------
    def _state_bound(self):
        n = self.n_links
        return np.hstack([[np.pi] * n, [np.pi] * n, [np.inf] * n, [np.inf] * self.n_ctx_obs, [np.inf]])

    def _make_observation_space(self):
        sb = self._state_bound()
        return Box(low=-sb, high=sb, shape=sb.shape, batch=self._batch_or_none())

    # ---- properties the MP wrappers expose (raw_interface_wrapper.py:24-53) ----------------------
    @property
    def dt(self):
        return self._dt

    @property
    def current_pos(self):
        return self.q.clone()

    @property
    def current_vel(self):
        return self.v.clone()

    # ---- reset ---------------------------------------------------------------------------------
    def _seeds(self, seed):
        B = self.num_envs
        if seed is None:
            if self._seed_rngs is None:
                ss = np.random.SeedSequence()
                self._seed_rngs = [np.random.Generator(np.random.PCG64(s)) for s in ss.spawn(B)]
            return None
        seeds = np.asarray(seed).reshape(-1)
        if seeds.size == 1:
            seeds = int(seeds[0]) + np.arange(B)
        if seeds.size != B:
            raise ValueError(f"need one seed or {B} seeds")
        self._seed_rngs = None
        return [int(s) for s in seeds]

    def _sample_numpy(self, seeds) -> Dict[str, np.ndarray]:
        raise NotImplementedError

    def reset(self, *, seed=None, options: Optional[Dict[str, Any]] = None):
        """-> (obs [B, O] float32 tensor on the device, {}).  options['contexts'] (dict of arrays)
        bypasses sampling; options['random_start'] as in base_reacher.py:77-80."""
        options = options or {}
        B, n, dev = self.num_envs, self.n_links, self.device
        random_start = options.get("random_start", self.random_start)
        if "contexts" in options:
            c = {k: torch.as_tensor(np.asarray(v), dtype=torch.float64) for k, v in options["contexts"].items()}
        elif self.context_sampler == "numpy":
            seeds = self._seeds(seed)
            if seeds is None:
                rngs = self._seed_rngs
            else:
                rngs = [_np_rng(s) for s in seeds]
                self._seed_rngs = rngs
            c = {k: torch.as_tensor(v, dtype=torch.float64) for k, v in self._sample_numpy(rngs, seeds, random_start).items()}
        else:
            return self.device_reset(seed, random_start=random_start), {}
        q0 = c.pop("q0").to(dev)
        self.q.zero_()
        self.q[:, 0] = q0
        self.v.zero_()
        self.steps.zero_()
        self.done.zero_()
        self._set_ctx({k: v.to(dev) for k, v in c.items()})
        self._was_reset = True
        self._last_action_dtype = None
        return self.get_obs(), {}

    def _set_ctx(self, c):
        raise NotImplementedError

    def _fixed_context(self):
        """(values[4], given[4]) of the constructor-fixed task context, laid out like `ctx`"""
        return [0.0] * 4, [0] * 4

    def device_reset(self, seed=None, obs_index=None, time_aware=False, random_start=None, out=None, mask=None, state=None):
        """fg_reset: one kernel samples the contexts (numpy-exact streams), resets the state buffers and writes the
        observation columns `obs_index` of the reset state (default: the full step observation).
        `state`: object with q / v / steps / done / ctx device tensors that receive the reset state instead of the env's own
        (several episode batches in flight, each with its own state: EpisodePipeline); the context streams advance all the same."""
        import ctypes as C
        B, n, dev = self.num_envs, self.n_links, self.device
        n_full = self.observation_space.shape[0] + (1 if time_aware else 0)
        idx = list(range(n_full)) if obs_index is None else [int(i) for i in obs_index]
        cfg = _lib.FgResetCfg()
        cfg.struct_size = C.sizeof(_lib.FgResetCfg)
        cfg.env_kind, cfg.n_dof = self.env_kind, n
        cfg.random_start = int(bool(self.random_start if random_start is None else random_start))
        cfg.time_aware = int(bool(time_aware))
        cfg.device = dev.index or 0
        vals, given = self._fixed_context()
        for i in range(4):
            cfg.fixed[i], cfg.has_fixed[i] = float(vals[i]), int(given[i])
        cfg.n_obs_out = len(idx)
        for j, i in enumerate(idx):
            cfg.obs_index[j] = i
        io = _lib.FgResetIO()
        io.struct_size = C.sizeof(_lib.FgResetIO)
        seeds_dev = None
        if seed is None and self._rng_state is not None:
            io.reseed = 0
        else:
            io.reseed = 1
            if seed is None:       # first unseeded reset: OS entropy, like np_random(None)
                io.seed0 = int(np.random.SeedSequence().entropy % (2 ** 62))
            else:
                seeds = np.asarray(seed).reshape(-1)
                if seeds.size == 1:
                    io.seed0 = int(seeds[0])
                elif seeds.size == B:
                    seeds_dev = torch.as_tensor(seeds.astype(np.int64), device=dev)
                    io.seeds = seeds_dev.data_ptr()
                else:
                    raise ValueError(f"need one seed or {B} seeds")
            if self._rng_state is None:
                self._rng_state = torch.zeros(B, 5, dtype=torch.int64, device=dev)
        io.rng_state = self._rng_state.data_ptr()
        if mask is not None:       # partial reset: only envs with mask != 0 (their rows of `out` are rewritten, the rest kept)
            mask = mask.to(dev, torch.uint8).contiguous()
            io.mask = mask.data_ptr()
        st = self if state is None else state
        io.q, io.v, io.steps, io.done, io.ctx = (st.q.data_ptr(), st.v.data_ptr(), st.steps.data_ptr(),
                                                 st.done.data_ptr(), st.ctx.data_ptr())
        obs = out if out is not None else torch.empty(B, len(idx), dtype=torch.float32, device=dev)
        io.obs = obs.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.lib.fg_reset(C.byref(cfg), C.byref(io), B, C.c_void_p(stream)))
        self._was_reset = True
        if mask is None and state is None:
            self._last_action_dtype = None
        return obs

    # ---- step: one control step of every env (the step-based ids) --------------------------------
    def _next_step_set(self):
        """output buffers of the next step() from a ring of two: what a call returns stays valid while the next one runs"""
        if self._step_sets is None:
            B, n, dev = self.num_envs, self.n_links, self.device
            self._step_sets = [dict(obs=torch.zeros(B, self.observation_space.shape[0], dtype=torch.float32, device=dev),
                                    reward=torch.zeros(B, dtype=torch.float64, device=dev),
                                    flags=torch.zeros(4, B, dtype=torch.bool, device=dev),
                                    info=torch.zeros(B, 2, dtype=torch.float64, device=dev),
                                    joints=torch.zeros(B, n, dtype=torch.float64, device=dev)) for _ in range(2)]
            if getattr(self, "rew_fct", None) == "unbounded":
                self._latch = torch.zeros(B, 2, dtype=torch.float64, device=dev)
        self._step_sets.reverse()
        return self._step_sets[0]

    def step(self, action):
        """base_reacher_direct.py:20-38 / base_reacher_torque.py:20-37 with the env's reward, for every env in ONE kernel
        launch (fg_env_step), plus gymnasium's TimeLimit (max_episode_steps of the registration; a directly constructed env
        never truncates).  action [B, n_links] (or [n_links] when num_envs == 1), torch tensor or numpy array, float32 or
        float64 — the arithmetic follows the dtype as in the reference, and no clip is applied.
        -> (obs [B, O] float32, reward [B] float64, terminated [B] bool, truncated [B] bool, infos), device tensors that
        stay valid until the step after the next.  Envs that terminated or were truncated keep being stepped until they
        are reset.  No device -> host copy and no synchronisation: the call can be captured in a CUDA graph."""
        import ctypes as C
        if not self._was_reset:
            raise RuntimeError("Cannot call env.step() before calling env.reset()")
        _lib.check_step_links(self.env_kind, self.n_links)
        a = action if torch.is_tensor(action) else torch.as_tensor(np.ascontiguousarray(action))
        if a.dtype not in (torch.float32, torch.float64):
            raise TypeError(f"action dtype must be float32 or float64, got {a.dtype}")
        B, n, dev = self.num_envs, self.n_links, self.device
        if a.dim() == 1 and B == 1:
            a = a[None]
        if tuple(a.shape) != (B, n):
            raise ValueError(f"expected an action of shape [{B}, {n}]" + (f" or [{n}]" if B == 1 else "") +
                             f", got {tuple(a.shape)}")
        a = a.to(dev, non_blocking=True).contiguous()
        f64 = a.dtype == torch.float64
        out = self._next_step_set()
        cfg = _lib.FgEnvStepCfg()
        cfg.struct_size = C.sizeof(_lib.FgEnvStepCfg)
        cfg.env_kind, cfg.n_dof = self.env_kind, n
        spec = getattr(self, "spec", None)
        cfg.max_episode_steps = int(spec.max_episode_steps or 0) if spec is not None else 0
        cfg.dt = float(self._dt)
        cfg.allow_self_collision = int(bool(self.allow_self_collision))
        cfg.allow_wall_collision = int(bool(getattr(self, "allow_wall_collision", False)))
        cfg.collision_penalty = float(getattr(self, "collision_penalty", 0.0))
        cfg.rew_fct = int(getattr(self, "rew_fct_code", 0))
        cfg.action_f64 = int(f64)
        io = _lib.FgEnvStepIO()
        io.struct_size = C.sizeof(_lib.FgEnvStepIO)
        io.action = a.data_ptr()
        # every env that has stepped since the last reset holds the previous float32 action in v (envs at step 0 hold the
        # float64 zeros of the reset; the kernel tells them apart by their step counter)
        io.v_is_f32 = int(not f64 and self._last_action_dtype in (None, torch.float32))
        io.q, io.v, io.steps, io.done, io.ctx = (self.q.data_ptr(), self.v.data_ptr(), self.steps.data_ptr(),
                                                 self.done.data_ptr(), self.ctx.data_ptr())
        if self._latch is not None:
            io.latch = self._latch.data_ptr()
        io.obs, io.reward, io.flag_bytes, io.info = (out["obs"].data_ptr(), out["reward"].data_ptr(),
                                                     out["flags"].data_ptr(), out["info"].data_ptr())
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(_lib.lib.fg_env_step(C.byref(cfg), C.byref(io), B, C.c_void_p(stream)))
        self._last_action_dtype = a.dtype
        terminated, truncated, success, collided = out["flags"]
        infos: Dict[str, Any] = {}
        if self.torque:
            infos["reward_dist"], infos["reward_ctrl"] = out["info"][:, 0], out["info"][:, 1]
        else:
            infos["is_success"], infos["is_collided"] = success, collided
            infos["end_effector"] = out["info"]
            if self._latch is not None:          # hr_unbounded_reward.py:53-56
                infos["joints"] = out["joints"].copy_(self.q)
        return out["obs"], out["reward"], terminated, truncated, infos

    def _first_joint(self, rng, random_start):
        # base_reacher.py:81-86 (random start angle of the first joint, the arm is straight)
        return rng.uniform(np.pi / 4, 3 * np.pi / 4) if random_start else self._start_pos[0]

    # ---- observation of the current state (reset-time; per-step observations come from the kernel)
    def end_effector(self):
        th = torch.cumsum(self.q, dim=1)
        return torch.stack([torch.cos(th).sum(1), torch.sin(th).sum(1)], dim=1)

    def _task_obs(self, ee):
        raise NotImplementedError

    def get_obs(self):
        ee = self.end_effector()
        parts = [torch.cos(self.q), torch.sin(self.q), self.v, *self._task_obs(ee), self.steps.to(torch.float64)[:, None]]
        return torch.cat(parts, dim=1).to(torch.float32)

    def close(self):
        pass


class HoleReacherEnv(BaseReacherEnv):
    env_kind = _lib.ENV_HOLE_REACHER
    n_ctx_obs = 3    # hole width, ee - goal (2)

    def __init__(self, n_links: int, hole_x: Union[None, float] = None, hole_depth: Union[None, float] = None,
                 hole_width: float = 1., random_start: bool = False, allow_self_collision: bool = False,
                 allow_wall_collision: bool = False, collision_penalty: float = 1000, rew_fct: str = "simple", **kwargs):
        if rew_fct not in ("simple", "vel_acc", "unbounded"):
            raise ValueError("Unknown reward function {}".format(rew_fct))      # hole_reacher.py:57-58
        self.initial_x, self.initial_width, self.initial_depth = hole_x, hole_width, hole_depth
        self.allow_wall_collision = allow_wall_collision
        self.collision_penalty = collision_penalty
        self.rew_fct = rew_fct
        self.rew_fct_code = ("simple", "vel_acc", "unbounded").index(rew_fct)     # fg_config.rew_fct
        super().__init__(n_links, random_start, allow_self_collision, **kwargs)

    def _sample_numpy(self, rngs, seeds, random_start):
        # hole_reacher.py:79-112 (_generate_hole) then base_reacher.py:73-93 on the same stream
        B = self.num_envs
        out = {k: np.zeros(B) for k in ("x", "width", "depth", "q0")}
        for i, rng in enumerate(rngs):
            width = rng.uniform(0.15, 0.5) if self.initial_width is None else float(self.initial_width)
            if self.initial_x is None:
                direction = rng.choice([-1, 1])
                x = direction * rng.uniform(width / 2, 3.5)
            else:
                x = float(self.initial_x)
            depth = rng.uniform(1, 1) if self.initial_depth is None else float(self.initial_depth)
            out["x"][i], out["width"][i], out["depth"][i] = x, width, depth
            out["q0"][i] = self._first_joint(rng, random_start)
        return out

    def _fixed_context(self):
        given = [self.initial_x is not None, self.initial_width is not None, self.initial_depth is not None, 0]
        vals = [self.initial_x or 0.0, self.initial_width or 0.0, self.initial_depth or 0.0, 0.0]
        return vals, given

    def _set_ctx(self, c):
        self.ctx.zero_()
        self.ctx[:, 0], self.ctx[:, 1], self.ctx[:, 2] = c["x"], c["width"], c["depth"]

    def _task_obs(self, ee):
        goal = torch.stack([self.ctx[:, 0], -self.ctx[:, 2]], dim=1)      # hole_reacher.py:100
        return [self.ctx[:, 1:2], ee - goal]


class ViaPointReacherEnv(BaseReacherEnv):
    env_kind = _lib.ENV_VIAPOINT_REACHER
    n_ctx_obs = 4    # ee - via (2), ee - goal (2)

    def __init__(self, n_links, random_start: bool = False, via_target: Union[None, Iterable] = None,
                 target: Union[None, Iterable] = None, allow_self_collision=False, collision_penalty=1000, **kwargs):
        self.intitial_target = target
        self.initial_via_target = via_target
        self.collision_penalty = collision_penalty
        super().__init__(n_links, random_start, allow_self_collision, **kwargs)

    def _goal_draws(self, rng):
        total = float(self.n_links)
        if self.initial_via_target is None:      # viapoint_reacher.py:59-64
            via = np.array([total, total])
            while np.linalg.norm(via) >= 0.5 * total:
                via = rng.uniform(low=-0.5 * total, high=0.5 * total, size=2)
        else:
            via = np.array(self.initial_via_target, dtype=np.float64)
        if self.intitial_target is None:         # viapoint_reacher.py:66-72
            goal = np.array([total, total])
            while np.linalg.norm(goal) >= total or np.linalg.norm(goal) <= 0.5 * total:
                goal = rng.uniform(low=-total, high=total, size=2)
        else:
            goal = np.array(self.intitial_target, dtype=np.float64)
        return via, goal

    def _sample_numpy(self, rngs, seeds, random_start):
        # viapoint_reacher.py:45-53: seeded reset (draws the start angle) -> _generate_goal on the same stream
        # -> seeded reset again: start angle = first variate, goal from the variates after it (App. A.6-Q4)
        B = self.num_envs
        out = dict(via=np.zeros((B, 2)), goal=np.zeros((B, 2)), q0=np.zeros(B))
        for i, rng in enumerate(rngs):
            if seeds is None:                          # unseeded: goal, start, goal, start on one running stream
                self._goal_draws(rng)
                self._first_joint(rng, random_start)
                out["via"][i], out["goal"][i] = self._goal_draws(rng)
                out["q0"][i] = self._first_joint(rng, random_start)
                continue
            q0 = self._first_joint(rng, random_start)
            out["via"][i], out["goal"][i] = self._goal_draws(rng)
            out["q0"][i] = q0
            rngs[i] = _np_rng(seeds[i])                # the second seeded reset restarts the stream
            self._first_joint(rngs[i], random_start)
        return out

    def _fixed_context(self):
        via, tgt = self.initial_via_target, self.intitial_target
        given = [via is not None] * 2 + [tgt is not None] * 2
        vals = list(np.asarray(via if via is not None else (0, 0), dtype=np.float64)) + \
            list(np.asarray(tgt if tgt is not None else (0, 0), dtype=np.float64))
        return vals, given

    def _set_ctx(self, c):
        self.ctx[:, 0:2] = c["via"]
        self.ctx[:, 2:4] = c["goal"]

    def _task_obs(self, ee):
        return [ee - self.ctx[:, 0:2], ee - self.ctx[:, 2:4]]


class SimpleReacherEnv(BaseReacherEnv):
    env_kind = _lib.ENV_SIMPLE_REACHER
    torque = True
    n_ctx_obs = 2    # ee - goal

    def __init__(self, n_links: int, target: Union[None, Iterable] = None, random_start: bool = True,
                 allow_self_collision: bool = False, **kwargs):
        self.inital_target = target
        super().__init__(n_links, random_start, allow_self_collision, **kwargs)
        self._start_pos = np.zeros(self.n_links)       # simple_reacher.py:29

    def _goal_draw(self, rng):
        if self.inital_target is None:                  # simple_reacher.py:87-94
            total = float(self.n_links)
            goal = np.array([total, total])
            while np.linalg.norm(goal) >= total:
                goal = rng.uniform(low=-total, high=total, size=2)
            return goal
        return np.array(self.inital_target, dtype=np.float64)

    def _sample_numpy(self, rngs, seeds, random_start):
        B = self.num_envs
        out = dict(goal=np.zeros((B, 2)), q0=np.zeros(B))
        for i, rng in enumerate(rngs):
            if seeds is None:
                self._goal_draw(rng)
                self._first_joint(rng, random_start)
                out["goal"][i] = self._goal_draw(rng)
                out["q0"][i] = self._first_joint(rng, random_start)
                continue
            q0 = self._first_joint(rng, random_start)
            out["goal"][i] = self._goal_draw(rng)
            out["q0"][i] = q0
            rngs[i] = _np_rng(seeds[i])
            self._first_joint(rngs[i], random_start)
        return out

    def _fixed_context(self):
        tgt = self.inital_target
        vals = list(np.asarray(tgt if tgt is not None else (0, 0), dtype=np.float64)) + [0.0, 0.0]
        return vals, [tgt is not None] * 2 + [0, 0]

    def _set_ctx(self, c):
        self.ctx.zero_()
        self.ctx[:, 0:2] = c["goal"]

    def _task_obs(self, ee):
        return [ee - self.ctx[:, 0:2]]
