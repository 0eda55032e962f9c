"""Batched black-box (episode-based) environment: the vectorised twin of
fancy_gym/black_box/black_box_wrapper.py.

step(params[B, P]) -> (obs[B, O], return[B], terminated[B], truncated[B], infos) runs, for all B
envs, trajectory generation + tracking controller + clip + env dynamics + reward aggregation as
ONE fused CUDA kernel launch (fg_rollout).  The Python side only keeps the bookkeeping of the
reference wrapper (plan counters, replanning schedule, finalised tau/delay, condition_on_desired)
and builds / caches the per-plan kernel handle.  There is no CPU fallback.

With num_envs == 1 and a 1-D numpy action the call returns the reference's scalar contract:
(obs[O] ndarray, float, bool, bool, dict).
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Callable, Dict, Optional

import numpy as np
import torch

from .. import _lib
from ..mp import MPInterface
from ..utils.gym_compat import Box, Wrapper
from .controller import BaseController
from .raw_interface_wrapper import RawInterfaceWrapper


def _masked_median(rewards: torch.Tensor, length: torch.Tensor) -> torch.Tensor:
    """np.median over the executed steps of every env, on the device: rewards [B, T] float64, length [B].  Sort with the
    steps past the episode's end pushed to +inf, then average the two middle elements (numpy's definition)."""
    B, T = rewards.shape
    t = torch.arange(T, device=rewards.device)[None, :]
    r = torch.where(t < length[:, None], rewards, torch.full_like(rewards, float("inf")))
    r, _ = torch.sort(r, dim=1)
    L = length.clamp(min=1).to(torch.int64)
    lo, hi = (L - 1) // 2, L // 2
    a, b = r.gather(1, lo[:, None])[:, 0], r.gather(1, hi[:, None])[:, 0]
    med = torch.where(a == b, a, (a + b) / 2)         # (equal -inf / +inf values must not turn into nan)
    return torch.where(length > 0, med, torch.zeros_like(med))


class BlackBoxWrapper(Wrapper):

    def __init__(self,
                 env: RawInterfaceWrapper,
                 trajectory_generator: MPInterface,
                 tracking_controller: BaseController,
                 duration: float,
                 verbose: int = 1,
                 learn_sub_trajectories: bool = False,
                 replanning_schedule: Optional[Callable] = None,
                 reward_aggregation: Callable[[np.ndarray], float] = np.sum,
                 max_planning_times: int = np.inf,
                 condition_on_desired: bool = False,
                 wall_mode: int = 0,
                 result_sets: int = 2,
                 schedule_host_callback: bool = False,
                 max_cached_plans: int = 8):
        super().__init__(env)
        self.duration = duration
        self.learn_sub_trajectories = learn_sub_trajectories
        self.do_replanning = replanning_schedule is not None
        self.replanning_schedule = replanning_schedule or (lambda *x: False)
        self.current_traj_steps = 0

        self.traj_gen = trajectory_generator
        self.tracking_controller = tracking_controller
        self.traj_gen.set_duration(self.duration, self.dt)

        self.tau_bound = [-np.inf, np.inf]
        self.delay_bound = [-np.inf, np.inf]
        if hasattr(self.traj_gen.phase_gn, "tau_bound"):
            self.tau_bound = self.traj_gen.phase_gn.tau_bound
        if hasattr(self.traj_gen.phase_gn, "delay_bound"):
            self.delay_bound = self.traj_gen.phase_gn.delay_bound

        self.reward_aggregation = reward_aggregation
        self.return_context_observation = not (learn_sub_trajectories or self.do_replanning)
        self.traj_gen_action_space = self._get_traj_gen_action_space()
        self.action_space = self._get_action_space()
        self.observation_space = self._get_observation_space()

        self.do_render = False
        self.verbose = verbose
        self.condition_on_desired = condition_on_desired
        self.condition_set = False
        self.max_planning_times = max_planning_times
        self.plan_steps = 0
        self.wall_mode = int(wall_mode)
        # A replanning_schedule that inspects pos / vel / obs / action cannot run inside the fused kernel.  On request it is
        # evaluated on the host from the recorded per-step state of a trial rollout (single env only; see _host_schedule_steps).
        self.schedule_host_callback = bool(schedule_host_callback)
        self._breaks = None
        self.max_cached_plans = int(max_cached_plans)
        self._interface_checked = False
        self._traj_buf = None
        self._fast_reset = self._can_fast_reset()

        # ---- device side ----
        base = self.env.unwrapped
        self._base = base
        self.num_envs = base.num_envs
        self.device = base.device
        self.traj_gen.device = self.device
        B, n = self.num_envs, base.n_links
        dev = self.device
        # A ring of result buffer sets (two by default): what step() returns stays valid until the step after the next
        # one, without a device-side copy per call.
        self._obs_index_np = np.asarray(self._obs_index())
        # (return | length | flags) of a step live in ONE contiguous byte block: the multi-GPU exchange is a single
        # all-gather of that block, with no packing kernels (fancy_gym_b200/dist).
        from ..dist import result_block_bytes, result_block_flag_bytes, result_block_views
        self._out_sets = []
        if int(result_sets) < 2:
            raise ValueError("result_sets must be >= 2 (what step() returns stays valid while the next step runs)")
        for _ in range(int(result_sets)):      # > 2: consumers on other streams (multi-GPU exchange) may lag several steps
            block = torch.zeros(result_block_bytes(B), dtype=torch.uint8, device=dev)
            r, ln, fl = result_block_views(block, B)
            self._out_sets.append(dict(block=block, ret=r, len=ln, flags=fl, flag_bytes=result_block_flag_bytes(block, B),
                                       info=torch.zeros(B, 4, dtype=torch.float64, device=dev),
                                       obs=torch.zeros(B, len(self._obs_index_np), dtype=torch.float32, device=dev)))
        self._out_i = 0
        self._obs_index_dev = None
        self._bind_outputs()
        self._cond_pos = torch.zeros(B, n, dtype=torch.float32, device=dev)
        self._cond_vel = torch.zeros(B, n, dtype=torch.float32, device=dev)
        self._handles: Dict[Any, C.c_void_p] = {}
        self._lo = torch.as_tensor(self.traj_gen_action_space.low, device=dev)
        self._hi = torch.as_tensor(self.traj_gen_action_space.high, device=dev)
        self._has_finite_bounds = bool(np.isfinite(self.traj_gen_action_space.low).any()
                                       or np.isfinite(self.traj_gen_action_space.high).any())

    def _can_fast_reset(self) -> bool:
        """True when reset() of every wrapper between this one and the step env is the plain pass-through (or the
        time-aware column, which fg_reset writes itself) and the env samples on the device"""
        from ..utils.wrappers import TimeAwareObservation
        base = self.env.unwrapped
        if not hasattr(base, "device_reset") or getattr(base, "context_sampler", None) != "device":
            return False
        layer = self.env
        while layer is not base:
            if type(layer).reset is not Wrapper.reset and not isinstance(layer, TimeAwareObservation):
                return False
            layer = layer.env
        return True

    def _bind_outputs(self):
        o = self._out_sets[self._out_i]
        self._ret, self._len, self._flags, self._info, self._obs = o["ret"], o["len"], o["flags"], o["info"], o["obs"]
        self._result_block = o["block"]
        self._flag_bytes = o["flag_bytes"]        # bool views: terminated, truncated, is_success, is_collided

    def _flip_outputs(self):
        """next result set.  Envs whose episode ended in an earlier call are skipped by the kernel, so while several plans
        share one episode (replanning / sub-trajectories) their last observation and infos are carried over; the "unbounded"
        HoleReacher reward keeps per-episode state in info[:, 2:4] (fg_rollout_io.info)."""
        self._prev_info, self._prev_obs = self._info, self._obs
        self._out_i = (self._out_i + 1) % len(self._out_sets)
        self._bind_outputs()
        if getattr(self._base, "rew_fct", None) == "unbounded":
            self._info[:, 2:4] = self._prev_info[:, 2:4]

    # ---- spaces (black_box_wrapper.py:122-148) --------------------------------------------------
    def _get_traj_gen_action_space(self):
        lo, hi = self.traj_gen.get_params_bounds()
        return Box(low=lo.numpy(), high=hi.numpy(), dtype=self.env.action_space.dtype,
                   batch=self.env.unwrapped.num_envs if self.env.unwrapped.num_envs > 1 else None)

    def _get_action_space(self):
        return self.traj_gen_action_space

    def _time_aware(self) -> bool:
        return bool(getattr(self.env, "time_aware", False))

    def _obs_index(self):
        full = self.env.observation_space.shape[0]
        if self.return_context_observation:
            return np.nonzero(np.asarray(self.env.context_mask, dtype=bool))[0]
        return np.arange(full)

    def _get_observation_space(self):
        space = self.env.observation_space
        if self.return_context_observation:
            mask = np.asarray(self.env.context_mask, dtype=bool)
            return Box(low=space.low[mask], high=space.high[mask], dtype=space.dtype, batch=space.batch)
        return space

    def observation(self, observation):
        if self.return_context_observation:
            if self._obs_index_dev is None:
                self._obs_index_dev = torch.as_tensor(self._obs_index_np, device=observation.device)
            observation = observation[..., self._obs_index_dev]
        return observation.to(torch.float32)

    # ---- kernel handle for the current plan -----------------------------------------------------
    def _controller_cfg(self, cfg):
        ctrl = self.tracking_controller
        code = getattr(ctrl, "abi_code", None)
        if code is None:
            raise NotImplementedError(f"controller {type(ctrl).__name__} is not available inside the fused kernel")
        cfg.ctrl_kind = code
        p, d = ctrl.gain_vectors(self._base.n_links)
        for i in range(self._base.n_links):
            cfg.p_gains[i], cfg.d_gains[i] = float(p[i]), float(d[i])

    def _handle(self, from_trajectory: bool = False):
        """kernel handle of the current plan; `from_trajectory`: the desired trajectory comes from HBM (FG_MP_TRAJ), used
        when the phase is per env (learned tau / delay) and fg_trajgen_phase has produced it"""
        tg, base = self.traj_gen, self._base
        key = ("traj", tg.n_steps) if from_trajectory else tg.table_key()
        h = self._handles.get(key)
        if h is not None:
            self._handles[key] = self._handles.pop(key)       # most recently used last
            return h
        if from_trajectory:
            from ..mp.mp import MPTables
            tb = MPTables(mp_kind=_lib.MP_TRAJ, n_basis=0, n_steps=tg.n_steps, tab_a=np.zeros(1, np.float32),
                          tab_b=np.zeros(1, np.float32))
        else:
            tb = tg.tables()
        hp = self._create_handle(tb)
        self._remember_handle(key, hp)
        return hp

    def _remember_handle(self, key, hp):
        """bounded cache: a learned scalar tau / delay gives a new table key almost every episode; the least recently used
        handle is destroyed (its launches are stream ordered before the destroy: cudaFree waits)"""
        self._handles[key] = hp
        while len(self._handles) > self.max_cached_plans:
            old_key = next(iter(self._handles))
            _lib.lib.fg_destroy(self._handles.pop(old_key))

    def _create_handle(self, tb):
        base = self._base
        cfg = _lib.FgConfig()
        cfg.struct_size = C.sizeof(_lib.FgConfig)
        cfg.env_kind, cfg.mp_kind = base.env_kind, tb.mp_kind
        self._controller_cfg(cfg)
        cfg.n_dof, cfg.n_steps, cfg.n_basis = base.n_links, tb.n_steps, tb.n_basis
        cfg.max_episode_steps = int(self.env.spec.max_episode_steps)
        cfg.dt = float(self.dt)
        cfg.tau, cfg.dmp_alpha = tb.tau, tb.dmp_alpha
        cfg.weights_scale, cfg.goal_scale, cfg.relative_goal = tb.weights_scale, tb.goal_scale, tb.relative_goal
        cfg.allow_self_collision = int(bool(getattr(base, "allow_self_collision", False)))
        cfg.allow_wall_collision = int(bool(getattr(base, "allow_wall_collision", False)))
        cfg.collision_penalty = float(getattr(base, "collision_penalty", 0.0))
        cfg.rew_fct = int(getattr(base, "rew_fct_code", 0))
        cfg.wall_mode = self.wall_mode
        cfg.time_aware = int(self._time_aware())
        idx = self._obs_index_np
        cfg.n_obs_out = len(idx)
        for j, i in enumerate(idx):
            cfg.obs_index[j] = int(i)
        ta = np.ascontiguousarray(tb.tab_a, dtype=np.float32)
        tbb = np.ascontiguousarray(tb.tab_b, dtype=np.float32)
        cfg.tab_a, cfg.tab_b = ta.ctypes.data, tbb.ctypes.data
        hp = C.c_void_p()
        _lib.check(_lib.lib.fg_create(C.byref(cfg), self.device.index or 0, C.byref(hp)))
        return hp

    # ---- replanning: how many steps does this plan execute? (black_box_wrapper.py:197) -----------
    def _break_points(self):
        """Steps t (1-based, counted over the episode) at which the schedule fires, evaluated ONCE with the step counter
        only — every schedule in the reference and its tests has the form `t % k == 0` (SURVEY.md §3.5).  None if the
        schedule needs the state (it raised on the None arguments)."""
        if self._breaks is None:
            n = int(self.env.spec.max_episode_steps)
            try:
                self._breaks = [t for t in range(1, n + 1) if self.replanning_schedule(None, None, None, None, t)]
            except Exception:      # noqa: BLE001  (whatever the callable does with None: it looks at the state)
                self._breaks = False
        return None if self._breaks is False else self._breaks

    def _segment_steps(self, n_steps: int):
        """(steps this plan executes, whether they end in a re-planning break) — black_box_wrapper.py:197."""
        if not self.do_replanning or not (self.plan_steps < self.max_planning_times):
            return n_steps, False
        breaks = self._break_points()
        if breaks is None:
            if not self.schedule_host_callback:
                raise NotImplementedError("replanning_schedule must depend on the step counter only (it is evaluated on the host, "
                                          "outside the fused kernel); pass black_box_kwargs={'schedule_host_callback': True} to "
                                          "evaluate a state-dependent schedule on the host (single env)")
            return None, True          # decided by _host_schedule_steps from a trial rollout
        import bisect
        i = bisect.bisect_right(breaks, self.current_traj_steps)
        if i < len(breaks) and breaks[i] - self.current_traj_steps <= n_steps:
            return breaks[i] - self.current_traj_steps, True
        return n_steps, False

    def _host_schedule_steps(self, local, T):
        """State-dependent schedule (fallback on request): the plan is rolled out once WITHOUT committing the state
        (keep_state) with the per-step buffers of verbose >= 2 plus the per-step joint state, the schedule is called on the
        host with (pos, vel, obs, action, t) exactly like black_box_wrapper.py:197, and the first firing step bounds the real
        launch.  One env only: in a batch every env would break at its own step and leave the shared plan clock."""
        if self.num_envs != 1:
            raise NotImplementedError("schedule_host_callback is available for num_envs == 1")
        n = self._base.n_links
        dbg = dict(rewards=torch.zeros(1, T, dtype=torch.float64, device=self.device),
                   actions=torch.zeros(1, T, n, dtype=torch.float64, device=self.device),
                   obs=torch.zeros(1, T, self.env.observation_space.shape[0], dtype=torch.float32, device=self.device),
                   state=torch.zeros(1, T, 2 * n, dtype=torch.float64, device=self.device))
        self.launch(local, T, False, dbg, keep_state=True)
        L = int(self._len[0])
        st, ob, ac = dbg["state"][0].cpu().numpy(), dbg["obs"][0].cpu().numpy(), dbg["actions"][0].cpu().numpy()
        self._out_i = (self._out_i - 1) % len(self._out_sets)      # the trial's result set is recycled by the real launch
        self._bind_outputs()
        for t in range(L):
            if self.replanning_schedule(st[t, :n], st[t, n:], ob[t], ac[t], t + 1 + self.current_traj_steps):
                return t + 1, True
        return T, False

    # ---- the hot path ---------------------------------------------------------------------------
    def get_trajectory(self, action):
        """black_box_wrapper.py:96-120 — stand-alone trajectory (fg_trajgen); the fused step does not call this."""
        params = self._prepare_params(action)[0]
        self._set_plan(params)
        if self.condition_set:
            self.traj_gen.set_initial_conditions(self.traj_gen.init_time, self._cond_pos, self._cond_vel)
        return self.traj_gen.get_traj_pos(), self.traj_gen.get_traj_vel()

    def _prepare_params(self, action):
        as_numpy = not torch.is_tensor(action)
        a = torch.as_tensor(np.asarray(action)) if as_numpy else action
        scalar = a.dim() == 1
        if scalar:
            if self.num_envs != 1:
                raise ValueError(f"expected params of shape [{self.num_envs}, {self.action_space.shape[0]}]")
            a = a[None]
        if a.shape != (self.num_envs, self.action_space.shape[0]):
            raise ValueError(f"expected params of shape [{self.num_envs}, {self.action_space.shape[0]}], got {tuple(a.shape)}")
        a = a.to(self.device, torch.float32, non_blocking=True)
        if self._has_finite_bounds:
            a = torch.minimum(torch.maximum(a, self._lo), self._hi)     # np.clip to the tau / delay bounds (:104-105)
        return a.contiguous(), as_numpy, scalar

    def _require_local_state(self):
        """The MP boundary condition is the env's current position / velocity (black_box_wrapper.py:110-111): a wrapper
        stack that does not expose them fails on the first step, like the reference (NotImplementedError from
        RawInterfaceWrapper.current_pos).  Checked once; the kernel reads the state buffers directly."""
        if not self._interface_checked:
            self.env.current_pos, self.env.current_vel   # noqa: B018  (raises if missing)
            self._interface_checked = True

    def _set_plan(self, params):
        self._require_local_state()
        tg = self.traj_gen
        duration = self.duration
        if self.learn_sub_trajectories:
            duration = None
            tg.reset()
        tg.set_params(params)
        init_time = 0 if not self.do_replanning else self.current_traj_steps * self.dt
        tg.set_initial_conditions(init_time, self._base.q, self._base.v)   # current_pos / current_vel (:110-111)
        tg.set_duration(duration, self.dt)

    def launch(self, params, seg_steps=None, replan_break=False, dbg=None, state=None, keep_state=False, trajectory=None,
               seg_steps_env=None):
        """Enqueues ONE fused rollout (fg_rollout) for the current plan on the current CUDA stream and returns
        immediately; results land in the wrapper's device buffers (_ret, _len, _flags, _obs, _info).
        `params` [B, P_local] float32 on the device (phase parameters already stripped).
        `state`: object with q / v / steps / done / ctx device tensors to start from instead of the env's own;
        `keep_state=True` leaves that state untouched (evaluate many parameter sets from one start state)."""
        base = self._base
        B = self.num_envs
        T = self.traj_gen.n_steps
        per_env_phase = not self.traj_gen.phase_gn.uniform()
        fused_phase = per_env_phase and trajectory is None and dbg is None and self._phase_fusable()
        if fused_phase:
            # learned tau / delay differ per env and the shape is one the rollout kernel evaluates itself (fg_rollout_io.phase):
            # the basis row of every step is computed in the thread — no fg_trajgen_phase launch, no trajectory in HBM
            per_env_phase = False
        if trajectory is not None:
            # the desired trajectory comes from the caller (an MPWrapper hook has seen / changed it): tracked from HBM
            self._traj_buf = tuple(x.to(self.device, torch.float32).contiguous() for x in trajectory)
            per_env_phase = True
        elif per_env_phase:
            # learned tau / delay differ per env: fg_trajgen_phase evaluates the basis per env, the fused rollout then
            # tracks that trajectory from HBM (8 KB per env, far below its compute time)
            if self._traj_buf is None or self._traj_buf[0].shape[1] != T:
                n = base.n_links
                self._traj_buf = (torch.empty(B, T, n, dtype=torch.float32, device=self.device),
                                  torch.empty(B, T, n, dtype=torch.float32, device=self.device))
            self._planned_trajectory(params, out=self._traj_buf)
        h = self._handle(from_trajectory=per_env_phase)
        self._flip_outputs()
        io = _lib.FgRolloutIO()
        io.struct_size = C.sizeof(_lib.FgRolloutIO)
        io.params = params.data_ptr()
        if per_env_phase:
            io.traj_pos, io.traj_vel = self._traj_buf[0].data_ptr(), self._traj_buf[1].data_ptr()
        st = base if state is None else state
        io.ctx = st.ctx.data_ptr()
        io.q, io.v, io.steps, io.done = st.q.data_ptr(), st.v.data_ptr(), st.steps.data_ptr(), st.done.data_ptr()
        io.keep_state = int(bool(keep_state))
        if fused_phase:
            tg = self.traj_gen
            pb = tg._phase_basis()
            tau_b, delay_b = tg.phase_gn.per_env(B, self.device)
            keep_alive = (pb, tau_b, delay_b, tg.times_dev())
            io.phase = C.addressof(pb)
            io.phase_tau, io.phase_delay, io.phase_times = tau_b.data_ptr(), delay_b.data_ptr(), keep_alive[3].data_ptr()
            if tg.n_steps_env is not None:
                io.seg_steps_env = tg.n_steps_env.data_ptr()
        io.cond_pos, io.cond_vel = self._cond_pos.data_ptr(), self._cond_vel.data_ptr()
        io.use_cond = int(self.condition_set)
        if not per_env_phase:
            # an assumption switch may move the state the plan starts from (mp/assumptions.py: DMP recurrence from t0)
            src = (self._cond_pos, self._cond_vel) if self.condition_set else (st.q.to(torch.float32), st.v.to(torch.float32))
            pre = self.traj_gen.boundary_prestep(params, *src)
            if pre is not None:
                self._cond_pos.copy_(pre[0])
                self._cond_vel.copy_(pre[1])
                io.use_cond = 1
        io.write_cond = (2 if replan_break else 1) if self.condition_on_desired else 0
        io.ret, io.length, io.flags = self._ret.data_ptr(), self._len.data_ptr(), self._flags.data_ptr()
        io.obs, io.info = self._obs.data_ptr(), self._info.data_ptr()
        io.flag_bytes = self._flag_bytes[0].data_ptr()
        if seg_steps_env is not None:
            io.seg_steps_env = seg_steps_env.data_ptr()
        elif per_env_phase and self.traj_gen.n_steps_env is not None:      # ragged sub-trajectories: per-env plan lengths
            io.seg_steps_env = self.traj_gen.n_steps_env.data_ptr()
        if self.do_replanning or self.learn_sub_trajectories:      # frozen envs keep reporting their last observation / infos
            io.prev_obs, io.prev_info = self._prev_obs.data_ptr(), self._prev_info.data_ptr()
        if dbg is not None:
            io.dbg_rewards = dbg["rewards"].data_ptr()
            if "actions" in dbg:
                io.dbg_actions = dbg["actions"].data_ptr()
            if "obs" in dbg:
                io.dbg_obs = dbg["obs"].data_ptr()
            if "state" in dbg:
                io.dbg_state = dbg["state"].data_ptr()
        peer = getattr(self, "_peer_exchange", None)
        if peer is not None:       # multi-GPU: the kernel stores the result rows into every rank's gather buffer (fancy_gym_b200/dist)
            io.peer_bufs, io.n_peers, io.peer_offset = peer.next_launch()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        _lib.check(_lib.lib.fg_rollout(h, C.byref(io), B, int(T if seg_steps is None else seg_steps), C.c_void_p(stream)))

    def evaluate(self, action):
        """step() WITHOUT advancing the episode: the same parameters-in / (obs, return, terminated, truncated, infos)-out
        contract, but the envs stay where they are (fg_rollout keep_state) — a population-based search evaluates
        candidate after candidate from one reset state / context.  Not available while plans are chained (replanning,
        sub-trajectories), where a step's outcome is the next step's start."""
        if self.do_replanning or self.learn_sub_trajectories:
            raise NotImplementedError("evaluate() is defined for envs that plan once per episode")
        self.traj_gen.reset()       # every candidate is a first plan: learned tau / delay apply (they finalize per plan otherwise)
        return self.step(action, _keep_state=True)

    def new_state_set(self):
        """a private copy of the env state buffers (q, v, steps, done, ctx): an episode batch of its own next to the env's
        (`reset_into` / `run_episode`; EpisodePipeline keeps one per batch in flight)"""
        from types import SimpleNamespace
        b = self._base
        return SimpleNamespace(q=b.q.clone(), v=b.v.clone(), steps=b.steps.clone(), done=b.done.clone(), ctx=b.ctx.clone())

    def reset_into(self, state):
        """reset(seed=None) whose state lands in `state` (new_state_set()) instead of the env's own buffers: every env draws the
        next context of its stream exactly as reset() would; returns the reset observation (device tensor)"""
        if not self._fast_reset:
            raise NotImplementedError("reset_into needs the device-side reset (context_sampler='device')")
        self.traj_gen.reset()
        return self._base.device_reset(None, obs_index=self._obs_index_np, time_aware=self._time_aware(), state=state)

    def run_episode(self, action, state):
        """step() for an env that plans once per episode, from `state` (reset_into) instead of the env's own buffers; the env
        itself is left where it is.  Same returns as reset() + step()."""
        if self.do_replanning or self.learn_sub_trajectories:
            raise NotImplementedError("run_episode() is defined for envs that plan once per episode")
        self.traj_gen.reset()
        return self.step(action, _keep_state=True, _state=state)

    def step(self, action, _keep_state: bool = False, _state=None):
        base = self._base
        _lib.check_step_links(base.env_kind, base.n_links)
        params, as_numpy, scalar = self._prepare_params(action)
        self._set_plan(params)
        local = self.traj_gen.params.contiguous()
        T = self.traj_gen.n_steps
        B, n = self.num_envs, base.n_links
        # ---- the env adaptor's trajectory hooks (black_box_wrapper.py:154-172), only when an MPWrapper overrides them ----
        trajectory, valid = None, None
        if self._hooks_overridden():
            pos, vel = self._planned_trajectory(local)
            pos, vel = self.env.set_episode_arguments(params, pos, vel)
            valid, pos, vel = self.env.preprocessing_and_validity_callback(params, pos, vel, self.tau_bound, self.delay_bound)
            trajectory = (pos, vel)
            valid = torch.as_tensor(valid, device=self.device).to(torch.bool).expand(B).contiguous()
            if bool(valid.all()):
                valid = None
        if not _keep_state and (valid is None or bool(valid.any())):
            self.plan_steps += 1           # (the reference returns before counting the plan when the trajectory is invalid)
        seg, replan_break = self._segment_steps(T)
        if seg is None:
            seg, replan_break = self._host_schedule_steps(local, T)
        dbg = None
        need_rewards = self.verbose >= 2 or self.reward_aggregation not in (np.sum, np.mean, sum)
        if need_rewards:
            dbg = dict(rewards=torch.zeros(B, T, dtype=torch.float64, device=self.device))
            if self.verbose >= 2:
                dbg["actions"] = torch.zeros(B, T, n, dtype=torch.float64, device=self.device)
                dbg["obs"] = torch.zeros(B, T, self.env.observation_space.shape[0], dtype=torch.float32, device=self.device)
        planned = (trajectory or self._planned_trajectory(local)) if self.verbose >= 2 else None   # before the state moves on
        seg_env = None
        if valid is not None:      # envs whose trajectory is invalid execute nothing (and report what invalid_traj_callback says)
            seg_env = torch.where(valid, int(seg), 0).to(torch.int32)
            if self.traj_gen.n_steps_env is not None:
                seg_env = torch.minimum(seg_env, self.traj_gen.n_steps_env)
        self.launch(local, seg, replan_break, dbg, state=_state, keep_state=_keep_state, trajectory=trajectory, seg_steps_env=seg_env)
        if self.condition_on_desired and replan_break and not _keep_state:
            # the desired state is recorded on a BREAK only (black_box_wrapper.py:196-201): at a re-planning break every
            # live env breaks at the same step (the kernel wrote its row); a plan that simply runs out records nothing, and
            # rows written by terminated / truncated envs belong to finished episodes
            self.condition_set = True

        if not _keep_state:
            self.current_traj_steps += seg     # live envs all advance by `seg`; finished envs are frozen
        length = self._len
        terminated, truncated, success, collided = self._flag_bytes      # written by the kernel: no unpacking ops
        ret = self._ret
        if self.reward_aggregation is np.mean:
            ret = ret / length.clamp(min=1)
        infos: Dict[str, Any] = {}
        if base.env_kind in (_lib.ENV_HOLE_REACHER, _lib.ENV_VIAPOINT_REACHER):
            infos["is_success"], infos["is_collided"] = success, collided
            infos["end_effector"] = self._info[:, 0:2]
            if getattr(base, "rew_fct", None) == "unbounded":        # hr_unbounded_reward.py:53-56
                infos["joints"] = (base if _state is None else _state).q.clone()
        elif base.env_kind == _lib.ENV_SIMPLE_REACHER:
            infos["reward_dist"] = self._info[:, 0]
            infos["reward_ctrl"] = self._info[:, 1]
        if need_rewards and self.reward_aggregation is np.median:
            ret = _masked_median(dbg["rewards"], length)          # on the device
        elif need_rewards and self.reward_aggregation not in (np.sum, np.mean, sum):
            # an arbitrary callable: per-env host loop over the executed steps (the reference's call, env by env)
            r = dbg["rewards"].cpu().numpy()
            ln = length.cpu().numpy()
            ret = torch.as_tensor(np.array([self.reward_aggregation(r[b, :ln[b]]) if ln[b] else 0.0 for b in range(B)]),
                                  device=self.device)
        if self.verbose >= 2:
            infos["positions"], infos["velocities"] = planned
            infos["step_actions"] = dbg["actions"]
            infos["step_observations"] = dbg["obs"]
            infos["step_rewards"] = dbg["rewards"]
        infos["trajectory_length"] = length
        obs = self._obs
        if valid is not None:
            obs, ret, terminated, truncated, infos = self._merge_invalid(valid, params, trajectory, obs, ret, terminated, truncated, infos)
        return self._format(obs, ret, terminated, truncated, infos, as_numpy, scalar)

    def _phase_fusable(self) -> bool:
        """can the rollout kernel evaluate this generator's per-env phase itself?  (instantiated for the registry's shapes:
        ProMP / DMP, 5 weighted RBFs of 5 or 6 in total with the zero padding in front, 5 or 2 links, velocity / motor control)"""
        import os
        tg, bg = self.traj_gen, self.traj_gen.basis_gn
        return (os.environ.get("FG_PHASE_FUSED", "1") != "0" and not os.environ.get("FG_PHASE_F32")
                and not getattr(tg, "per_env_basis_f32", False)
                and tg.mp_kind in (_lib.MP_PROMP, _lib.MP_DMP) and bg.num_basis == 5 and bg.total_num_basis in (5, 6)
                and bg.first_learnable == bg.total_num_basis - 5 and self._base.n_links in (2, 5)
                and getattr(self.tracking_controller, "abi_code", None) in (_lib.CTRL_VELOCITY, _lib.CTRL_MOTOR)
                and tg.phase_gn.assume["dmp_init_on_first_grid_point"])

    def _hooks_overridden(self) -> bool:
        """does any wrapper between this one and the step env override a trajectory hook of RawInterfaceWrapper?"""
        if getattr(self, "_hooks", None) is None:
            names = ("set_episode_arguments", "preprocessing_and_validity_callback", "invalid_traj_callback")
            layer, found = self.env, False
            while layer is not None and not found:
                found = any(getattr(type(layer), nm, None) not in (None, getattr(RawInterfaceWrapper, nm)) for nm in names)
                layer = getattr(layer, "env", None)
            self._hooks = found
        return self._hooks

    def _merge_invalid(self, valid, params, trajectory, obs, ret, terminated, truncated, infos):
        """envs with an invalid trajectory return the tuple of invalid_traj_callback (black_box_wrapper.py:169-172; called with
        the reference's six arguments) and their episode is marked over when the callback says so"""
        c_obs, c_ret, c_te, c_tr, c_info = self.env.invalid_traj_callback(params, trajectory[0], trajectory[1],
                                                                          self.return_context_observation, self.tau_bound,
                                                                          self.delay_bound)
        dev, B = self.device, self.num_envs
        inv = ~valid

        def bc(x, like):
            x = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x, device=dev).to(like.dtype)
            return x.expand_as(like) if x.dim() <= like.dim() and x.numel() in (1, like[0].numel(), like.numel()) else x

        c_obs = torch.as_tensor(np.asarray(c_obs) if not torch.is_tensor(c_obs) else c_obs, device=dev).to(obs.dtype)
        if c_obs.shape[-1] != obs.shape[-1]:
            c_obs = self.observation(c_obs) if c_obs.shape[-1] == self.env.observation_space.shape[0] else c_obs[..., :1].expand(obs.shape[-1])
        obs = torch.where(inv[:, None], c_obs.expand_as(obs), obs)
        ret = torch.where(inv, bc(c_ret, ret), ret)
        terminated = torch.where(inv, bc(c_te, terminated), terminated)
        truncated = torch.where(inv, bc(c_tr, truncated), truncated)
        self._base.done |= (inv & (terminated | truncated)).to(self._base.done.dtype)
        infos = dict(infos, trajectory_valid=valid)
        for k_, v_ in (c_info or {}).items():
            infos.setdefault(k_, v_)
        return obs, ret, terminated, truncated, infos

    # ---- re-planning inside ONE launch ----------------------------------------------------------------------------
    def plan_schedule(self, n_plans: int):
        """[(first episode step, steps executed)] of the next `n_plans` plans from the current step on, following
        black_box_wrapper.py:197: a plan ends at the next step the schedule fires on (while plan_steps < max_planning_times)
        or runs its full duration"""
        breaks = self._break_points()
        if breaks is None:
            raise NotImplementedError("the plans of a state-dependent replanning_schedule cannot be laid out in advance")
        import bisect
        T = int(round(self.duration / self.dt))
        horizon = int(self.env.spec.max_episode_steps)
        out, s0, done_plans = [], self.current_traj_steps, self.plan_steps
        for j in range(n_plans):
            if s0 >= horizon:
                raise ValueError(f"only {j} plan(s) fit into the rest of the episode ({horizon} steps)")
            seg = T
            if done_plans + j + 1 < self.max_planning_times:
                i = bisect.bisect_right(breaks, s0)
                if i < len(breaks) and breaks[i] - s0 <= T:
                    seg = breaks[i] - s0
            out.append((s0, seg))
            s0 += seg
        return out

    def _plans_fusable(self) -> bool:
        tg = self.traj_gen
        return (self.do_replanning and not self.learn_sub_trajectories and self._break_points() is not None
                and self.verbose < 2 and self.reward_aggregation in (np.sum, np.mean, sum) and tg.phase_gn.num_params == 0
                and tg.phase_gn.assume["dmp_init_on_first_grid_point"] and not self._hooks_overridden())

    def _plans_handle(self, sched):
        """handle whose tables hold the rows of every plan of `sched`, one after the other (fg_rollout_io.n_plans): plan j is
        planned from its own start time init_time = start_j * dt and contributes its first seg_j + 1 rows (the extra one is the
        look-ahead row of ProMP's finite difference)"""
        tg = self.traj_gen
        key = ("plans", tuple(sched), tg.phase_gn.scalar_tau(), tg.phase_gn.scalar_delay())
        h = self._handles.get(key)
        if h is not None:
            self._handles[key] = self._handles.pop(key)
            return h[0], h[1]
        from ..mp.mp import MPTables
        rows_a, rows_b, row0, r = [], [], [], 0
        tb = None
        for s0, seg in sched:
            tg.set_initial_conditions(s0 * self.dt, self._base.q, self._base.v)
            tg.set_duration(self.duration, self.dt)
            tb = tg.tables()
            n = seg + 1
            a = np.zeros((n,) + tb.tab_a.shape[1:], np.float32)
            m = min(n, tb.tab_a.shape[0])
            a[:m] = tb.tab_a[:m]
            b = np.ones((n,) + tb.tab_b.shape[1:], np.float32)
            m = min(n, tb.tab_b.shape[0])
            b[:m] = tb.tab_b[:m]
            rows_a.append(a); rows_b.append(b); row0.append(r)
            r += n
        tab_a, tab_b = np.concatenate(rows_a), np.concatenate(rows_b)
        if tb.mp_kind != _lib.MP_PRODMP:
            tab_b = tab_b[:-1]           # ProMP / DMP: n_steps - 1 increments
        allp = MPTables(mp_kind=tb.mp_kind, n_basis=tb.n_basis, n_steps=r, tab_a=tab_a, tab_b=tab_b, tau=tb.tau,
                        dmp_alpha=tb.dmp_alpha, weights_scale=tb.weights_scale, goal_scale=tb.goal_scale,
                        relative_goal=tb.relative_goal)
        hp = self._create_handle(allp)
        self._remember_handle(key, (hp, row0))
        return hp, row0

    def step_plans(self, actions):
        """`n_plans` consecutive step() calls of a re-planning env as ONE fused launch: actions [B, n_plans, P] ->
        (obs [n_plans, B, O], return [n_plans, B], terminated [n_plans, B], truncated [n_plans, B], infos of [n_plans, B, ...]).
        Row j is exactly what the j-th step(actions[:, j]) would return (black_box_wrapper.py:150-217 called n_plans times:
        the schedule's break points, max_planning_times, condition_on_desired and the per-plan boundary conditions are
        followed inside the kernel); use it when the plans do not depend on the observations in between (open-loop
        sequences, population-based search over plan sequences).  Falls back to a loop over step() where the plans cannot be
        laid out in advance (state-dependent schedule, learned tau / delay, verbose >= 2, trajectory hooks)."""
        _lib.check_step_links(self._base.env_kind, self._base.n_links)
        a = actions if torch.is_tensor(actions) else torch.as_tensor(np.asarray(actions))
        if a.dim() == 2 and self.num_envs == 1:
            a = a[None]
        B, P = self.num_envs, self.action_space.shape[0]
        if a.dim() != 3 or a.shape[0] != B or a.shape[2] != P:
            raise ValueError(f"expected actions of shape [{B}, n_plans, {P}], got {tuple(a.shape)}")
        n_plans = a.shape[1]
        if n_plans > _lib.FG_MAX_PLANS or not self._plans_fusable():
            outs = [self.step(a[:, j].to(self.device)) for j in range(n_plans)]
            keys = outs[0][4].keys()
            return (torch.stack([o[0] for o in outs]), torch.stack([o[1] for o in outs]), torch.stack([o[2] for o in outs]),
                    torch.stack([o[3] for o in outs]), {k_: torch.stack([o[4][k_] for o in outs]) for k_ in keys})
        self._require_local_state()
        base, tg, dev = self._base, self.traj_gen, self.device
        local = tg._prepare_local(a.to(dev, torch.float32).reshape(B * n_plans, P)).reshape(B, n_plans, P).contiguous()
        tg.params = local[:, -1]
        sched = self.plan_schedule(n_plans)
        h, row0 = self._plans_handle(sched)
        n_obs = len(self._obs_index_np)
        from ..dist import result_block_bytes, result_block_flag_bytes, result_block_views
        cache = self.__dict__.setdefault("_plan_out", {})
        sets = cache.get(n_plans)
        if sets is None:
            sets = [dict(blocks=torch.zeros(n_plans, result_block_bytes(B), dtype=torch.uint8, device=dev),
                         ret=torch.zeros(n_plans, B, dtype=torch.float64, device=dev),
                         len=torch.zeros(n_plans, B, dtype=torch.int32, device=dev),
                         flags=torch.zeros(n_plans, B, dtype=torch.uint8, device=dev),
                         fb=torch.zeros(n_plans, 4, B, dtype=torch.bool, device=dev),
                         info=torch.zeros(n_plans, B, 4, dtype=torch.float64, device=dev),
                         obs=torch.zeros(n_plans, B, n_obs, dtype=torch.float32, device=dev)) for _ in range(2)]
            cache[n_plans] = sets
        o = sets[0]
        sets.reverse()                # what this call returns stays valid during the next one
        io = _lib.FgRolloutIO()
        io.struct_size = C.sizeof(_lib.FgRolloutIO)
        io.params = local.data_ptr()
        io.ctx = base.ctx.data_ptr()
        io.q, io.v, io.steps, io.done = base.q.data_ptr(), base.v.data_ptr(), base.steps.data_ptr(), base.done.data_ptr()
        io.cond_pos, io.cond_vel = self._cond_pos.data_ptr(), self._cond_vel.data_ptr()
        io.use_cond = int(self.condition_set)
        last_break = sched[-1][1] < int(round(self.duration / self.dt)) and sched[-1][0] + sched[-1][1] < int(self.env.spec.max_episode_steps)
        io.write_cond = (2 if last_break else 1) if self.condition_on_desired else 0
        io.ret, io.length, io.flags = o["ret"].data_ptr(), o["len"].data_ptr(), o["flags"].data_ptr()
        io.obs, io.info, io.flag_bytes = o["obs"].data_ptr(), o["info"].data_ptr(), o["fb"].data_ptr()
        io.prev_obs, io.prev_info = self._obs.data_ptr(), self._info.data_ptr()
        io.n_plans, io.plan_T = n_plans, int(round(self.duration / self.dt))
        for j, (s0, seg) in enumerate(sched):
            io.plan_seg[j], io.plan_row0[j] = seg, row0[j]
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.lib.fg_rollout(h, C.byref(io), B, int(sched[0][1]), C.c_void_p(stream)))
        self.plan_steps += n_plans
        self.current_traj_steps += sum(seg for _, seg in sched)
        if self.condition_on_desired and (n_plans > 1 or last_break):
            self.condition_set = True
        self._obs, self._info = o["obs"][-1], o["info"][-1]          # what a following step() carries over for frozen envs
        length, ret = o["len"], o["ret"]
        if self.reward_aggregation is np.mean:
            ret = ret / length.clamp(min=1)
        fb = o["fb"]
        infos: Dict[str, Any] = {}
        if base.env_kind in (_lib.ENV_HOLE_REACHER, _lib.ENV_VIAPOINT_REACHER):
            infos["is_success"], infos["is_collided"] = fb[:, 2], fb[:, 3]
            infos["end_effector"] = o["info"][:, :, 0:2]
        elif base.env_kind == _lib.ENV_SIMPLE_REACHER:
            infos["reward_dist"], infos["reward_ctrl"] = o["info"][:, :, 0], o["info"][:, :, 1]
        infos["trajectory_length"] = length
        return o["obs"], ret, fb[:, 0], fb[:, 1], infos

    def _planned_trajectory(self, local_params, out=None):
        tg = self.traj_gen
        saved = tg.params
        tg.params = local_params
        if self.condition_set:
            tg.set_initial_conditions(tg.init_time, self._cond_pos, self._cond_vel)
        pos, vel = tg._run_trajgen(out=out)
        tg.params = saved
        return pos, vel

    def _format(self, obs, ret, terminated, truncated, infos, as_numpy, scalar):
        if not as_numpy:
            return obs, ret, terminated, truncated, infos

        def host(x):
            return x.cpu().numpy() if torch.is_tensor(x) else x
        obs, ret, terminated, truncated = host(obs), host(ret), host(terminated), host(truncated)
        infos = {k: host(v) for k, v in infos.items()}
        if scalar:
            L = int(infos["trajectory_length"][0])
            out = {}
            for k, v in infos.items():
                v0 = v[0]
                if k in ("step_actions", "step_rewards", "step_observations"):
                    v0 = v0[:L]
                elif k == "trajectory_length":
                    v0 = L
                elif np.ndim(v0) == 0:
                    v0 = v0.item()
                out[k] = v0
            return obs[0], float(ret[0]), bool(terminated[0]), bool(truncated[0]), out
        return obs, ret, terminated, truncated, infos

    def render(self):
        self.do_render = True

    def reset(self, *, seed: Optional[int] = None, options: Optional[Dict[str, Any]] = None):
        """black_box_wrapper.py:222-229"""
        self.current_traj_steps = 0
        self.plan_steps = 0
        self.traj_gen.reset()
        self.condition_set = False
        base = self._base
        if self._fast_reset and not {k for k in (options or {}) if k != "as_numpy"}:
            # one kernel: numpy-exact context sampling + state reset + context observation (fg_reset)
            obs, info = base.device_reset(seed, obs_index=self._obs_index_np, time_aware=self._time_aware()), {}
        else:
            obs, info = self.env.reset(seed=seed, options={k: v for k, v in (options or {}).items() if k != "as_numpy"} or None)
            obs = self.observation(obs).contiguous()
        as_numpy = (options or {}).get("as_numpy", self.num_envs == 1)
        if as_numpy:
            obs = obs.cpu().numpy()
            if self.num_envs == 1:
                obs = obs[0]
        return obs, info

    def reset_done(self, mask=None):
        """Auto-reset for vector-env use: starts a new episode in every env whose last step ended one (or where `mask`
        is set), continuing each env's own context stream, in one fg_reset launch.  Returns the observation of ALL envs
        (rows of envs that were not reset are unchanged).  Only meaningful when every env plans on the same schedule,
        i.e. without replanning / sub-trajectories (there a finished env waits for reset())."""
        if not self._fast_reset:
            raise NotImplementedError("reset_done() needs the device-side sampler (context_sampler='device')")
        if self.do_replanning or self.learn_sub_trajectories:
            raise NotImplementedError("partial resets are not defined while envs share one replanning clock")
        if mask is None:
            mask = self._base.done
        # a new episode: the phase generator un-finalizes like in reset() (black_box_wrapper.py:226), otherwise a learned tau /
        # delay would stay frozen at the first episode's values
        self.traj_gen.reset()
        obs = self._obs.clone()
        self._base.device_reset(None, obs_index=self._obs_index_np, time_aware=self._time_aware(), out=obs, mask=mask)
        return obs

    def close(self):
        for h in self._handles.values():
            _lib.lib.fg_destroy(h)
        self._handles.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
