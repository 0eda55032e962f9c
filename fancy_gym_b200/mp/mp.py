"""Trajectory generators (host facade over the CUDA kernels): the role of mp_pytorch.mp.{ProMP,
DMP, ProDMP} behind fancy_gym/black_box/factory/trajectory_generator_factory.py:7-21.

The method names are the ones BlackBoxWrapper calls (black_box_wrapper.py:57,62-65,102,106,
113-118,124,226): set_duration, set_params, set_initial_conditions, get_traj_pos, get_traj_vel,
get_params_bounds, reset, plus the attributes phase_gn / basis_gn / tau / learn_tau.

Nothing here computes a trajectory on the CPU: this class only builds the small shared tables
(float64 -> float32, a few KB) and launches fg_trajgen; inside the fused rollout the same tables
are evaluated per env and per step in registers.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from .. import _lib
from .basis_gn import NormalizedRBFBasisGenerator, ProDMPBasisGenerator


def time_grid32(duration: float, dt: float, init_time: float) -> np.ndarray:
    """float32 time grid exactly as the library builds it: torch.linspace(0, duration, T+1) in
    float32, plus the float32 init_time, first point dropped (SURVEY.md App. B.1)."""
    T = int(round(duration / dt))
    grid = torch.linspace(0, float(duration), T + 1, dtype=torch.float32).numpy()
    return (grid + np.float32(init_time)).astype(np.float32)[1:]


class MPTables:
    """What fg_create needs from a trajectory generator for one plan."""
    __slots__ = ("mp_kind", "n_basis", "n_steps", "tab_a", "tab_b", "tau", "dmp_alpha", "weights_scale",
                 "goal_scale", "relative_goal")

    def __init__(self, **kw):
        self.tau, self.dmp_alpha, self.weights_scale, self.goal_scale, self.relative_goal = 1.0, 25.0, 1.0, 1.0, 0
        for k, v in kw.items():
            setattr(self, k, v)


class MPInterface:
    mp_kind = -1

    def __init__(self, basis_gn: NormalizedRBFBasisGenerator, num_dof: int, weights_scale: float = 1.0,
                 device=None, **kwargs):
        self.basis_gn = basis_gn
        self.phase_gn = basis_gn.phase_generator
        self.num_dof = int(num_dof)
        self.weights_scale = weights_scale
        self.device = torch.device(device) if device is not None else torch.device("cuda")
        self.duration = None
        self.dt = None
        self.init_time = 0.0
        self.init_pos = None
        self.init_vel = None
        self.params = None
        self._handles = {}
        self._pc_dev = None
        self.n_steps_env = None

    # ---- attributes the reference reads -----------------------------------------------------
    @property
    def learn_tau(self):
        return self.phase_gn.learn_tau

    @property
    def learn_delay(self):
        return self.phase_gn.learn_delay

    @property
    def tau(self):
        return self.phase_gn.tau

    @property
    def _num_local_params(self) -> int:
        raise NotImplementedError

    @property
    def num_params(self) -> int:
        return self.phase_gn.num_params + self._num_local_params

    # ---- BlackBoxWrapper-facing API -----------------------------------------------------------
    def reset(self):
        self.phase_gn.reset()

    def get_params_bounds(self) -> torch.Tensor:
        lo, hi = self.phase_gn.get_params_bounds()
        n = self._num_local_params
        return torch.tensor([lo + [-float("inf")] * n, hi + [float("inf")] * n], dtype=torch.float32)

    def set_params(self, params):
        params = torch.as_tensor(params)
        if params.shape[-1] != self.num_params:
            raise ValueError(f"expected {self.num_params} params, got {tuple(params.shape)}")
        self.params = self._prepare_local(self.phase_gn.set_params(params))

    def _prepare_local(self, local):
        """hook: the MP parameters as the kernels consume them (identity unless an assumption switch moves a scale / offset
        onto the parameters, mp/assumptions.py)"""
        return local

    def _param_scale(self, device):
        """hook: float32 factors [params per dof] that multiply the parameters because the switch scale_on_library_side
        moved the scales off the basis table; None while the scales sit on the table"""
        return None

    def boundary_prestep(self, params, pos, vel):
        """hook: boundary condition the kernels should start from instead of (pos, vel); None = as given"""
        return None

    def set_initial_conditions(self, init_time, init_pos, init_vel):
        self.init_time = float(np.asarray(init_time if not torch.is_tensor(init_time) else init_time.cpu()))
        self.init_pos = init_pos
        self.init_vel = init_vel

    def set_duration(self, duration, dt):
        self.dt = float(dt)
        self.n_steps_env = None
        if duration is None:     # learn_sub_trajectories: trajectory length follows the learned tau
            if not self.phase_gn.collapse_if_equal():
                # the envs of the batch chose different taus: ragged plans.  Env b plans round(tau_b / dt) points; buffers and
                # launches are sized for the longest admissible plan (tau_bound), the lengths stay on the device.
                hi = float(self.phase_gn.tau_bound[1])
                if not np.isfinite(hi):
                    # a phase generator built without make_bb has tau_bound = [1e-5, inf]: buffers cannot be sized for an
                    # unbounded plan length (make_bb sets [2 dt, duration] when tau is learned, make_env_helpers.py:121-126)
                    raise ValueError("ragged sub-trajectories need a finite phase_generator_kwargs['tau_bound'] upper bound "
                                     "(the longest plan the buffers are sized for)")
                t_max = int(np.round(hi / dt))
                tau = self.phase_gn.tau.to(self.device, torch.float64)
                self.n_steps_env = torch.round(tau / dt).clamp_(2, t_max).to(torch.int32).contiguous()
                duration = float(t_max * dt)
            else:
                duration = float(np.round(self.phase_gn.scalar_tau() / dt) * dt)
        self.duration = float(duration)

    def _times_table(self):
        """[T_max + 1, T_max] float32: row n is the library's time grid of an n-point plan (torch.linspace on the host, so
        the rounding pattern is the library's), zero padded — the per-env grids of ragged plans are looked up here"""
        key = (self.n_steps, self.dt, float(np.float32(self.init_time)))
        if getattr(self, "_tt_key", None) != key:
            t_max = self.n_steps
            tab = np.zeros((t_max + 1, t_max), dtype=np.float32)
            for n in range(1, t_max + 1):
                tab[n, :n] = time_grid32(float(n * self.dt), self.dt, self.init_time)
            self._tt = torch.as_tensor(tab, device=self.device)
            self._tt_key = key
        return self._tt

    @property
    def n_steps(self) -> int:
        return int(round(self.duration / self.dt))

    def times32(self) -> np.ndarray:
        return time_grid32(self.duration, self.dt, self.init_time)

    def times_dev(self) -> torch.Tensor:
        """the plan's float32 time grid on the device (cached per plan)"""
        key = (self.n_steps, self.dt, float(np.float32(self.init_time)), str(self.device))
        if getattr(self, "_td_key", None) != key:
            self._td = torch.as_tensor(self.times32(), device=self.device)
            self._td_key = key
        return self._td

    def tables(self) -> MPTables:
        raise NotImplementedError

    def table_key(self):
        """identifies the shared tables of the current plan (handles are cached under it)"""
        pg = self.phase_gn
        return (self.n_steps, round(self.init_time / self.dt), pg.scalar_tau(), pg.scalar_delay())

    def _phase_basis(self) -> "_lib.FgPhaseBasis":
        """constants of the phase / basis generators for the per-env-phase kernel (fg_phase_basis)"""
        bg, pg = self.basis_gn, self.phase_gn
        pb = _lib.FgPhaseBasis()
        pb.struct_size = C.sizeof(_lib.FgPhaseBasis)
        pb.phase_kind = 1 if pg.kind == "exp" else 0
        pb.alpha_phase = float(getattr(pg, "alpha_phase", 0.0))
        pb.n_basis_total, pb.first_learnable = bg.total_num_basis, bg.first_learnable
        if bg.total_num_basis > 16:
            raise NotImplementedError("per-env phase: at most 16 basis functions")
        for k in range(bg.total_num_basis):
            pb.centers[k], pb.bandwidth[k] = float(bg.centers_p[k]), float(bg.bandwidth[k])
        if self.mp_kind == _lib.MP_PRODMP:
            # the pre-integrated bases depend on the construction-time tau only; per env only the lookup changes
            if self._pc_dev is None:
                self._pc_dev = tuple(torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=self.device)
                                     for x in (bg.pc_pos_basis, bg.pc_vel_basis, bg.pc_y))
            if pg.assume["prodmp_interpolate"]:
                raise NotImplementedError("prodmp_interpolate: only the shared-table path (no per-env tau / delay)")
            pb.pc_pos, pb.pc_vel, pb.pc_y = (x.data_ptr() for x in self._pc_dev)
            pb.n_pc = int(bg.pc_y.shape[0])
            pb.scaled_dt = float(np.float32(np.float32(bg.dt) / np.float32(pg._tau0)))
            pb.init_time = float(np.float32(self.init_time))
            for k, v in enumerate(self.weights_goal_scale()):
                pb.scale[k] = float(v)
        # float64 rounded once (the arithmetic of the shared tables; default) or, FG_PHASE_F32=1 / traj_gen.per_env_basis_f32,
        # float32 elementwise like the library's own tensors (12 % faster; velocities then carry the library's float32 noise)
        pb.eval_f64 = 0 if (getattr(self, "per_env_basis_f32", False) or os.environ.get("FG_PHASE_F32")) else 1
        pb.exp_right_clip = int(bool(pg.assume["exp_phase_right_clip"]))
        pb.basis_scale = float(self._forcing_basis_scale()) if self.mp_kind == _lib.MP_DMP else 1.0
        if self.n_steps_env is not None:
            tt = self._times_table()
            pb.n_steps_env, pb.times_table, pb.times_stride = self.n_steps_env.data_ptr(), tt.data_ptr(), tt.shape[1]
        return pb

    # ---- stand-alone trajectory generation on the GPU (fg_trajgen) ------------------------------
    def _trajgen_handle(self):
        key = (*self.table_key(), self.device.index or 0)
        h = self._handles.get(key)
        if h is None:
            tb = self.tables()
            cfg = _lib.FgConfig()
            cfg.struct_size = C.sizeof(_lib.FgConfig)
            cfg.env_kind, cfg.mp_kind, cfg.ctrl_kind = _lib.ENV_TOY, tb.mp_kind, _lib.CTRL_VELOCITY
            cfg.n_dof, cfg.n_steps, cfg.n_basis = self.num_dof, tb.n_steps, tb.n_basis
            cfg.max_episode_steps, cfg.dt = tb.n_steps, self.dt
            cfg.tau, cfg.dmp_alpha = tb.tau, tb.dmp_alpha
            cfg.weights_scale, cfg.goal_scale, cfg.relative_goal = tb.weights_scale, tb.goal_scale, tb.relative_goal
            ta = np.ascontiguousarray(tb.tab_a, dtype=np.float32)
            tbb = np.ascontiguousarray(tb.tab_b, dtype=np.float32)
            cfg.tab_a, cfg.tab_b = ta.ctypes.data, tbb.ctypes.data
            hp = C.c_void_p()
            _lib.check(_lib.lib.fg_create(C.byref(cfg), self.device.index or 0, C.byref(hp)))
            h = hp
            self._handles[key] = h
        return h

    def _run_trajgen(self, out=None):
        """Launches fg_trajgen for the current params / plan.  `out=(pos, vel)` re-uses caller-owned
        [B, T, dof] float32 device buffers (no allocation on the call path)."""
        if self.params is None:
            raise RuntimeError("set_params() must be called before get_traj_pos()/get_traj_vel()")
        p = self.params.to(self.device, torch.float32)
        batched = p.dim() == 2
        if not batched:
            p = p[None]
        p = p.contiguous()
        B, T, N = p.shape[0], self.n_steps, self.num_dof

        def bc(x):
            if x is None:
                return None
            x = torch.as_tensor(x).to(self.device, torch.float32)
            return x.expand(B, N).contiguous() if x.dim() < 2 else x.contiguous()

        bp, bv = bc(self.init_pos), bc(self.init_vel)
        if bp is not None and bv is not None:
            pre = self.boundary_prestep(p, bp, bv)
            if pre is not None:
                bp, bv = pre
        if out is None:
            pos = torch.empty(B, T, N, device=self.device, dtype=torch.float32)
            vel = torch.empty_like(pos)
        else:
            pos, vel = out
            assert pos.shape == (B, T, N) and vel.shape == (B, T, N) and pos.is_contiguous() and vel.is_contiguous()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if self.phase_gn.uniform():
            _lib.check(_lib.lib.fg_trajgen(self._trajgen_handle(), p.data_ptr(), bp.data_ptr() if bp is not None else None,
                                           bv.data_ptr() if bv is not None else None, pos.data_ptr(), vel.data_ptr(), B,
                                           C.c_void_p(stream)))
        else:       # per-env tau / delay: basis evaluated in the kernel (fg_trajgen_phase)
            pb = self._phase_basis()
            tau, delay = self.phase_gn.per_env(B, self.device)
            times = torch.as_tensor(self.times32(), device=self.device)
            _lib.check(_lib.lib.fg_trajgen_phase(self._trajgen_handle(), C.byref(pb), times.data_ptr(), tau.data_ptr(),
                                                 delay.data_ptr(), p.data_ptr(), bp.data_ptr() if bp is not None else None,
                                                 bv.data_ptr() if bv is not None else None, pos.data_ptr(), vel.data_ptr(),
                                                 B, C.c_void_p(stream)))
        return (pos, vel) if batched else (pos[0], vel[0])

    # ---- trajectory covariance of the probabilistic MPs (fg_traj_cov; mp_pytorch: set_mp_params_variances,
    # ---- get_traj_pos_cov, get_traj_pos_std — no call site inside fancy_gym, SURVEY.md §8 row a20) ----------------
    probabilistic = False

    def set_mp_params_variances(self, params_L):
        """params_L [B, D, D] (or [D, D]): lower-triangular Cholesky factor of the weight covariance, D = num_dof * Kc"""
        if not self.probabilistic:
            raise NotImplementedError(f"{type(self).__name__} is not a probabilistic MP")
        self.params_L = None if params_L is None else torch.as_tensor(params_L)

    def _run_traj_cov(self, want_cov, want_std, reg=1e-4, batch_scope=None, path=0):
        if batch_scope is None:
            batch_scope = self.phase_gn.assume["cov_reg_batch_global"]
        if getattr(self, "params_L", None) is None:
            raise RuntimeError("set_mp_params_variances() must be called first")
        L = self.params_L.to(self.device, torch.float32)
        batched = L.dim() == 3
        if not batched:
            L = L[None]
        L = L.contiguous()
        B, T, N = L.shape[0], self.n_steps, self.num_dof
        D = self._num_local_params
        if L.shape[1:] != (D, D):
            raise ValueError(f"params_L must be [.., {D}, {D}], got {tuple(L.shape)}")
        s = self._param_scale(L.device)
        if s is not None:
            # the kernels read the basis table, which then lacks the scales: the trajectories are Psi (S w), so their
            # covariance is Psi (S L)(S L)^T Psi^T; scaling rows keeps L lower triangular
            L = (L.view(B, N, D // N, D) * s[:, None]).view(B, D, D)
        h = self._trajgen_handle()
        cov = torch.empty(B, N * T, N * T, device=self.device, dtype=torch.float32) if want_cov else None
        std = torch.empty(B, T, N, device=self.device, dtype=torch.float32) if want_std else None
        if B > 0:       # (empty tensors have null data pointers, which fg_traj_cov refuses)
            work = torch.empty(int(_lib.lib.fg_traj_cov_work_floats(h, B)), device=self.device, dtype=torch.float32)
            stream = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(_lib.lib.fg_traj_cov(h, L.data_ptr(), float(reg), int(bool(batch_scope)),
                                            cov.data_ptr() if want_cov else None, std.data_ptr() if want_std else None,
                                            work.data_ptr(), int(path), B, C.c_void_p(stream)))
        if not batched:
            cov, std = (cov[0] if want_cov else None), (std[0] if want_std else None)
        return cov, std

    def get_traj_pos_cov(self, reg: float = 1e-4, batch_scope: bool = None, path: int = 0):
        """[.., dof*T, dof*T] float32, dof-major rows / columns (d * T + t)"""
        return self._run_traj_cov(True, False, reg, batch_scope, path)[0]

    def get_traj_pos_std(self, reg: float = 1e-4, batch_scope: bool = None):
        """[.., T, dof]: sqrt of the regularised covariance diagonal (the full matrix is never materialised)"""
        return self._run_traj_cov(False, True, reg, batch_scope)[1]

    def get_traj_pos(self):
        return self._run_trajgen()[0]

    def get_traj_vel(self):
        return self._run_trajgen()[1]

    def __del__(self):
        try:
            for h in self._handles.values():
                _lib.lib.fg_destroy(h)
        except Exception:
            pass


class ProMP(MPInterface):
    """pos = (weights_scale * Phi) W^T, vel = forward finite difference over the float32 time grid,
    last row duplicated (SURVEY.md App. B.4)."""
    mp_kind = _lib.MP_PROMP
    probabilistic = True

    @property
    def _num_local_params(self):
        return self.num_dof * self.basis_gn.num_basis

    def _basis_scale(self) -> float:
        return float(self.weights_scale) if self.phase_gn.assume["scale_on_library_side"] else 1.0

    def _prepare_local(self, local):
        if not self.phase_gn.assume["scale_on_library_side"]:       # the scale sits on the parameters (one float32 multiply)
            local = local.to(torch.float32) * float(np.float32(self.weights_scale))
        return local

    def _param_scale(self, device):
        if self.phase_gn.assume["scale_on_library_side"]:
            return None
        return torch.full((self.basis_gn.num_basis,), float(np.float32(self.weights_scale)), dtype=torch.float32, device=device)

    def tables(self) -> MPTables:
        t32 = self.times32()
        b = self.basis_gn.learnable_basis32(t32)
        tab_a = (b * np.float32(self._basis_scale())).astype(np.float32)
        tab_b = np.diff(t32).astype(np.float32)
        # (weights_scale is folded into tab_a; the per-env-phase kernel, which has no table, takes it from the config)
        return MPTables(mp_kind=self.mp_kind, n_basis=self.basis_gn.num_basis, n_steps=len(t32), tab_a=tab_a, tab_b=tab_b,
                        tau=self.phase_gn.scalar_tau(), weights_scale=self._basis_scale())


class DMP(MPInterface):
    """Semi-implicit Euler of  y'' = alpha (beta (g - y) - y') + x Phi w  in scaled time (App. B.6)."""
    mp_kind = _lib.MP_DMP

    def __init__(self, basis_gn, num_dof, weights_scale=1.0, goal_scale=1.0, alpha=25, goal_offset=0.0, **kwargs):
        super().__init__(basis_gn, num_dof, weights_scale, **kwargs)
        self.goal_scale = goal_scale
        self.goal_offset = float(goal_offset)
        self.alpha = alpha
        self.beta = alpha / 4

    def _forcing_basis_scale(self) -> float:
        """DMP: the library scales the parameters; with the switch flipped the scale sits on the forcing basis"""
        return 1.0 if self.phase_gn.assume["scale_on_library_side"] else float(self.weights_scale)

    def _param_weights_scale(self) -> float:
        return float(self.weights_scale) if self.phase_gn.assume["scale_on_library_side"] else 1.0

    def _prepare_local(self, local):
        if self.goal_offset:       # goal = goal_scale * theta_g + offset (switch goal_offset_after_scale) in parameter units
            off = self.goal_offset / float(self.goal_scale) if self.phase_gn.assume["goal_offset_after_scale"] else self.goal_offset
            local = local.to(torch.float32).clone()
            local.view(*local.shape[:-1], self.num_dof, -1)[..., -1] += float(np.float32(off))
        return local

    def boundary_prestep(self, params, pos, vel):
        """switch dmp_init_on_first_grid_point = False: the Euler recurrence starts at the boundary time t0 itself, so the
        state the kernels start from (the plan's first grid point) is one step further.  A handful of elementwise float32
        ops on [B, dof] (the kernels' own recurrence, float32; the forcing contraction is a plain sum here)."""
        pg = self.phase_gn
        if pg.assume["dmp_init_on_first_grid_point"]:
            return None
        dev, f32 = self.device, torch.float32
        p = params.to(dev, f32).reshape(-1, self.num_dof, self.basis_gn.num_basis + 1)
        B = p.shape[0]
        tau, delay = pg.per_env(B, dev)
        t0 = torch.tensor(float(np.float32(self.init_time)), dtype=f32, device=dev)
        t1 = torch.tensor(float(self.times32()[0]), dtype=f32, device=dev)
        z0, z1 = torch.clamp((t0 - delay) / tau, min=0), torch.clamp((t1 - delay) / tau, min=0)
        h = (z1 - z0)[:, None]
        arg = z0 if not pg.assume["exp_phase_right_clip"] else torch.clamp(z0, max=1)
        x = torch.exp(-pg.alpha_phase * arg.double())
        cen = torch.as_tensor(self.basis_gn.centers_p, device=dev)
        bw = torch.as_tensor(self.basis_gn.bandwidth, device=dev)
        phi = torch.exp(-((x[:, None] - cen) ** 2 * bw) / 2)
        if self.basis_gn.total_num_basis > 1:
            phi = phi / phi.sum(-1, keepdim=True)
        z = self.basis_gn.first_learnable
        xb = (x[:, None] * phi * self._forcing_basis_scale()).to(f32)[:, z:z + self.basis_gn.num_basis]
        w = p[..., :-1] * float(np.float32(self._param_weights_scale()))
        g = p[..., -1] * float(np.float32(self.goal_scale))
        f = (xb[:, None, :] * w).sum(-1)
        y = pos.to(dev, f32).expand(B, self.num_dof)
        yd = vel.to(dev, f32).expand(B, self.num_dof) * tau[:, None]
        a = float(self.alpha) * (float(self.beta) * (g - y) - yd) + f
        yd1 = yd + h * a
        y1 = y + h * yd1
        return y1.contiguous(), (yd1 / tau[:, None]).contiguous()

    @property
    def _num_local_params(self):
        return self.num_dof * (self.basis_gn.num_basis + 1)

    def tables(self) -> MPTables:
        pg = self.phase_gn
        t32 = self.times32()
        lin = pg.phase_argument32(t32)
        z = self.basis_gn.first_learnable
        xb = (pg.phase64(lin)[:, None] * self.basis_gn.basis64(lin) * self._forcing_basis_scale()).astype(np.float32)
        xb = np.ascontiguousarray(xb[:, z:z + self.basis_gn.num_basis])
        sc = pg.linear_phase32(t32, clip_hi=False)            # left-bounded scaled time, float32 ops
        tab_b = np.diff(sc).astype(np.float32)
        return MPTables(mp_kind=self.mp_kind, n_basis=self.basis_gn.num_basis, n_steps=len(t32), tab_a=xb, tab_b=tab_b,
                        tau=pg.scalar_tau(), dmp_alpha=float(self.alpha), weights_scale=self._param_weights_scale(),
                        goal_scale=float(self.goal_scale))


class ProDMP(MPInterface):
    """Closed-form DMP solution with boundary conditions (App. B.7):
    pos = xi1 y_b + xi2 tau dy_b + H_pos [w; g],  vel = (xi3 y_b + xi4 tau dy_b + H_vel [w; g]) / tau."""
    mp_kind = _lib.MP_PRODMP
    probabilistic = True

    def __init__(self, basis_gn, num_dof, weights_scale=1.0, goal_scale=1.0, auto_scale_basis=False,
                 relative_goal=False, disable_weights=False, disable_goal=False, goal_offset=0.0, **kwargs):
        assert isinstance(basis_gn, ProDMPBasisGenerator)      # trajectory_generator_factory.py:16-17
        if disable_weights or disable_goal:
            raise NotImplementedError("disable_weights / disable_goal are not used by any fancy_gym config")
        super().__init__(basis_gn, num_dof, weights_scale, **kwargs)
        self.goal_scale = goal_scale
        self.goal_offset = float(goal_offset)
        self.auto_scale_basis = auto_scale_basis
        self.relative_goal = relative_goal

    @property
    def _num_local_params(self):
        return self.num_dof * (self.basis_gn.num_basis + 1)

    def weights_goal_scale(self) -> np.ndarray:
        K = self.basis_gn.num_basis
        s = np.zeros(K + 1)
        s[:K] = self.weights_scale
        s[K] = self.goal_scale
        if not self.phase_gn.assume["scale_on_library_side"]:      # the scales sit on the parameters (_prepare_local)
            s[:] = 1.0
        if self.auto_scale_basis:
            s = s * self.basis_gn.auto_basis_scale_factors
        return s

    def _prepare_local(self, local):
        A = self.phase_gn.assume
        on_basis = A["scale_on_library_side"]
        if on_basis and not self.goal_offset:
            return local
        K = self.basis_gn.num_basis
        local = local.to(torch.float32).clone()
        v = local.view(*local.shape[:-1], self.num_dof, K + 1)
        gs = float(self.goal_scale)
        if not on_basis:
            v *= self._param_scale(local.device)
        if self.goal_offset:
            if A["goal_offset_after_scale"]:
                off = self.goal_offset / gs if on_basis else self.goal_offset
            else:
                off = self.goal_offset if on_basis else self.goal_offset * gs
            v[..., -1] += float(np.float32(off))
        return local

    def _param_scale(self, device):
        if self.phase_gn.assume["scale_on_library_side"]:
            return None
        K = self.basis_gn.num_basis
        sc = torch.full((K + 1,), float(np.float32(self.weights_scale)), dtype=torch.float32, device=device)
        sc[K] = float(np.float32(self.goal_scale))
        return sc

    def tables(self) -> MPTables:
        bg = self.basis_gn
        t32 = self.times32()
        t64, tb64 = t32.astype(np.float64), np.float64(np.float32(self.init_time))
        y1, y2, dy1, dy2 = (bg.lookup(bg.pc_y, t64)[..., j] for j in range(4))
        y1b, y2b, dy1b, dy2b = (bg.lookup(bg.pc_y, tb64)[..., j] for j in range(4))
        pb, vb = bg.lookup(bg.pc_pos_basis, tb64), bg.lookup(bg.pc_vel_basis, tb64)
        det = y1b * dy2b - y2b * dy1b
        xi1 = dy2b / det * y1 - dy1b / det * y2
        xi2 = y1b / det * y2 - y2b / det * y1
        xi3 = dy2b / det * dy1 - dy1b / det * dy2
        xi4 = y1b / det * dy2 - y2b / det * dy1
        s = self.weights_goal_scale()
        pos_h = (bg.lookup(bg.pc_pos_basis, t64) - xi1[:, None] * pb - xi2[:, None] * vb) * s
        vel_h = (bg.lookup(bg.pc_vel_basis, t64) - xi3[:, None] * pb - xi4[:, None] * vb) * s
        tab_a = np.concatenate([xi1[:, None], xi2[:, None], pos_h], axis=1).astype(np.float32)
        tab_b = np.concatenate([xi3[:, None], xi4[:, None], vel_h], axis=1).astype(np.float32)
        return MPTables(mp_kind=self.mp_kind, n_basis=bg.num_basis, n_steps=len(t32), tab_a=tab_a, tab_b=tab_b,
                        tau=self.phase_gn.scalar_tau(), relative_goal=int(bool(self.relative_goal)))
