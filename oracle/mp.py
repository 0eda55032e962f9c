"""Restatement of the movement-primitive arithmetic the reference delegates to mp_pytorch.

TEST INFRASTRUCTURE (see oracle/__init__.py).

PARITY UNPINNED.  The arithmetic restated here lives in the third-party package
`mp_pytorch<=0.1.3` (reference pin: pyproject.toml:30, setup.py:63; upstream ALRhub/MP_PyTorch).
It is not vendored under /root/reference and not installed in this image, and the reference's
tests hold no numeric golden vector for it (SURVEY.md §8c).  This file restates the library's
published algorithm (SURVEY.md App. B) and is anchored on the reference's call sites
(fancy_gym/black_box/black_box_wrapper.py:57,62-65,102,106,113-118,124,226; factories under
fancy_gym/black_box/factory/) and structural tests (test/test_black_box.py:168-368,
test/test_replanning_sequencing.py:64-364).

Three arithmetic modes (argument `mode`):
  'gold'    everything float64: the mathematical definition.
  'shipped' everything float32 with the library's operation order (what the reference's
            torch-fp32 path computes up to BLAS summation order).
  'mirror'  what the CUDA path is specified to compute: basis/phase tables evaluated in float64
            and rounded once to float32, per-env contraction as a float32 FMA chain in index
            order, float32 IEEE division for the finite-difference velocity.  The CUDA kernels
            must match this mode to the last bit on table-driven paths; 'shipped' and 'gold'
            bound how far that is from the reference's own fp32 rounding noise.

All generators accept a leading batch axis on params ([B,P]); tau / delay may be per-env
arrays of shape [B] (learn_tau / learn_delay).
"""
from __future__ import annotations

import numpy as np

F32, F64 = np.float32, np.float64

# ----------------------------------------------------------------------------------------------
# Named switches for every point where this restatement of mp_pytorch could not be checked against the package
# (SURVEY.md App. B.8 i-vi plus two more).  The DEFAULT of each switch is what the restatement assumes; flipping one
# gives the alternative reading.  fancy_gym_b200/mp/assumptions.py holds the same table for the CUDA path (a CPU test keeps
# the two in step) and DESIGN.md carries the sensitivity of every BASELINE env to every switch
# (tools/mp_sensitivity.py).  A generator captures the switches when it is constructed.
# ----------------------------------------------------------------------------------------------
ASSUMPTIONS = {
    # B.8 (i)  DMP: the first grid point t0 + dt carries the initial state (set_duration(include_init_time=False) drops t0 and
    #          the Euler recurrence starts on the first remaining point).  False: the recurrence starts at t0 itself and the
    #          row of t0 is dropped afterwards (every output row is one Euler step further).
    "dmp_init_on_first_grid_point": True,
    # B.8 (ii) weights_scale / goal_scale multiply the BASIS (ProMP, ProDMP) resp. the PARAMETERS (DMP).  False: the other
    #          way round.  Algebraically identical; float32 rounding differs.
    "scale_on_library_side": True,
    # B.8 (iii) default alpha_phase of the exponential phase when a config does not give one (registry.py:112-115, ProDMP)
    "alpha_phase_default": 3.0,
    # B.8 (iv) RBF centres are mapped through the UNBOUNDED phase.  False: through the bounded one (identical for
    #          num_basis_outside = 0, which is every fancy_gym config).
    "centres_through_unbounded_phase": True,
    # B.8 (v)  covariance regulariser: max(diag) per sample.  True: over the whole batch (torch.max of a batched tensor).
    "cov_reg_batch_global": False,
    # B.8 (vi) goal_offset (kwarg, default 0; no classic_control config sets it) is added AFTER goal_scale.  False: before.
    "goal_offset_after_scale": True,
    # exponential phase x = exp(-alpha_phase * z): z is the linear phase clipped to [0, 1].  False: only left-bounded
    # (z = max((t - delay) / tau, 0)), so x keeps decaying after t = delay + tau.  Matters whenever tau < duration
    # (fancy_ProDMP/*: tau = 1.5 < 2.0).
    "exp_phase_right_clip": True,
    # ProDMP: pre-integrated bases are read at the NEAREST grid index.  True: linear interpolation between grid points.
    "prodmp_interpolate": False,
}
_DEFAULT_ASSUMPTIONS = dict(ASSUMPTIONS)


class assume:
    """context manager: `with assume(exp_phase_right_clip=False): orc = make_oracle(...)`"""

    def __init__(self, **switches):
        unknown = set(switches) - set(ASSUMPTIONS)
        if unknown:
            raise KeyError(f"unknown assumption switch(es): {sorted(unknown)}")
        self.switches = switches

    def __enter__(self):
        self.saved = dict(ASSUMPTIONS)
        ASSUMPTIONS.update(self.switches)
        return self

    def __exit__(self, *exc):
        ASSUMPTIONS.clear()
        ASSUMPTIONS.update(self.saved)
        return False


# ----------------------------------------------------------------------------------------------
# exact float32 FMA emulation (round-to-odd in float64, then one rounding to float32)
# ----------------------------------------------------------------------------------------------
def fma32(a, b, c):
    """Correctly rounded float32 fma(a,b,c) for float32 inputs (same result as CUDA fmaf)."""
    a64 = np.asarray(a, dtype=F32).astype(F64)
    b64 = np.asarray(b, dtype=F32).astype(F64)
    c64 = np.asarray(c, dtype=F32).astype(F64)
    p = a64 * b64                       # exact: 24+24 bits fit in 53
    s = p + c64
    bb = s - p
    err = (p - (s - bb)) + (c64 - bb)   # TwoSum: p + c == s + err exactly
    toward = np.where(err > 0, np.inf, -np.inf)
    s_next = np.nextafter(s, toward)
    even = (s.view(np.int64) & 1) == 0
    s_odd = np.where((err != 0) & even, s_next, s)
    return s_odd.astype(F32)


def fma_chain32(table, w):
    """out[..., t, d] = fma-chain over k of table[..., t, k] * w[..., d, k], k ascending, acc0 = 0."""
    table = np.asarray(table, dtype=F32)
    w = np.asarray(w, dtype=F32)
    K = table.shape[-1]
    acc = np.zeros(np.broadcast_shapes(table[..., :, None, 0].shape, w[..., None, :, 0].shape), dtype=F32)
    for k in range(K):
        acc = fma32(table[..., :, None, k], w[..., None, :, k], acc)
    return acc


def _dt_of(mode):
    return F64 if mode == "gold" else F32


def time_grid(duration, dt, init_time, mode):
    """App. B.1.  The library builds `torch.linspace(0, duration, round(duration/dt)+1)` in float32,
    adds the float32 init_time and drops the first point; the float32 modes call torch.linspace so
    that the rounding pattern of the grid (and hence of the finite-difference velocity) is the
    library's.  'gold' uses the exact float64 grid."""
    T = int(round(duration / dt))
    if mode == "gold":
        return np.asarray(init_time, dtype=F64)[..., None] + np.linspace(0, duration, T + 1, dtype=F64)[1:]
    import torch
    grid = torch.linspace(0, float(duration), T + 1, dtype=torch.float32).numpy()
    t0 = np.asarray(init_time, dtype=F64).astype(F32)
    return (grid + t0[..., None]).astype(F32)[..., 1:]


# ----------------------------------------------------------------------------------------------
# phase generators  (mp_pytorch.phase_gn.LinearPhaseGenerator / ExpDecayPhaseGenerator)
# ----------------------------------------------------------------------------------------------
class PhaseGenerator:
    """App. B.2.  params consumed from the front of the vector: [tau][delay] (then, for the exp
    phase, [alpha_phase] if learn_alpha_phase).  tau/delay freeze after the first set_params()
    until reset() ("finalize")."""

    def __init__(self, phase_generator_type="linear", tau=3.0, delay=0.0, learn_tau=False,
                 learn_delay=False, alpha_phase=None, learn_alpha_phase=False, tau_bound=None,
                 delay_bound=None, alpha_phase_bound=None, mode="gold", **kwargs):
        t = phase_generator_type.lower()
        if t in ("rhythmic", "smooth"):
            raise NotImplementedError()      # fancy_gym/black_box/factory/phase_generator_factory.py:15-20
        if t not in ("linear", "exp"):
            raise ValueError(f"Specified phase generator type {t} not supported")
        self.kind = t
        self.mode = mode
        self.dtype = _dt_of(mode)
        self.assume = dict(ASSUMPTIONS)
        if alpha_phase is None:
            alpha_phase = self.assume["alpha_phase_default"]
        self.tau0, self.delay0, self.alpha0 = float(tau), float(delay), float(alpha_phase)
        self.learn_tau, self.learn_delay = bool(learn_tau), bool(learn_delay)
        self.learn_alpha_phase = bool(learn_alpha_phase) and t == "exp"
        self.tau_bound = list(tau_bound) if tau_bound is not None else [1e-5, np.inf]
        self.delay_bound = list(delay_bound) if delay_bound is not None else [0, np.inf]
        self.alpha_phase_bound = list(alpha_phase_bound) if alpha_phase_bound is not None else [1e-5, np.inf]
        self.reset()

    def reset(self):
        self.tau = np.asarray(self.tau0, dtype=self.dtype)
        self.delay = np.asarray(self.delay0, dtype=self.dtype)
        self.alpha_phase = np.asarray(self.alpha0, dtype=self.dtype)
        self.is_finalized = False

    @property
    def num_params(self):
        return int(self.learn_tau) + int(self.learn_delay) + int(self.learn_alpha_phase)

    def set_params(self, params):
        i = 0
        if self.learn_tau:
            if not self.is_finalized:
                self.tau = np.asarray(params[..., i], dtype=self.dtype)
                assert self.tau.min() > 0
            i += 1
        if self.learn_delay:
            if not self.is_finalized:
                self.delay = np.asarray(params[..., i], dtype=self.dtype)
                assert self.delay.min() >= 0
            i += 1
        if self.learn_alpha_phase:
            if not self.is_finalized:
                self.alpha_phase = np.asarray(params[..., i], dtype=self.dtype)
            i += 1
        self.is_finalized = True
        return params[..., i:]

    def get_params_bounds(self):
        lo, hi = [], []
        for flag, b in ((self.learn_tau, self.tau_bound), (self.learn_delay, self.delay_bound),
                        (self.learn_alpha_phase, self.alpha_phase_bound)):
            if flag:
                lo.append(b[0])
                hi.append(b[1])
        return np.array(lo, dtype=F64), np.array(hi, dtype=F64)

    # times: [T] or [B,T]; tau/delay scalar or [B]
    def _bc(self, x):
        return x[..., None] if np.ndim(x) > 0 else x

    def unbound_linear_phase(self, times):
        return (times - self._bc(self.delay)) / self._bc(self.tau)

    def left_bound_linear_phase(self, times):
        return np.maximum(self.unbound_linear_phase(times), 0).astype(self.dtype)

    def linear_phase(self, times):
        return np.clip(self.unbound_linear_phase(times), 0, 1).astype(self.dtype)

    def linear_phase_to_time(self, z):
        return z * self._bc(self.tau) + self._bc(self.delay)

    def exp_argument(self, times):
        """the scaled time z the exponential phase decays over (switch exp_phase_right_clip)"""
        return self.linear_phase(times) if self.assume["exp_phase_right_clip"] else self.left_bound_linear_phase(times)

    def phase(self, times):
        if self.kind == "linear":
            return self.linear_phase(times)
        return np.exp(-self._bc(self.alpha_phase) * self.exp_argument(times)).astype(self.dtype)

    def phase_argument(self, times):
        """what the canonical phase is a function of: the clipped linear phase, or (exp phase without the right clip) the
        left-bounded one"""
        return self.linear_phase(times) if self.kind == "linear" else self.exp_argument(times)

    def bound_phase(self, times):
        """canonical phase of the linear phase clipped to [0, 1] (switch centres_through_unbounded_phase = False)"""
        if self.kind == "linear":
            return self.linear_phase(times)
        return np.exp(-self._bc(self.alpha_phase) * self.linear_phase(times)).astype(self.dtype)

    def unbound_phase(self, times):
        if self.kind == "linear":
            return self.unbound_linear_phase(times)
        return np.exp(-self._bc(self.alpha_phase) * self.unbound_linear_phase(times)).astype(self.dtype)


# ----------------------------------------------------------------------------------------------
# basis generators (mp_pytorch.basis_gn.*)
# ----------------------------------------------------------------------------------------------
class NormalizedRBFBasis:
    """App. B.3: centres equally spaced in *time* over [delay, delay+tau] (construction-time tau
    and delay), mapped through the unbounded phase; bandwidth h_k = f / (spacing_k)^2 with the
    last spacing repeated; b = exp(-h (phase - c)^2 / 2), normalised over k."""

    def __init__(self, phase_generator, num_basis=10, basis_bandwidth_factor=3, num_basis_outside=0,
                 mode=None, **kwargs):
        self.phase_generator = phase_generator
        self.mode = mode or phase_generator.mode
        self.dtype = _dt_of(self.mode)
        self._num_basis = int(num_basis)
        self.basis_bandwidth_factor = basis_bandwidth_factor
        self.num_basis_outside = num_basis_outside
        self._build_centres()

    def _build_centres(self):
        pg = self.phase_generator
        assert np.ndim(pg.tau) == 0, "centres are built from the construction-time scalar tau"
        dt = self.dtype
        K = self._num_basis
        if K > 1:
            tau, delay = dt(pg.tau), dt(pg.delay)
            basis_dist = tau / dt(K - 2 * self.num_basis_outside - 1)
            centres_t = np.linspace(-self.num_basis_outside * basis_dist + delay,
                                    tau + self.num_basis_outside * basis_dist + delay, K, dtype=dt)
            through = pg.unbound_phase if pg.assume["centres_through_unbounded_phase"] else pg.bound_phase
            self.centres_p = np.asarray(through(centres_t), dtype=dt)
            spacing = np.concatenate([self.centres_p[1:] - self.centres_p[:-1],
                                      self.centres_p[-1:] - self.centres_p[-2:-1]])
            self.bandwidth = (dt(self.basis_bandwidth_factor) / spacing ** 2).astype(dt)
        else:
            self.centres_p = np.array([0.5], dtype=dt)
            self.bandwidth = np.array([3.0], dtype=dt)

    @property
    def num_basis(self):
        return self._num_basis

    @property
    def total_num_basis(self):
        return self._num_basis

    def basis_from_phase(self, phase):
        """phase [...,T] -> [...,T,K_total]"""
        ph = np.asarray(phase, dtype=self.dtype)[..., None]
        tmp = (ph - self.centres_p) ** 2 * self.bandwidth
        b = np.exp(-tmp / 2)
        if self.total_num_basis > 1:
            b = b / b.sum(axis=-1, keepdims=True)
        return b.astype(self.dtype)

    def basis(self, times):
        return self.basis_from_phase(self.phase_generator.phase(times))


class ZeroPaddingNormalizedRBFBasis(NormalizedRBFBasis):
    """K learnable RBFs padded with `num_basis_zero_start` / `num_basis_zero_goal` RBFs whose
    weights are fixed to zero (HoleReacher: 5 + 1 RBFs on centres linspace(0,1,6), h = 75)."""

    def __init__(self, phase_generator, num_basis=10, num_basis_zero_start=2, num_basis_zero_goal=0,
                 basis_bandwidth_factor=3, mode=None, **kwargs):
        self.num_basis_zero_start = int(num_basis_zero_start)
        self.num_basis_zero_goal = int(num_basis_zero_goal)
        total = int(num_basis) + self.num_basis_zero_start + self.num_basis_zero_goal
        super().__init__(phase_generator, num_basis=total, basis_bandwidth_factor=basis_bandwidth_factor,
                         num_basis_outside=0, mode=mode)

    @property
    def num_basis(self):
        return self._num_basis - self.num_basis_zero_start - self.num_basis_zero_goal

    @property
    def total_num_basis(self):
        return self._num_basis


class ProDMPBasis(NormalizedRBFBasis):
    """App. B.7: position / velocity bases pre-integrated by cumulative trapezoid on the scaled
    time grid z_j = j * dt/tau, j = 0 .. factor*round(tau/dt); evaluated at the *nearest* grid
    index (interpolate=True switches to linear interpolation, B.8)."""

    def __init__(self, phase_generator, num_basis=10, basis_bandwidth_factor=3, num_basis_outside=0,
                 dt=0.01, alpha=25, pre_compute_length_factor=6, interpolate=None, mode=None, **kwargs):
        assert phase_generator.kind == "exp"      # basis_generator_factory.py:16
        super().__init__(phase_generator, num_basis, basis_bandwidth_factor, num_basis_outside, mode)
        self.alpha = alpha
        self.dt = dt
        self.pre_compute_length_factor = pre_compute_length_factor
        self.interpolate = phase_generator.assume["prodmp_interpolate"] if interpolate is None else interpolate
        self.pre_compute()

    @property
    def num_basis_g(self):
        return self._num_basis + 1

    def pre_compute(self):
        pg = self.phase_generator
        # tables are always integrated in float64 and cast: in 'shipped' mode the library does this in
        # float32, whose exp(alpha z/2) up to z=6 is itself noisy (SURVEY §7 "ProDMP numerics"); the
        # cast happens at the end so the three modes share one table definition.
        tau = float(pg.tau0)
        self.scaled_dt = self.dt / tau
        n_pc = self.pre_compute_length_factor * int(round(1.0 / self.scaled_dt)) + 1
        z = np.linspace(0, self.pre_compute_length_factor, n_pc, dtype=F64)
        a = float(self.alpha)
        y1 = np.exp(-0.5 * a * z)
        y2 = z * y1
        dy1 = -0.5 * a * y1
        dy2 = -0.5 * a * y2 + y1
        q1 = (0.5 * a * z - 1) * np.exp(0.5 * a * z) + 1
        q2 = 0.5 * a * (np.exp(0.5 * a * z) - 1)
        # RBF basis and canonical phase on the grid, with construction-time tau/delay
        delay = float(pg.delay0)
        pc_times = z * tau + delay
        lin = np.clip((pc_times - delay) / tau, 0, 1 if pg.assume["exp_phase_right_clip"] else None)
        x = np.exp(-float(pg.alpha0) * lin)
        cen, bw = _gold_centres(self)
        b = np.exp(-((x[:, None] - cen) ** 2 * bw) / 2)
        if self._num_basis > 1:
            b = b / b.sum(axis=1, keepdims=True)
        e = np.exp(a * z / 2)
        dp1 = (z * e * x)[:, None] * b
        dp2 = (e * x)[:, None] * b
        dz = np.diff(z)[:, None]
        p1 = np.concatenate([np.zeros((1, b.shape[1])), np.cumsum(0.5 * (dp1[1:] + dp1[:-1]) * dz, axis=0)])
        p2 = np.concatenate([np.zeros((1, b.shape[1])), np.cumsum(0.5 * (dp2[1:] + dp2[:-1]) * dz, axis=0)])
        pos_w = p2 * y2[:, None] - p1 * y1[:, None]
        pos_g = q2 * y2 - q1 * y1
        vel_w = p2 * dy2[:, None] - p1 * dy1[:, None]
        vel_g = q2 * dy2 - q1 * dy1
        self.pc_pos_basis = np.concatenate([pos_w, pos_g[:, None]], axis=1)
        self.pc_vel_basis = np.concatenate([vel_w, vel_g[:, None]], axis=1)
        self.pc_y = np.stack([y1, y2, dy1, dy2], axis=1)
        self.auto_basis_scale_factors = 1.0 / np.abs(self.pc_pos_basis).max(axis=0)

    def _lookup(self, table, times):
        z = self.phase_generator.left_bound_linear_phase(np.asarray(times)).astype(F64)
        if z.max() > self.pre_compute_length_factor:
            raise RuntimeError("Time is beyond the pre-computation range.")
        idx = z / self.scaled_dt
        if not self.interpolate:
            # the library rounds in float32: torch.round(scaled_times / self.scaled_dt) with both operands float32
            # (scaled_dt = dt / tau0 is a float32 tensor); ties (k * tau0 / tau = x.5) depend on that rounding
            z32 = self.phase_generator.left_bound_linear_phase(np.asarray(times)).astype(F32)
            sd32 = F32(F32(self.dt) / F32(self.phase_generator.tau0))
            return table[np.rint((z32 / sd32).astype(F32)).astype(np.int64)]
        i0 = np.clip(np.floor(idx).astype(np.int64), 0, table.shape[0] - 2)
        fr = (idx - i0)[..., None]
        return table[i0] * (1 - fr) + table[i0 + 1] * fr

    def basis(self, times):
        return self._lookup(self.pc_pos_basis, times)

    def vel_basis(self, times):
        return self._lookup(self.pc_vel_basis, times)

    def general_solution_values(self, times):
        v = self._lookup(self.pc_y, times)
        return v[..., 0], v[..., 1], v[..., 2], v[..., 3]


# ----------------------------------------------------------------------------------------------
# trajectory generators (mp_pytorch.mp.ProMP / DMP / ProDMP)
# ----------------------------------------------------------------------------------------------
class MPBase:
    def __init__(self, basis_gn, num_dof, weights_scale=1.0, mode=None, **kwargs):
        self.basis_gn = basis_gn
        self.phase_gn = basis_gn.phase_generator
        self.num_dof = int(num_dof)
        self.weights_scale = weights_scale
        self.mode = mode or basis_gn.mode
        self.dtype = _dt_of(self.mode)
        self.learn_tau = self.phase_gn.learn_tau
        self.learn_delay = self.phase_gn.learn_delay
        self.times = None
        self.params = None
        self.init_time = None
        self.init_pos = None
        self.init_vel = None
        self.duration = None
        self.dt = None

    @property
    def tau(self):
        return self.phase_gn.tau

    # ---- interface used by BlackBoxWrapper ------------------------------------------------------
    def reset(self):
        self.phase_gn.reset()

    @property
    def _num_local_params(self):
        raise NotImplementedError

    @property
    def num_params(self):
        return self.phase_gn.num_params + self._num_local_params

    def get_params_bounds(self):
        lo, hi = self.phase_gn.get_params_bounds()
        n = self._num_local_params
        return np.stack([np.concatenate([lo, -np.inf * np.ones(n)]),
                         np.concatenate([hi, np.inf * np.ones(n)])])

    def set_params(self, params):
        params = np.asarray(params)
        assert params.shape[-1] == self.num_params, (params.shape, self.num_params)
        self.params = np.asarray(self.phase_gn.set_params(params), dtype=self.dtype)

    def set_initial_conditions(self, init_time, init_pos, init_vel):
        self.init_time = np.asarray(init_time, dtype=F64)
        self.init_pos = np.asarray(init_pos, dtype=self.dtype)
        self.init_vel = np.asarray(init_vel, dtype=self.dtype)

    def set_duration(self, duration, dt):
        """App. B.1: T = round(duration/dt) points init_time + dt*(1..T); duration None -> round(tau/dt)*dt.
        With per-env tau (a batch whose envs chose different sub-trajectory lengths) every env gets its own grid; the
        rows are padded to the longest one by repeating the last time point and `n_valid[b]` holds the true length."""
        self.dt = float(dt)
        self.n_valid = None
        t0 = 0.0 if self.init_time is None else self.init_time
        if duration is None:
            tau = np.asarray(self.phase_gn.tau, dtype=F64)
            if tau.ndim and not np.all(tau == tau.flat[0]):
                steps = np.round(tau / dt).astype(np.int64)
                rows = [time_grid(float(n * dt), dt, t0, self.mode) for n in steps]
                tmax = int(steps.max())
                self.times = np.stack([np.concatenate([r, np.full(tmax - len(r), r[-1], dtype=r.dtype)]) for r in rows])
                self.n_valid = steps
                self.duration = float(tmax * dt)
                return
            duration = float(np.round(float(tau.flat[0]) / dt) * dt)
        self.duration = duration
        self.times = time_grid(duration, dt, t0, self.mode)

    def _phase_times(self):
        return self.times


class ProMP(MPBase):
    """App. B.4."""

    @property
    def _num_local_params(self):
        return self.num_dof * self.basis_gn.num_basis

    def _basis_scale(self):
        return self.weights_scale if self.phase_gn.assume["scale_on_library_side"] else 1.0

    def _weights(self):
        w = self.params.reshape(*self.params.shape[:-1], self.num_dof, self.basis_gn.num_basis)
        if not self.phase_gn.assume["scale_on_library_side"]:
            w = (w * self.dtype(self.weights_scale)).astype(self.dtype)
        return w

    def _scaled_basis_learnable(self):
        """[...,T,K_learnable] = basis * weights_scale restricted to the learnable columns."""
        bg = self.basis_gn
        if self.mode == "mirror":
            b = _basis_from_linear_phase(bg, self.phase_gn.phase_argument(self.times)).astype(F32)
            b = (b * F32(self._basis_scale())).astype(F32)
        else:
            b = (bg.basis(self.times) * self.dtype(self._basis_scale())).astype(self.dtype)
        z0 = getattr(bg, "num_basis_zero_start", 0)
        return b[..., z0:z0 + bg.num_basis]

    def cov_basis(self):
        """[T, Kc] basis of traj_pos_cov: weights_scale * Phi wherever the switch scale_on_library_side puts the scale
        (on the parameters it scales Sigma_w to S Sigma_w S, the same as scaling the basis columns)"""
        b = self._scaled_basis_learnable()
        return b if self.phase_gn.assume["scale_on_library_side"] else b * self.dtype(self.weights_scale)

    def get_traj_pos(self):
        b = self._scaled_basis_learnable()
        w = self._weights()
        if self.mode == "mirror":
            return fma_chain32(b, w)
        return np.einsum("...ik,...jk->...ij", b, w).astype(self.dtype)

    def get_traj_vel(self):
        pos = self.get_traj_pos()
        vel = np.zeros_like(pos)
        dts = np.diff(self.times, axis=-1)
        with np.errstate(divide="ignore", invalid="ignore"):
            vel[..., :-1, :] = np.diff(pos, axis=-2) / dts[..., None]
        vel[..., -1, :] = vel[..., -2, :]
        if getattr(self, "n_valid", None) is not None:        # ragged batch: the last VALID row duplicates its predecessor
            for b, n in enumerate(self.n_valid):
                vel[b, n - 1] = vel[b, n - 2]
        return vel


def _phase_from_linear_phase(pg, lin):
    """canonical phase in float64 from a given (float32 or float64) linear phase z."""
    lin = np.asarray(lin).astype(F64)
    if pg.kind == "exp":
        alpha = np.asarray(pg.alpha_phase).astype(F64)
        return np.exp(-(alpha[..., None] if alpha.ndim else alpha) * lin)
    return lin


def _basis_from_linear_phase(bg, lin):
    """normalised RBF basis in float64 from a given linear phase z (mirror-mode transcendental part)."""
    ph = _phase_from_linear_phase(bg.phase_generator, lin)
    cen, bw = _gold_centres(bg)
    b = np.exp(-((ph[..., None] - cen) ** 2 * bw) / 2)
    if bg.total_num_basis > 1:
        b = b / b.sum(axis=-1, keepdims=True)
    return b


def _gold_centres(bg):
    pg = bg.phase_generator
    K = bg.total_num_basis
    if K <= 1:
        return np.array([0.5]), np.array([3.0])
    tau, delay = float(pg.tau0), float(pg.delay0)
    dist = tau / (K - 2 * bg.num_basis_outside - 1)
    ct = np.linspace(-bg.num_basis_outside * dist + delay, tau + bg.num_basis_outside * dist + delay, K)
    cp = (ct - delay) / tau
    if not pg.assume["centres_through_unbounded_phase"]:
        cp = np.clip(cp, 0, 1)
    if pg.kind == "exp":
        cp = np.exp(-float(pg.alpha0) * cp)
    sp = np.concatenate([cp[1:] - cp[:-1], cp[-1:] - cp[-2:-1]])
    return cp, float(bg.basis_bandwidth_factor) / sp ** 2


class DMP(MPBase):
    """App. B.6.  params per dof: K weights then the goal."""

    def __init__(self, basis_gn, num_dof, weights_scale=1.0, goal_scale=1.0, alpha=25, goal_offset=0.0, mode=None, **kwargs):
        super().__init__(basis_gn, num_dof, weights_scale, mode)
        self.goal_scale = goal_scale
        self.goal_offset = goal_offset
        self.alpha = alpha
        self.beta = alpha / 4

    @property
    def _num_local_params(self):
        return self.num_dof * (self.basis_gn.num_basis + 1)

    def _split(self):
        dt = self.dtype
        A = self.phase_gn.assume
        p = self.params.reshape(*self.params.shape[:-1], self.num_dof, self.basis_gn.num_basis + 1)
        w = p[..., :-1]
        if A["scale_on_library_side"]:          # DMP: the library scales the parameters
            w = (w * dt(self.weights_scale)).astype(dt)
        g = _scaled_goal(p[..., -1], self.goal_scale, self.goal_offset, A, dt)
        return w, g

    def _grid(self):
        """the time points the recurrence runs over: the plan's grid, or (switch dmp_init_on_first_grid_point = False) the
        grid with the boundary time t0 in front"""
        if self.phase_gn.assume["dmp_init_on_first_grid_point"]:
            return self.times
        t0 = np.asarray(self.init_time, dtype=F64).astype(self.times.dtype)
        t0 = np.broadcast_to(t0[..., None] if t0.ndim else t0, (*self.times.shape[:-1], 1))
        return np.concatenate([t0, self.times], axis=-1)

    def _forcing(self, w, times):
        scale = 1.0 if self.phase_gn.assume["scale_on_library_side"] else self.weights_scale
        if self.mode == "mirror":
            lin = self.phase_gn.phase_argument(times)
            xb = (_phase_from_linear_phase(self.phase_gn, lin)[..., None]
                  * _basis_from_linear_phase(self.basis_gn, lin) * scale).astype(F32)
            return fma_chain32(xb, w)
        x = self.phase_gn.phase(times)
        b = (self.basis_gn.basis(times) * self.dtype(scale)).astype(self.dtype)
        return np.einsum("...i,...ik,...jk->...ij", x, b, w).astype(self.dtype)

    def _integrate(self):
        dt = self.dtype
        w, g = self._split()
        times = self._grid()
        f = self._forcing(w, times)
        sc = self.phase_gn.left_bound_linear_phase(times)
        sdt = np.diff(sc, axis=-1).astype(dt)
        T = times.shape[-1]
        batch = np.broadcast_shapes(f.shape[:-2], np.shape(self.init_pos)[:-1])
        pos = np.zeros((*batch, T, self.num_dof), dtype=dt)
        vel = np.zeros_like(pos)
        tau = np.asarray(self.phase_gn.tau, dtype=dt)
        tau_b = tau[..., None] if tau.ndim else tau
        pos[..., 0, :] = self.init_pos
        vel[..., 0, :] = self.init_vel * tau_b
        alpha, beta = dt(self.alpha), dt(self.beta)
        for i in range(T - 1):
            acc = alpha * (beta * (g - pos[..., i, :]) - vel[..., i, :]) + f[..., i, :]
            h = sdt[..., i]
            h = h[..., None] if np.ndim(h) else h
            vel[..., i + 1, :] = vel[..., i, :] + h * acc
            pos[..., i + 1, :] = pos[..., i, :] + h * vel[..., i + 1, :]
        vel = vel / (tau_b[..., None] if np.ndim(tau_b) else tau_b)
        if T != self.times.shape[-1]:       # the row of t0 is not part of the plan
            pos, vel = pos[..., 1:, :], vel[..., 1:, :]
        return pos.astype(dt), vel.astype(dt)

    def get_traj_pos(self):
        return self._integrate()[0]

    def get_traj_vel(self):
        return self._integrate()[1]


def _scaled_goal(theta_g, goal_scale, goal_offset, A, dt):
    """goal parameter -> goal (switch goal_offset_after_scale; the offset is 0 in every classic_control config)"""
    if A["goal_offset_after_scale"]:
        g = (theta_g * dt(goal_scale)).astype(dt)
        return (g + dt(goal_offset)).astype(dt) if goal_offset else g
    return ((theta_g + dt(goal_offset)) * dt(goal_scale)).astype(dt)


class ProDMP(MPBase):
    """App. B.7.  params per dof: K weights then the goal."""

    def __init__(self, basis_gn, num_dof, weights_scale=1.0, goal_scale=1.0, auto_scale_basis=False,
                 relative_goal=False, disable_weights=False, disable_goal=False, goal_offset=0.0, mode=None, **kwargs):
        assert isinstance(basis_gn, ProDMPBasis)   # trajectory_generator_factory.py:16-17
        super().__init__(basis_gn, num_dof, weights_scale, mode)
        self.goal_scale = goal_scale
        self.goal_offset = goal_offset
        self.auto_scale_basis = auto_scale_basis
        self.relative_goal = relative_goal
        self.disable_weights = disable_weights
        self.disable_goal = disable_goal
        self.kwargs_duration = kwargs.get("duration")

    @property
    def _num_local_params(self):
        n = 0
        if not self.disable_weights:
            n += self.basis_gn.num_basis
        if not self.disable_goal:
            n += 1
        return self.num_dof * n

    def weights_goal_scale(self):
        K = self.basis_gn.num_basis
        s = np.zeros(K + 1)
        s[:K] = self.weights_scale
        s[K] = self.goal_scale
        if not self.phase_gn.assume["scale_on_library_side"]:     # the scales sit on the parameters instead (_full_params)
            s[:] = 1.0
        if self.auto_scale_basis:
            s = s * self.basis_gn.auto_basis_scale_factors
        return s

    def _param_scale(self):
        """[K+1] weights_scale per weight, goal_scale for the goal: the factors the switch scale_on_library_side=False
        moves from the basis onto the parameters"""
        K = self.basis_gn.num_basis
        sc = np.full(K + 1, float(self.weights_scale))
        sc[K] = float(self.goal_scale)
        return sc

    def cov_basis(self):
        """[T, K+1] basis of traj_pos_cov: pos_H with the scales wherever the switch scale_on_library_side puts them
        (on the parameters they scale Sigma_w to S Sigma_w S, the same as scaling the basis columns)"""
        pos_H = self.tables()[0]
        return pos_H if self.phase_gn.assume["scale_on_library_side"] else pos_H * self._param_scale()

    def _full_params(self):
        K = self.basis_gn.num_basis
        lead = self.params.shape[:-1]
        if self.disable_weights and self.disable_goal:
            return np.zeros((*lead, self.num_dof, K + 1))
        p = self.params.reshape(*lead, self.num_dof, -1).astype(F64)
        if self.disable_weights:
            p = np.concatenate([np.zeros((*lead, self.num_dof, K)), p], axis=-1)
        elif self.disable_goal:
            p = np.concatenate([p, np.zeros((*lead, self.num_dof, 1))], axis=-1)
        A = self.phase_gn.assume
        if not A["scale_on_library_side"]:
            sc = self._param_scale()
            p = (p.astype(F32) * sc.astype(F32)).astype(F32).astype(F64) if self.mode != "gold" else p * sc
        if self.goal_offset:
            p = p.copy()
            off, gs = float(self.goal_offset), float(self.goal_scale)
            on_basis = A["scale_on_library_side"]         # the goal column of the basis still multiplies by goal_scale
            if A["goal_offset_after_scale"]:
                off = off / gs if on_basis else off       # goal = goal_scale * theta_g + offset
            else:
                off = off if on_basis else off * gs       # goal = goal_scale * (theta_g + offset)
            p[..., -1] = p[..., -1] + off
        if self.relative_goal:
            p = p.copy()
            p[..., -1] = p[..., -1] + np.asarray(self.init_pos, dtype=F64)
        return p

    def tables(self):
        """(pos_H [..,T,K+1], vel_H, xi [..,T,4]) in float64, *including* weights_goal_scale."""
        bg = self.basis_gn
        t64 = self.times.astype(F64)
        t0 = np.asarray(self.init_time, dtype=F64)
        y1, y2, dy1, dy2 = bg.general_solution_values(t64)
        y1b, y2b, dy1b, dy2b = bg.general_solution_values(t0[..., None] if t0.ndim else t0)
        pb, vb = bg.basis(t0[..., None] if t0.ndim else t0), bg.vel_basis(t0[..., None] if t0.ndim else t0)
        if t0.ndim:
            y1b, y2b, dy1b, dy2b = (a[..., 0:1] for a in (y1b, y2b, dy1b, dy2b))
        det = y1b * dy2b - y2b * dy1b
        xi1 = dy2b / det * y1 - dy1b / det * y2
        xi2 = y1b / det * y2 - y2b / det * y1
        xi3 = dy2b / det * dy1 - dy1b / det * dy2
        xi4 = y1b / det * dy2 - y2b / det * dy1
        s = self.weights_goal_scale()
        pos_H = (bg.basis(t64) - xi1[..., None] * pb - xi2[..., None] * vb) * s
        vel_H = (bg.vel_basis(t64) - xi3[..., None] * pb - xi4[..., None] * vb) * s
        return pos_H, vel_H, np.stack([xi1, xi2, xi3, xi4], axis=-1)

    def _traj(self):
        dt = self.dtype
        pos_H, vel_H, xi = self.tables()
        tau = np.asarray(self.phase_gn.tau, dtype=F64)
        tau_b = tau[..., None] if tau.ndim else tau
        p = self._full_params()
        if self.mode == "gold":
            yb = np.asarray(self.init_pos, dtype=F64)
            vb = np.asarray(self.init_vel, dtype=F64) * tau_b
            pos = xi[..., 0][..., None] * yb[..., None, :] + xi[..., 1][..., None] * vb[..., None, :] \
                + np.einsum("...tk,...dk->...td", pos_H, p)
            vel = (xi[..., 2][..., None] * yb[..., None, :] + xi[..., 3][..., None] * vb[..., None, :]
                   + np.einsum("...tk,...dk->...td", vel_H, p)) / (tau_b[..., None] if np.ndim(tau_b) else tau_b)
            return pos, vel
        # float32 paths: 'shipped' (einsum) and 'mirror' (fma chain seeded with the BC terms)
        pos_H32, vel_H32, xi32 = pos_H.astype(F32), vel_H.astype(F32), xi.astype(F32)
        p32 = p.astype(F32)
        yb = np.asarray(self.init_pos, dtype=F32)
        vbs = (np.asarray(self.init_vel, dtype=F32) * np.asarray(tau_b, dtype=F32)).astype(F32)
        tau32 = np.asarray(tau_b, dtype=F32)
        tau32 = tau32[..., None] if np.ndim(tau32) else tau32
        if self.mode == "shipped":
            pos = xi32[..., 0][..., None] * yb[..., None, :] + xi32[..., 1][..., None] * vbs[..., None, :] \
                + np.einsum("...tk,...dk->...td", pos_H32, p32)
            vel = (xi32[..., 2][..., None] * yb[..., None, :] + xi32[..., 3][..., None] * vbs[..., None, :]
                   + np.einsum("...tk,...dk->...td", vel_H32, p32)) / tau32
            return pos.astype(F32), vel.astype(F32)
        # mirror: the table carries [xi_a, xi_b, H_0..H_K] and the "weights" are [y_b, tau*dy_b, w.., g]
        tab_p = np.concatenate([xi32[..., 0:2], pos_H32], axis=-1)
        tab_v = np.concatenate([xi32[..., 2:4], vel_H32], axis=-1)
        lead = np.broadcast_shapes(p32.shape[:-2], yb.shape[:-1])
        wext = np.concatenate([np.broadcast_to(yb, (*lead, self.num_dof))[..., None],
                               np.broadcast_to(vbs, (*lead, self.num_dof))[..., None],
                               np.broadcast_to(p32, (*lead, self.num_dof, p32.shape[-1]))], axis=-1)
        pos = fma_chain32(tab_p, wext)
        vel = (fma_chain32(tab_v, wext) / tau32).astype(F32)
        return pos, vel

    def get_traj_pos(self):
        return self._traj()[0]

    def get_traj_vel(self):
        return self._traj()[1]


# ----------------------------------------------------------------------------------------------
# factories with the reference's type strings and error conventions
# (fancy_gym/black_box/factory/{phase,basis,trajectory}_generator_factory.py)
# ----------------------------------------------------------------------------------------------
def get_phase_generator(phase_generator_type, mode="gold", **kwargs):
    return PhaseGenerator(phase_generator_type, mode=mode, **kwargs)


def get_basis_generator(basis_generator_type, phase_generator, **kwargs):
    t = basis_generator_type.lower()
    if t == "rbf":
        return NormalizedRBFBasis(phase_generator, **kwargs)
    if t == "zero_rbf":
        return ZeroPaddingNormalizedRBFBasis(phase_generator, **kwargs)
    if t == "prodmp":
        return ProDMPBasis(phase_generator, **kwargs)
    if t == "rhythmic":
        raise NotImplementedError()
    raise ValueError(f"Specified basis generator type {t} not supported")


def get_trajectory_generator(trajectory_generator_type, action_dim, basis_generator, **kwargs):
    t = trajectory_generator_type.lower()
    if t == "promp":
        return ProMP(basis_generator, action_dim, **kwargs)
    if t == "dmp":
        return DMP(basis_generator, action_dim, **kwargs)
    if t == "prodmp":
        return ProDMP(basis_generator, action_dim, **kwargs)
    raise ValueError(f"Specified movement primitive type {t} not supported")


# ----------------------------------------------------------------------------------------------
# trajectory covariance (App. B.5) — PARITY UNPINNED: mp_pytorch is absent and fancy_gym never calls it
def traj_pos_cov(basis, params_L, num_dof, reg=1e-4, batch_scope=None):
    """Sigma_y = Psi (L L^T) Psi^T + reg * max(diag Sigma_y) * I in float64.
    basis [T, Kc] (already scaled: weights_scale * Phi for ProMP, the bracketed H = [H_w | H_g] for ProDMP; `cov_basis()`),
    params_L [B, D, D] with D = num_dof * Kc (lower triangle used), rows / columns dof-major (d * T + t).
    Returns (cov [B, dof*T, dof*T], std [B, T, dof]); the max is per env unless batch_scope (mp_pytorch takes torch.max
    over whatever batch it is given; the reference never batches)."""
    if batch_scope is None:
        batch_scope = ASSUMPTIONS["cov_reg_batch_global"]
    basis = np.asarray(basis, dtype=F64)
    L = np.tril(np.asarray(params_L, dtype=F64))
    T, Kc = basis.shape
    B = L.shape[0]
    psi = np.zeros((num_dof * T, num_dof * Kc))
    for d in range(num_dof):
        psi[d * T:(d + 1) * T, d * Kc:(d + 1) * Kc] = basis
    sigma_w = L @ np.swapaxes(L, -1, -2)
    cov = psi[None] @ sigma_w @ psi.T[None]
    diag = np.einsum("bii->bi", cov)
    mx = diag.max() if batch_scope else diag.max(axis=1)[:, None, None]
    cov = cov + reg * mx * np.eye(num_dof * T)[None]
    std = np.sqrt(np.einsum("bii->bi", cov)).reshape(B, num_dof, T).transpose(0, 2, 1)
    return cov, std
