"""Host-side logic of the drop-in facade, no GPU needed: tracking laws (the reference's only numeric KAT,
test/test_controller.py), factories and their error types, registry / id scheme / config layering
(test/test_fancy_registry.py, envs/registry.py), make_bb argument handling, spaces and parameter layout
(test/test_black_box.py:168-193)."""
import itertools

import numpy as np
import pytest

import fancy_gym_b200 as fancy_gym
from fancy_gym_b200.black_box.factory import (basis_generator_factory, controller_factory, phase_generator_factory,
                                              trajectory_generator_factory)
from fancy_gym_b200.envs.registry import DefaultMPWrapper, nested_update
from tests.toy import ToyWrapper, register_toy

VECS = [np.zeros(3), np.ones(3), np.arange(0, 3)]
GAINS = [0, 1, 0.5, np.zeros(3), np.ones(3), np.arange(0, 3)]


@pytest.fixture(scope="module", autouse=True)
def _toy():
    register_toy(fancy_gym)


# ---- tracking laws (test/test_controller.py:9-69) ----------------------------------------------------------------
@pytest.mark.parametrize("ctrl_type", controller_factory.ALL_TYPES)
def test_every_advertised_controller_builds(ctrl_type):
    controller_factory.get_controller(ctrl_type)


def test_velocity_and_position_laws():
    vel, pos = controller_factory.get_controller("velocity"), controller_factory.get_controller("position")
    for p, v in itertools.product(VECS, VECS):
        assert np.array_equal(vel(p, v, None, None), v)
        assert np.array_equal(pos(p, v, None, None), p)


def test_pd_law_all_gain_shapes():
    for pg, dg in itertools.product(GAINS, GAINS):
        ctrl = controller_factory.get_controller("motor", p_gains=pg, d_gains=dg)
        assert np.array_equal(ctrl.p_gains, pg) and np.array_equal(ctrl.d_gains, dg)
        for p, v, cp, cv in itertools.product(VECS, VECS, VECS, VECS):
            assert np.array_equal(ctrl(p, v, cp, cv), pg * (p - cp) + dg * (v - cv))
        gp, gd = ctrl.gain_vectors(3)
        assert np.array_equal(gp, np.broadcast_to(pg, 3)) and np.array_equal(gd, np.broadcast_to(dg, 3))


@pytest.mark.parametrize("pos_vel", [(np.ones(3), np.ones(4)), (np.ones(4), np.ones(3)), (np.ones(4), np.ones(4))])
def test_pd_rejects_mismatched_shapes(pos_vel):
    ctrl = controller_factory.get_controller("motor")
    with pytest.raises(ValueError):
        ctrl(pos_vel[0], pos_vel[1], np.ones(3), np.ones(3))


def test_metaworld_law():
    ctrl = controller_factory.get_controller("metaworld")
    for p, cp, g in itertools.product(VECS, VECS, [0, 1, 0.5]):
        a = ctrl(np.append(p, g), None, np.append(cp, -1), None)
        assert np.array_equal(a, np.append(p - cp, g))
    with pytest.raises(ValueError):
        ctrl(np.ones(5), None, np.ones(4), None)


def test_kernel_codes_of_the_laws():
    from fancy_gym_b200 import _lib
    codes = {t: controller_factory.get_controller(t).abi_code for t in controller_factory.ALL_TYPES}
    assert codes == {"motor": _lib.CTRL_MOTOR, "velocity": _lib.CTRL_VELOCITY, "position": _lib.CTRL_POSITION,
                     "metaworld": None}


# ---- factories: error types (SURVEY §8b "Error conventions") ---------------------------------------------------
def test_factories_error_types():
    with pytest.raises(ValueError):
        controller_factory.get_controller("nope")
    with pytest.raises(ValueError):
        phase_generator_factory.get_phase_generator("nope")
    for reserved in ("rhythmic", "smooth"):
        with pytest.raises(NotImplementedError):
            phase_generator_factory.get_phase_generator(reserved)
    lin = phase_generator_factory.get_phase_generator("linear", tau=2.0)
    exp = phase_generator_factory.get_phase_generator("EXP", tau=2.0)          # case-insensitive
    with pytest.raises(NotImplementedError):
        basis_generator_factory.get_basis_generator("rhythmic", lin)
    with pytest.raises(ValueError):
        basis_generator_factory.get_basis_generator("nope", lin)
    with pytest.raises(AssertionError):
        basis_generator_factory.get_basis_generator("prodmp", lin)             # ProDMP needs the exp phase
    rbf = basis_generator_factory.get_basis_generator("rbf", exp, num_basis=4)
    with pytest.raises(ValueError):
        trajectory_generator_factory.get_trajectory_generator("idmp", 2, rbf, device="cpu")
    with pytest.raises(AssertionError):
        trajectory_generator_factory.get_trajectory_generator("prodmp", 2, rbf, device="cpu")
    assert trajectory_generator_factory.get_trajectory_generator("promp", 2, rbf, device="cpu").num_params == 8
    assert trajectory_generator_factory.get_trajectory_generator("dmp", 2, rbf, device="cpu").num_params == 10


# ---- registry ----------------------------------------------------------------------------------------------------
def test_registered_ids_match_the_reference_matrix():
    """fancy_gym/envs/__init__.py:38-87: four classic_control envs x {ProMP, DMP, ProDMP}"""
    names = ["SimpleReacher-v0", "LongSimpleReacher-v0", "ViaPointReacher-v0", "HoleReacher-v0"]
    for mp in ("ProMP", "DMP", "ProDMP"):
        assert fancy_gym.ALL_MOVEMENT_PRIMITIVE_ENVIRONMENTS[mp] == [f"fancy_{mp}/{n}" for n in names]
        assert fancy_gym.MOVEMENT_PRIMITIVE_ENVIRONMENTS_FOR_NS["fancy"][mp] == [f"fancy_{mp}/{n}" for n in names]
    assert len(fancy_gym.ALL_MOVEMENT_PRIMITIVE_ENVIRONMENTS["all"]) == 12
    assert fancy_gym.ALL_FANCY_MOVEMENT_PRIMITIVE_ENVIRONMENTS["all"] == fancy_gym.ALL_MOVEMENT_PRIMITIVE_ENVIRONMENTS["all"]


def test_nested_update_type_key_replaces_instead_of_merging():
    base = {"controller_kwargs": {"controller_type": "motor", "p_gains": 1.0, "d_gains": 0.1}, "x": {"a": 1, "b": 2}}
    nested_update(base, {"controller_kwargs": {"controller_type": "velocity"}, "x": {"b": 3}})
    assert base == {"controller_kwargs": {"controller_type": "velocity"}, "x": {"a": 1, "b": 3}}   # Q5: gains are gone


def test_register_upgrade_and_id_rules():
    from tests.toy import ToyEnv
    fancy_gym.register("dummyns/Thing-v3", entry_point=ToyEnv, mp_wrapper=ToyWrapper, max_episode_steps=50)
    assert "dummyns_ProMP/Thing-v3" in fancy_gym.MOVEMENT_PRIMITIVE_ENVIRONMENTS_FOR_NS["dummyns"]["ProMP"]
    fancy_gym.upgrade("NoNamespace-v1", ToyWrapper, base_id="toy-v0", add_mp_types=["DMP"])
    assert "gym_DMP/NoNamespace-v1" in fancy_gym.ALL_MOVEMENT_PRIMITIVE_ENVIRONMENTS["DMP"]
    with pytest.raises(AssertionError):
        fancy_gym.upgrade("ns/NoVersion", ToyWrapper)
    with pytest.raises(ValueError):
        fancy_gym.upgrade("a/b/c-v0", ToyWrapper)
    with pytest.raises(AssertionError):
        fancy_gym.register("ns/X-v0", entry_point=None)


def test_make_layers_the_config(monkeypatch):
    """defaults < mp_wrapper.mp_config < register-time < make-time; HoleReacher/ProMP ends with a velocity controller
    WITHOUT gains (the `_type` quirk) and weights_scale 2"""
    env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=2, device="cpu")
    assert type(env.tracking_controller).__name__ == "VelController" and not hasattr(env.tracking_controller, "p_gains")
    assert env.traj_gen.weights_scale == 2 and env.traj_gen.basis_gn.num_basis == 5
    assert env.action_space.shape == (25,) and env.observation_space.shape == (18,)
    env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=2, device="cpu",
                         mp_config_override={"basis_generator_kwargs": {"num_basis": 7},
                                             "controller_kwargs": {"controller_type": "motor", "p_gains": 3.0, "d_gains": 0.2}})
    assert env.action_space.shape == (35,) and env.tracking_controller.p_gains == 3.0
    env = fancy_gym.make("fancy_DMP/ViaPointReacher-v0", num_envs=1, device="cpu")
    assert env.action_space.shape == (30,) and env.traj_gen.weights_scale == 50
    env = fancy_gym.make("fancy_ProDMP/SimpleReacher-v0", num_envs=1, device="cpu")
    assert env.action_space.shape == (12,) and type(env.tracking_controller).__name__ == "PDController"
    assert (env.tracking_controller.p_gains, env.tracking_controller.d_gains) == (1.0, 0.1)       # registry defaults
    env = fancy_gym.make("fancy_ProMP/SimpleReacher-v0", num_envs=1, device="cpu")
    assert (env.tracking_controller.p_gains, env.tracking_controller.d_gains) == (0.6, 0.075)     # simple_reacher/mp_wrapper.py:10-30


# ---- make_bb: spaces, parameter layout, argument errors (test/test_black_box.py) ---------------------------------
@pytest.mark.parametrize("mp_type", ["promp", "dmp", "prodmp"])
@pytest.mark.parametrize("num_dof", [0, 1, 2, 5])
@pytest.mark.parametrize("num_basis", [1, 2, 5])
@pytest.mark.parametrize("learn_tau", [True, False])
@pytest.mark.parametrize("learn_delay", [True, False])
def test_action_space(mp_type, num_dof, num_basis, learn_tau, learn_delay):
    basis_type = "prodmp" if mp_type == "prodmp" else "rbf"
    env = fancy_gym.make_bb("toy-v0", [ToyWrapper], {}, {"trajectory_generator_type": mp_type, "action_dim": num_dof},
                            {"controller_type": "motor"},
                            {"phase_generator_type": "exp", "learn_tau": learn_tau, "learn_delay": learn_delay},
                            {"basis_generator_type": basis_type, "num_basis": num_basis}, device="cpu")
    extra = num_dof if "dmp" in mp_type else 0
    assert env.action_space.shape[0] == num_dof * num_basis + int(learn_tau) + int(learn_delay) + extra


def test_tau_delay_bounds_lead_the_parameter_vector():
    env = fancy_gym.make_bb("toy-v0", [ToyWrapper], {}, {"trajectory_generator_type": "promp"}, {"controller_type": "motor"},
                            {"phase_generator_type": "linear", "learn_tau": True, "learn_delay": True},
                            {"basis_generator_type": "rbf", "num_basis": 3}, device="cpu")
    lo, hi = env.action_space.low, env.action_space.high
    dur, dt = 50 * 0.02, 0.02
    assert np.allclose(lo[:2], [2 * dt, 0]) and np.allclose(hi[:2], [dur, dur - 2 * dt])      # make_env_helpers.py:119-126
    assert np.all(np.isinf(lo[2:])) and np.all(np.isinf(hi[2:]))
    assert env.tau_bound == [2 * dt, dur] and env.delay_bound == [0, dur - 2 * dt]


@pytest.mark.parametrize("mp_type", ["promp", "dmp"])
@pytest.mark.parametrize("env_id,wrapper", [("fancy/HoleReacher-v0", "MPWrapper_HoleReacher"),
                                            ("fancy/ViaPointReacher-v0", "MPWrapper_ViaPointReacher"),
                                            ("fancy/SimpleReacher-v0", "MPWrapper_SimpleReacher")])
def test_context_space(mp_type, env_id, wrapper):
    from fancy_gym_b200.envs import classic_control
    wrapper_class = getattr(classic_control, wrapper)
    env = fancy_gym.make_bb(env_id, [wrapper_class], {}, {"trajectory_generator_type": mp_type}, {"controller_type": "motor"},
                            {"phase_generator_type": "exp"}, {"basis_generator_type": "rbf"}, device="cpu")
    w = wrapper_class(fancy_gym.make(env_id, device="cpu"))
    mask = np.asarray(w.context_mask, dtype=bool)
    assert env.observation_space.shape == mask[mask].shape


def test_make_bb_argument_errors():
    args = ({"trajectory_generator_type": "promp"}, {"controller_type": "motor"}, {"phase_generator_type": "linear"},
            {"basis_generator_type": "rbf"})
    with pytest.raises(ValueError):       # no RawInterfaceWrapper in the stack
        fancy_gym.make_bb("toy-v0", [], {}, *[dict(a) for a in args], device="cpu")
    with pytest.raises(ValueError):       # sub-trajectories and replanning are exclusive
        fancy_gym.make_bb("toy-v0", [ToyWrapper], {"learn_sub_trajectories": True, "replanning_schedule": lambda *a: True},
                          *[dict(a) for a in args], device="cpu")
    with pytest.raises(AssertionError):   # time_limit vs MP duration
        fancy_gym.make_bb("toy-v0", [ToyWrapper], {}, {"trajectory_generator_type": "promp", "duration": 2.0},
                          *[dict(a) for a in args[1:]], time_limit=1.0, device="cpu")
    # replanning adds the time-aware observation (make_env_helpers.py:94-97) and returns the full observation
    env = fancy_gym.make_bb("toy-v0", [ToyWrapper], {"replanning_schedule": lambda c_pos, c_vel, obs, c_action, t: t % 10 == 0},
                            *[dict(a) for a in args], device="cpu")
    assert env.do_replanning and env.observation_space.shape == (2,)
    # Q6: an explicit learn_sub_trajectories=False still switches learn_tau on
    env = fancy_gym.make_bb("toy-v0", [ToyWrapper], {"learn_sub_trajectories": False}, *[dict(a) for a in args], device="cpu")
    assert env.traj_gen.learn_tau and env.action_space.shape[0] == 1 + 10


def test_default_mp_wrapper_needs_pos_vel():
    from tests.toy import ToyEnv
    w = DefaultMPWrapper(ToyEnv(device="cpu"))
    assert np.all(w.context_mask)
    with pytest.raises(AssertionError):
        w.current_pos


def test_replanning_schedule_is_evaluated_on_the_host():
    args = ({"trajectory_generator_type": "prodmp"}, {"controller_type": "motor"}, {"phase_generator_type": "exp"},
            {"basis_generator_type": "prodmp"})
    env = fancy_gym.make_bb("toy-v0", [ToyWrapper], {"replanning_schedule": lambda c_pos, c_vel, obs, c_action, t: t % 10 == 0,
                                                     "max_planning_times": 3}, *[dict(a) for a in args], device="cpu")
    env.traj_gen.set_duration(env.duration, env.dt)
    assert env._segment_steps(env.traj_gen.n_steps) == (10, True)
    env.plan_steps = 3                                     # planning budget exhausted: run to the end
    assert env._segment_steps(env.traj_gen.n_steps) == (env.traj_gen.n_steps, False)


# ---- ragged sub-trajectories and the ring of result sets: host side (no kernel runs) ------------------------------
def test_ragged_plan_lengths_and_time_grids_follow_the_oracle():
    """learn_sub_trajectories with a different learned tau per env: env b plans round(tau_b / dt) points (clamped to 2 .. the
    longest admissible plan), buffers are sized for the longest plan, and row n of the per-length time-grid table is the
    float32 grid the oracle (and the library: torch.linspace) builds for an n-point plan — bit for bit."""
    import torch
    from oracle.mp import time_grid
    env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=6, device="cpu",
                         mp_config_override={"black_box_kwargs": {"learn_sub_trajectories": True}})
    tg = env.traj_gen
    P = env.action_space.shape[0]
    params = torch.zeros(6, P)
    params[:, 0] = torch.tensor([0.37, 0.8, 0.02, 2.0, 0.015, 1.234])
    tg.reset()
    tg.set_params(params)
    tg.set_duration(None, 0.01)
    t_max = int(round(float(tg.phase_gn.tau_bound[1]) / 0.01))
    assert tg.n_steps == t_max and tg.n_steps_env.dtype == torch.int32
    want = np.clip(np.round(params[:, 0].double().numpy() / 0.01), 2, t_max).astype(np.int32)
    assert np.array_equal(tg.n_steps_env.numpy(), want) and len(set(want.tolist())) > 3
    tab = tg._times_table().numpy()
    assert tab.shape == (t_max + 1, t_max) and tab.dtype == np.float32
    for n in (2, 37, 80, 123, t_max):
        ref = time_grid(float(n * 0.01), 0.01, 0.0, "mirror")
        assert np.array_equal(tab[n, :n], ref.astype(np.float32)) and not tab[n, n:].any()
    # equal learned taus collapse to the shared-table path: no per-env lengths
    params[:, 0] = 0.5
    tg.reset()
    tg.set_params(params)
    tg.set_duration(None, 0.01)
    assert tg.n_steps_env is None and tg.n_steps == 50


def test_result_set_ring():
    """what step() returns lives in a ring of result sets (two by default; more for consumers that lag several steps)"""
    with pytest.raises(ValueError):
        fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=2, device="cpu",
                       mp_config_override={"black_box_kwargs": {"result_sets": 1}})
    for n in (2, 4):
        env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=2, device="cpu",
                             mp_config_override={"black_box_kwargs": {"result_sets": n}})
        seen = []
        for _ in range(2 * n):
            env._flip_outputs()
            seen.append(env._ret.data_ptr())
            assert env._result_block.data_ptr() == env._out_sets[env._out_i]["block"].data_ptr()
        assert len(set(seen)) == n and seen[:n] == seen[n:]


# ---- re-planning schedules, plans laid out in advance, bounded handle cache, device median: host side ----------------
def test_schedule_is_evaluated_once_and_plans_are_laid_out_like_the_reference_loop():
    """black_box_wrapper.py:197: a plan breaks at the next step the schedule fires on while plan_steps < max_planning_times"""
    calls = []

    def sched(pos, vel, obs, action, t):
        calls.append(t)
        return t % 25 == 0

    over = {"black_box_kwargs": {"replanning_schedule": sched, "max_planning_times": 4}}
    env = fancy_gym.make("fancy_ProDMP/SimpleReacher-v0", num_envs=3, device="cpu", mp_config_override=over)
    assert env._break_points() == [25, 50, 75, 100, 125, 150, 175, 200] and len(calls) == 200
    env.traj_gen.set_duration(env.duration, env.dt)
    for _ in range(5):
        env._segment_steps(200)
    assert len(calls) == 200                       # cached: no more host calls per step
    assert env.plan_schedule(4) == [(0, 25), (25, 25), (50, 25), (75, 200)]      # the 4th plan is the last allowed: no break
    env.current_traj_steps, env.plan_steps = 30, 1
    assert env.plan_schedule(2) == [(30, 20), (50, 25)]
    env.plan_steps = 0
    env.current_traj_steps = 190
    with pytest.raises(ValueError):
        env.plan_schedule(3)                       # 190 -> 200, then the episode is over
    free = fancy_gym.make("fancy_ProDMP/SimpleReacher-v0", num_envs=3, device="cpu",
                          mp_config_override={"black_box_kwargs": {"replanning_schedule": lambda p, v, o, a, t: t % 60 == 0}})
    assert free.plan_schedule(4) == [(0, 60), (60, 60), (120, 60), (180, 200)] and free._plans_fusable()


def test_state_dependent_schedule_is_detected():
    def sched(pos, vel, obs, action, t):
        return float(np.abs(vel).max()) > 1.0

    env = fancy_gym.make("fancy_ProDMP/SimpleReacher-v0", num_envs=1, device="cpu",
                         mp_config_override={"black_box_kwargs": {"replanning_schedule": sched}})
    assert env._break_points() is None and not env._plans_fusable()
    env.traj_gen.set_duration(env.duration, env.dt)
    with pytest.raises(NotImplementedError):
        env._segment_steps(200)
    env.schedule_host_callback = True
    assert env._segment_steps(200) == (None, True)


def test_handle_cache_is_bounded(monkeypatch):
    """a learned scalar tau gives a new table key almost every episode: the cache evicts the least recently used handle"""
    from fancy_gym_b200 import _lib
    env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=1, device="cpu",
                         mp_config_override={"black_box_kwargs": {"max_cached_plans": 3}})
    destroyed = []
    monkeypatch.setattr(_lib.lib, "fg_destroy", lambda h: destroyed.append(h) or 0)
    for i in range(5):
        env._remember_handle(("k", i), f"h{i}")
    assert list(env._handles) == [("k", 2), ("k", 3), ("k", 4)] and destroyed == ["h0", "h1"]
    env._handles.clear()


def test_masked_median_equals_numpy():
    import torch
    from fancy_gym_b200.black_box.black_box_wrapper import _masked_median
    rng = np.random.default_rng(0)
    r = rng.standard_normal((64, 50))
    r[3, :4] = -np.inf
    L = rng.integers(0, 51, size=64)
    got = _masked_median(torch.as_tensor(r), torch.as_tensor(L)).numpy()
    want = np.array([np.median(r[b, :L[b]]) if L[b] else 0.0 for b in range(64)])
    assert np.array_equal(got, want)


def test_ragged_plans_need_a_finite_tau_bound():
    """a phase generator built without make_bb has tau_bound = [1e-5, inf]: a clear ValueError instead of an OverflowError"""
    import torch
    from fancy_gym_b200 import mp
    pg = mp.LinearPhaseGenerator(tau=2.0, learn_tau=True)
    bg = mp.NormalizedRBFBasisGenerator(pg, num_basis=5)
    tg = mp.ProMP(bg, 2, device="cpu")
    p = torch.zeros(3, tg.num_params)
    p[:, 0] = torch.tensor([0.3, 0.5, 0.7])
    tg.set_params(p)
    with pytest.raises(ValueError, match="tau_bound"):
        tg.set_duration(None, 0.01)


def test_rbf_recurrence_error_stays_far_inside_the_tie_margin():
    """fg_device.cuh RbfRec (restated in numpy): normalised RBFs at a linear phase by phi_{k+1} = phi_k * r_k with a geometric
    ratio — the float64 values stay within a few hundred ulps of the direct evaluation, the kernels fall back to the direct
    evaluation within 2**12 ulps of a float32 rounding boundary: the float32 basis cannot change."""
    import numpy as np
    from fancy_gym_b200.mp.phase_gn import LinearPhaseGenerator
    from fancy_gym_b200.mp.basis_gn import ZeroPaddingNormalizedRBFBasisGenerator as Z
    for kw in (dict(num_basis=5, num_basis_zero_start=1), dict(num_basis=5, num_basis_zero_start=0), dict(num_basis=7, num_basis_zero_start=1)):
        bg = Z(LinearPhaseGenerator(tau=2.0, delay=0.0, learn_tau=True, learn_delay=True), basis_bandwidth_factor=3.0, **kw)
        cen, bw = np.asarray(bg.centers_p, np.float64), np.asarray(bg.bandwidth, np.float64)
        n = cen.size
        L = np.longdouble
        A = -(L(bw[1:]) - L(bw[:-1])) / 2
        Bc = L(bw[1:]) * L(cen[1:]) - L(bw[:-1]) * L(cen[:-1])
        C = -(L(bw[1:]) * L(cen[1:]) ** 2 - L(bw[:-1]) * L(cen[:-1]) ** 2) / 2
        assert abs(A[0]) < 1e-9 and np.all(np.abs(np.diff(A)) + np.abs(np.diff(Bc)) < 1e-9)      # what the host checks
        q = np.exp(np.diff(C)).astype(np.float64)
        da, db = np.diff(A).astype(np.float64), np.diff(Bc).astype(np.float64)
        a0, b0, c0 = float(A[0]), float(Bc[0]), float(C[0])
        p = np.float32(np.random.default_rng(0).random(200_000)).astype(np.float64)              # the phase is a float32 value
        direct = np.exp(-((p[:, None] - cen) ** 2 * bw) / 2)
        phi = np.empty_like(direct)
        phi[:, 0] = direct[:, 0]
        r = np.exp(b0 * p + c0)
        r = r + r * (a0 * p * p)
        for k in range(n - 1):
            phi[:, k + 1] = phi[:, k] * r
            if k + 2 < n:
                rq = r * q[k]
                r = rq + rq * ((da[k] * p + db[k]) * p)
        direct /= direct.sum(1, keepdims=True)
        phi /= phi.sum(1, keepdims=True)
        rel = np.abs(phi - direct) / direct
        assert rel.max() < 2.0 ** -40 / 8, rel.max()          # margin of the fall-back: 2**12 ulps = 2**-40 relative


# ---- link counts the step kernels exist for ---------------------------------------------------------------------------
def test_step_link_range_is_checked_on_the_host():
    from fancy_gym_b200 import _lib
    for kind in (_lib.ENV_HOLE_REACHER, _lib.ENV_VIAPOINT_REACHER, _lib.ENV_SIMPLE_REACHER):
        for n in range(1, _lib.FG_MAX_DOF + 1):
            if n in _lib.STEP_LINKS:
                _lib.check_step_links(kind, n)
            else:
                with pytest.raises(NotImplementedError, match=r"n_links=%d: .* 2\.\.7 links" % n):
                    _lib.check_step_links(kind, n)
    _lib.check_step_links(_lib.ENV_TOY, 1)          # the test env has its own instantiations (1, 2, 5)
