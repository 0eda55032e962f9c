"""Re-planning inside one launch (BlackBoxWrapper.step_plans / fg_rollout_io.n_plans), the env adaptor's trajectory hooks,
state-dependent schedules evaluated on the host, device-side median aggregation, and episode boundaries of learned tau /
delay (reference: fancy_gym/black_box/black_box_wrapper.py:150-217, :222-229; raw_interface_wrapper.py:55-121)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.blackbox import make_oracle  # noqa: E402
from tests.golden.make_golden import BB_CASES, bb_case, mp_config_override_of  # noqa: E402

DEV = "cuda:0"
_R25 = dict(replanning_schedule=lambda p, v, o, a, t: t % 25 == 0, max_planning_times=4)
PLAN_CASES = [
    ("fancy_ProDMP/SimpleReacher-v0", dict(_R25, condition_on_desired=False), {}, 4, 1.0),
    ("fancy_ProDMP/SimpleReacher-v0", dict(_R25, condition_on_desired=True), {}, 4, 1.0),
    ("fancy_ProDMP/SimpleReacher-v0", dict(replanning_schedule=lambda p, v, o, a, t: t % 25 == 0), {}, 8, 1.0),
    ("fancy_ProMP/HoleReacher-v0", dict(replanning_schedule=lambda p, v, o, a, t: t % 50 == 0), {}, 4, 0.5),
    ("fancy_DMP/HoleReacher-v0", dict(replanning_schedule=lambda p, v, o, a, t: t % 40 == 0, condition_on_desired=True), {}, 5, 0.3),
    ("fancy_ProDMP/HoleReacher-v0", dict(replanning_schedule=lambda p, v, o, a, t: t % 60 == 0, condition_on_desired=True),
     dict(rew_fct="unbounded"), 4, 0.5),
    ("fancy_DMP/ViaPointReacher-v0", dict(replanning_schedule=lambda p, v, o, a, t: t % 30 == 0, max_planning_times=3), {}, 3, 1.0),
    ("fancy_ProMP/SimpleReacher-v0", dict(replanning_schedule=lambda p, v, o, a, t: t % 64 == 0, reward_aggregation=np.mean), {}, 4, 0.5),
]
# plans inside one launch at link counts other than the registered ones: every env, re-planning with condition_on_desired
PLAN_CASES += [(env_id, dict(replanning_schedule=lambda p, v, o, a, t: t % 40 == 0, condition_on_desired=True), dict(n_links=n), 5, 0.5)
               for env_id in ("fancy_DMP/HoleReacher-v0", "fancy_DMP/ViaPointReacher-v0", "fancy_ProDMP/SimpleReacher-v0")
               for n in (3, 7)]


def _eq(a, b):
    a, b = a.double(), b.double()
    return torch.equal(torch.nan_to_num(a, neginf=-1e300), torch.nan_to_num(b, neginf=-1e300))


@pytest.mark.parametrize("env_id,bbk,env_kw,n_plans,sigma", PLAN_CASES, ids=[f"{c[0]}-{i}" for i, c in enumerate(PLAN_CASES)])
def test_plans_in_one_launch_equal_one_launch_per_plan(env_id, bbk, env_kw, n_plans, sigma):
    """step_plans(actions[B, n, P]) == n calls of step(actions[:, j]), bit for bit, including envs whose episode ends in the
    middle (frozen afterwards) and the state the env is left in"""
    import fancy_gym_b200 as fancy_gym
    B = 1000 + 19
    over = {"black_box_kwargs": dict(bbk)}
    seq = fancy_gym.make(env_id, num_envs=B, device=DEV, mp_config_override=over, **env_kw)
    one = fancy_gym.make(env_id, num_envs=B, device=DEV, mp_config_override=over, **env_kw)
    assert one._plans_fusable()
    seq.reset(seed=11)
    one.reset(seed=11)
    gen = torch.Generator(device=DEV).manual_seed(2)
    P = seq.action_space.shape[0]
    actions = sigma * torch.randn(B, n_plans, P, generator=gen, device=DEV)
    obs, ret, te, tr, info = one.step_plans(actions)
    assert obs.shape[:2] == (n_plans, B) and ret.shape == (n_plans, B)
    for j in range(n_plans):
        s_obs, s_ret, s_te, s_tr, s_info = seq.step(actions[:, j])
        assert torch.equal(info["trajectory_length"][j], s_info["trajectory_length"]), j
        assert torch.equal(te[j], s_te) and torch.equal(tr[j], s_tr), j
        assert _eq(ret[j], s_ret) and torch.equal(obs[j], s_obs), j
        for k in ("is_success", "is_collided", "end_effector", "reward_dist", "reward_ctrl"):
            if k in s_info:
                assert _eq(info[k][j], s_info[k]), (j, k)
    assert torch.equal(one.unwrapped.q, seq.unwrapped.q) and torch.equal(one.unwrapped.v, seq.unwrapped.v)
    assert torch.equal(one.unwrapped.steps, seq.unwrapped.steps) and torch.equal(one.unwrapped.done, seq.unwrapped.done)
    assert one.current_traj_steps == seq.current_traj_steps and one.plan_steps == seq.plan_steps
    assert int(info["trajectory_length"].sum(0).max()) <= 200
    if "HoleReacher" in env_id:
        assert bool(te.any()) and bool((info["trajectory_length"] == 0).any())     # some episodes ended early: frozen rows


def test_plans_then_single_steps_continue_the_episode():
    """two plans fused, the rest of the episode with ordinary step() calls == all ordinary"""
    import fancy_gym_b200 as fancy_gym
    B = 515
    over = {"black_box_kwargs": dict(replanning_schedule=lambda p, v, o, a, t: t % 25 == 0, condition_on_desired=True)}
    a_env = fancy_gym.make("fancy_ProDMP/SimpleReacher-v0", num_envs=B, device=DEV, mp_config_override=over)
    b_env = fancy_gym.make("fancy_ProDMP/SimpleReacher-v0", num_envs=B, device=DEV, mp_config_override=over)
    a_env.reset(seed=3); b_env.reset(seed=3)
    gen = torch.Generator(device=DEV).manual_seed(0)
    acts = torch.randn(B, 8, 12, generator=gen, device=DEV)
    b_env.step_plans(acts[:, :2])
    b_env.step_plans(acts[:, 2:5])
    for j in range(8):
        ra = a_env.step(acts[:, j])
        if j >= 5:
            rb = b_env.step(acts[:, j])
            assert torch.equal(ra[0], rb[0]) and _eq(ra[1], rb[1]) and torch.equal(ra[3], rb[3])
    assert torch.equal(a_env.unwrapped.q, b_env.unwrapped.q)


REPLAN_GOLDENS = [c for c in BB_CASES if "replan" in c[0]]


@pytest.mark.parametrize("case", REPLAN_GOLDENS, ids=[c[0] for c in REPLAN_GOLDENS])
def test_plans_in_one_launch_match_reference_goldens(case, golden_dir):
    """the re-planning goldens (generated by the reference's own BlackBoxWrapper, one step() per plan) through step_plans"""
    import fancy_gym_b200 as fancy_gym
    fname, env_id, seeds, bbk, env_over, mp_over = bb_case(case)
    g = np.load(os.path.join(golden_dir, fname + ".npz"))
    B = len(seeds)
    env = fancy_gym.make(env_id, num_envs=B, device=DEV, mp_config_override=mp_config_override_of(env_id, mp_over, dict(bbk)), **env_over)
    env.reset(seed=np.array(seeds))
    n_plans = int(g["n_calls"].max())
    obs, ret, te, tr, info = env.step_plans(torch.as_tensor(g["params"][:, :n_plans], device=DEV))
    obs, ret, te, tr = obs.cpu().numpy(), ret.cpu().numpy(), te.cpu().numpy(), tr.cpu().numpy()
    length = info["trajectory_length"].cpu().numpy()
    for b in range(B):
        for i in range(n_plans):
            if i >= g["n_calls"][b]:
                assert length[i, b] == 0
                continue
            assert length[i, b] == g["length"][b, i], (fname, b, i)
            assert bool(te[i, b]) == bool(g["terminated"][b, i]) and bool(tr[i, b]) == bool(g["truncated"][b, i])
            assert abs(ret[i, b] - g["ret"][b, i]) <= 2.2e-6 * max(1.0, abs(g["ret"][b, i]))
            assert (np.abs(obs[i, b] - g["obs"][b, i]) <= 4.8e-5 * np.maximum(1.0, np.abs(g["obs"][b, i]))).all()


# ---- trajectory hooks (black_box_wrapper.py:154-172) --------------------------------------------------------------------
def test_trajectory_hooks_are_called_and_invalid_trajectories_return_the_callback():
    import fancy_gym_b200 as fancy_gym
    from fancy_gym_b200.envs.classic_control.mp_wrappers import MPWrapper_HoleReacher
    calls = []

    class Hooked(MPWrapper_HoleReacher):
        def set_episode_arguments(self, action, pos_traj, vel_traj):
            calls.append("set")
            return pos_traj, vel_traj

        def preprocessing_and_validity_callback(self, action, pos_traj, vel_traj, tau_bound=None, delay_bound=None):
            calls.append("valid")
            ok = pos_traj.abs().amax(dim=(1, 2)) < 1.5           # a joint-limit style predicate over the PLANNED trajectory
            return ok, pos_traj, vel_traj

        def invalid_traj_callback(self, action, pos_traj, vel_traj, return_contextual_obs, tau_bound, delay_bound):
            calls.append("invalid")
            return torch.zeros(1), -7.5, False, True, {"note": "invalid"}

    B = 257
    env = fancy_gym.make_bb("fancy/HoleReacher-v0", [Hooked], {}, {"trajectory_generator_type": "promp", "weights_scale": 2},
                            {"controller_type": "velocity"}, {"phase_generator_type": "linear"},
                            {"basis_generator_type": "zero_rbf", "num_basis": 5, "num_basis_zero_start": 1, "basis_bandwidth_factor": 3.0},
                            device=DEV, num_envs=B)
    plain = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=B, device=DEV)
    env.reset(seed=4); plain.reset(seed=4)
    params = 0.6 * torch.randn(B, 25, generator=torch.Generator(device=DEV).manual_seed(1), device=DEV)
    pos, _ = plain.get_trajectory(params)
    ok = (pos.abs().amax(dim=(1, 2)) < 1.5)
    assert 0 < int(ok.sum()) < B
    obs, ret, te, tr, info = env.step(params)
    assert calls == ["set", "valid", "invalid"]
    p_obs, p_ret, p_te, p_tr, p_info = plain.step(params)
    assert torch.equal(info["trajectory_valid"], ok)
    # valid envs: exactly the plain env (the hooks returned the trajectory unchanged, tracked from HBM: same float32 values)
    assert _eq(ret[ok], p_ret[ok]) and torch.equal(obs[ok], p_obs[ok]) and torch.equal(te[ok], p_te[ok])
    assert torch.equal(info["trajectory_length"][ok], p_info["trajectory_length"][ok])
    # invalid envs: the callback's tuple, nothing executed, episode over
    inv = ~ok
    assert bool((ret[inv] == -7.5).all()) and not bool(te[inv].any()) and bool(tr[inv].all())
    assert bool((info["trajectory_length"][inv] == 0).all()) and bool((obs[inv] == 0).all())
    assert bool((env.unwrapped.steps[inv] == 0).all()) and bool((env.unwrapped.done[inv] == 1).all())
    assert info["note"] == "invalid"


def test_hooks_can_change_the_trajectory():
    """set_episode_arguments returns a modified trajectory: the rollout tracks what the hook returned"""
    import fancy_gym_b200 as fancy_gym
    from fancy_gym_b200.envs.classic_control.mp_wrappers import MPWrapper_SimpleReacher

    class Halved(MPWrapper_SimpleReacher):
        def set_episode_arguments(self, action, pos_traj, vel_traj):
            return 0.5 * pos_traj, 0.5 * vel_traj

    B = 64
    kw = ({"trajectory_generator_type": "promp"}, {"controller_type": "motor", "p_gains": 0.6, "d_gains": 0.075},
          {"phase_generator_type": "linear"}, {"basis_generator_type": "zero_rbf", "num_basis": 5, "num_basis_zero_start": 1,
                                               "basis_bandwidth_factor": 3.0})
    env = fancy_gym.make_bb("fancy/SimpleReacher-v0", [Halved], {"verbose": 2}, *[dict(k) for k in kw], device=DEV, num_envs=B)
    ref = fancy_gym.make_bb("fancy/SimpleReacher-v0", [MPWrapper_SimpleReacher], {"verbose": 2}, *[dict(k) for k in kw], device=DEV, num_envs=B)
    env.reset(seed=1); ref.reset(seed=1)
    p = torch.randn(B, 10, generator=torch.Generator(device=DEV).manual_seed(0), device=DEV)
    o1 = env.step(p)
    o2 = ref.step(0.5 * p)           # ProMP is linear in the weights: half the weights == half the trajectory
    assert torch.allclose(o1[4]["positions"], o2[4]["positions"], rtol=0, atol=2e-7)
    assert torch.allclose(o1[1], o2[1], rtol=1e-5, atol=1e-6)


# ---- state-dependent replanning schedule: host callback on request ------------------------------------------------------
def test_state_dependent_schedule_needs_the_flag_and_follows_the_oracle():
    import fancy_gym_b200 as fancy_gym

    def sched(pos, vel, obs, action, t):
        return bool(np.abs(np.asarray(vel)).max() > 1.2) or t % 70 == 0

    env_id = "fancy_ProDMP/SimpleReacher-v0"
    bad = fancy_gym.make(env_id, num_envs=1, device=DEV, mp_config_override={"black_box_kwargs": {"replanning_schedule": sched}})
    bad.reset(seed=0)
    with pytest.raises(NotImplementedError):
        bad.step(np.zeros(12, np.float32))
    env = fancy_gym.make(env_id, num_envs=1, device=DEV,
                         mp_config_override={"black_box_kwargs": {"replanning_schedule": sched, "schedule_host_callback": True}})
    orc = make_oracle(env_id, mode="mirror", replanning_schedule=sched)
    for seed in (0, 1, 2):
        env.reset(seed=seed)
        orc.reset(seeds=[seed])
        rng = np.random.default_rng(seed)
        total, lengths = 0, []
        for _ in range(12):
            a = rng.standard_normal(12).astype(np.float32)
            obs, ret, te, tr, info = env.step(a)
            o_obs, o_ret, o_te, o_tr, o_info = orc.step(a[None])
            assert info["trajectory_length"] == o_info["trajectory_length"][0]
            assert te == o_te[0] and tr == o_tr[0]
            assert abs(ret - o_ret[0]) <= 1e-5 * max(1.0, abs(o_ret[0]))
            assert np.abs(obs - o_obs[0]).max() <= 2e-5
            lengths.append(info["trajectory_length"])
            total += info["trajectory_length"]
            if te or tr:
                break
        assert total == 200 and len(set(lengths)) > 1          # the state-dependent part of the schedule fired somewhere


# ---- reward aggregation on the device -------------------------------------------------------------------------------
def test_median_aggregation_runs_on_the_device_and_equals_numpy():
    import fancy_gym_b200 as fancy_gym
    B = 2000
    env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=B, device=DEV,
                         mp_config_override={"black_box_kwargs": {"reward_aggregation": np.median}})
    dbg = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=B, device=DEV, mp_config_override={"black_box_kwargs": {"verbose": 2}})
    env.reset(seed=8); dbg.reset(seed=8)
    p = torch.randn(B, 25, generator=torch.Generator(device=DEV).manual_seed(5), device=DEV)
    ret = env.step(p)[1].cpu().numpy()
    info = dbg.step(p)[4]
    r, L = info["step_rewards"].cpu().numpy(), info["trajectory_length"].cpu().numpy()
    want = np.array([np.median(r[b, :L[b]]) for b in range(B)])
    assert np.array_equal(ret, want)
    assert len(set(L.tolist())) > 20


# ---- learned tau / delay across episode boundaries of the vector env (finalize / un-finalize) --------------------------
def test_vector_env_applies_the_learned_tau_of_every_new_episode():
    """reset_done() (the vector env's auto-reset) and evaluate() un-finalize the phase generator like reset() does
    (black_box_wrapper.py:226): the tau of EVERY episode / candidate is used, not the first one's for ever"""
    import fancy_gym_b200 as fancy_gym
    B = 8
    over = {"phase_generator_kwargs": {"phase_generator_type": "linear", "learn_tau": True}}
    venv = fancy_gym.make_vec("fancy_ProMP/HoleReacher-v0", num_envs=B, device=DEV, mp_config_override=over)
    venv.reset(seed=0)
    seen = []
    launch = venv.env.launch

    def spy(*a, **k):
        seen.append(float(venv.env.traj_gen.phase_gn.tau.reshape(-1)[0]))
        return launch(*a, **k)

    venv.env.launch = spy
    w = torch.zeros(B, 26, device=DEV)
    w[:, 1:] = 0.05
    for tau in (2.0, 0.5, 1.25):
        w[:, 0] = tau
        venv.step(w)
        assert not venv.env.traj_gen.phase_gn.is_finalized
    assert seen == [2.0, 0.5, 1.25]
    env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=B, device=DEV, mp_config_override=over)
    env.reset(seed=0)
    outs = []
    for tau in (2.0, 0.5):
        w[:, 0] = tau
        outs.append(env.evaluate(w)[1].clone())
        assert float(env.traj_gen.phase_gn.tau.reshape(-1)[0]) == tau
    assert not torch.equal(outs[0], outs[1])


# ---- per-env learned tau / delay evaluated inside the rollout (fg_rollout_io.phase) ---------------------------------------
_LIN_TAU_DELAY = {"phase_generator_kwargs": dict(phase_generator_type="linear", learn_tau=True, learn_delay=True)}
_EXP_TAU = {"phase_generator_kwargs": dict(phase_generator_type="exp", alpha_phase=2, learn_tau=True)}
FUSED_PHASE_CASES = [
    ("fancy_ProMP/HoleReacher-v0", _LIN_TAU_DELAY, {}, {}),
    ("fancy_ProMP/HoleReacher-v0", {"phase_generator_kwargs": dict(phase_generator_type="linear", learn_delay=True)}, {}, {}),
    ("fancy_DMP/ViaPointReacher-v0", _EXP_TAU, {}, {}),
    ("fancy_DMP/HoleReacher-v0", {"phase_generator_kwargs": dict(phase_generator_type="exp", alpha_phase=2.5, learn_tau=True, learn_delay=True)}, {}, {}),
    ("fancy_ProMP/SimpleReacher-v0", {"phase_generator_kwargs": dict(phase_generator_type="linear", learn_tau=True)}, {}, {}),
    ("fancy_DMP/LongSimpleReacher-v0", _EXP_TAU, {}, {}),
    ("fancy_ProMP/HoleReacher-v0", {}, {"learn_sub_trajectories": True}, {}),
    ("fancy_DMP/ViaPointReacher-v0", {}, {"learn_sub_trajectories": True, "condition_on_desired": True}, {}),
    # the in-rollout phase is instantiated for 5 and 2 links: the velocity-controlled envs at 2
    ("fancy_ProMP/HoleReacher-v0", _LIN_TAU_DELAY, {}, dict(n_links=2)),
    ("fancy_DMP/ViaPointReacher-v0", _EXP_TAU, {}, dict(n_links=2)),
]


@pytest.mark.parametrize("env_id,over,bbk,env_kw", FUSED_PHASE_CASES, ids=[f"{c[0]}-{i}" for i, c in enumerate(FUSED_PHASE_CASES)])
def test_phase_inside_the_rollout_equals_trajgen_then_rollout(env_id, over, bbk, env_kw, monkeypatch):
    """the basis of a per-env phase evaluated by the rollout thread itself == fg_trajgen_phase writing the trajectory to HBM and
    a FG_MP_TRAJ rollout reading it back: bit for bit, incl. ragged sub-trajectory plans and condition_on_desired"""
    import fancy_gym_b200 as fancy_gym
    B = 1000 + 7
    cfg = dict(over)
    if bbk:
        cfg["black_box_kwargs"] = dict(bbk)
    fused = fancy_gym.make(env_id, num_envs=B, device=DEV, mp_config_override=cfg, **env_kw)
    split = fancy_gym.make(env_id, num_envs=B, device=DEV, mp_config_override=cfg, **env_kw)
    assert fused._phase_fusable()
    fused.reset(seed=9); split.reset(seed=9)
    gen = torch.Generator(device=DEV).manual_seed(4)
    P = fused.action_space.shape[0]
    n_calls = 4 if bbk else 1
    for call in range(n_calls):
        p = 0.4 * torch.randn(B, P, generator=gen, device=DEV)
        ph = over.get("phase_generator_kwargs", {})
        i = 0
        if ph.get("learn_tau") or bbk:
            p[:, i] = (0.05 + 0.9 * torch.rand(B, generator=gen, device=DEV)) if bbk else (0.3 + 2.0 * torch.rand(B, generator=gen, device=DEV))
            i += 1
        if ph.get("learn_delay"):
            p[:, i] = 0.5 * torch.rand(B, generator=gen, device=DEV)
        monkeypatch.setenv("FG_PHASE_FUSED", "1")
        a = fused.step(p)
        monkeypatch.setenv("FG_PHASE_FUSED", "0")
        b = split.step(p)
        assert torch.equal(a[4]["trajectory_length"], b[4]["trajectory_length"]), call
        assert torch.equal(a[0], b[0]) and _eq(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), call
        assert torch.equal(fused.unwrapped.q, split.unwrapped.q) and torch.equal(fused.unwrapped.v, split.unwrapped.v)
    assert fused._traj_buf is None and split._traj_buf is not None        # the fused env never materialised a trajectory


@pytest.mark.parametrize("fused", [True, False])
def test_rbf_recurrence_leaves_the_float32_basis_unchanged(fused, monkeypatch):
    """linear phase, learned tau + delay per env: the two-exp recurrence for the normalised RBFs (with its fall-back to the
    direct evaluation next to a float32 rounding boundary) gives, bit for bit, what evaluating every RBF directly gives —
    inside the rollout and in the stand-alone trajectory kernel, 65 536 envs x 200 time points"""
    import fancy_gym_b200 as fancy_gym
    B = 65536
    over = {"phase_generator_kwargs": {"phase_generator_type": "linear", "learn_tau": True, "learn_delay": True}}
    env = fancy_gym.make("fancy_ProMP/HoleReacher-v0", num_envs=B, device=DEV, mp_config_override=over)
    gen = torch.Generator(device=DEV).manual_seed(11)
    p = 0.3 * torch.randn(B, env.action_space.shape[0], generator=gen, device=DEV)
    p[:, 0] = 0.3 + 2.0 * torch.rand(B, generator=gen, device=DEV)
    p[:, 1] = 0.5 * torch.rand(B, generator=gen, device=DEV)
    monkeypatch.setenv("FG_PHASE_FUSED", "1" if fused else "0")
    outs = []
    for direct in (False, True):
        if direct:
            monkeypatch.setenv("FG_PHASE_NO_RECURRENCE", "1")
        else:
            monkeypatch.delenv("FG_PHASE_NO_RECURRENCE", raising=False)
        env.reset(seed=5)
        o = env.step(p)
        outs.append((o[0].clone(), o[1].clone(), o[4]["trajectory_length"].clone(),
                     None if fused else (env._traj_buf[0].clone(), env._traj_buf[1].clone())))
    a, b = outs
    assert torch.equal(a[2], b[2]) and torch.equal(a[0], b[0]) and _eq(a[1], b[1])
    if not fused:
        assert torch.equal(a[3][0], b[3][0]) and torch.equal(a[3][1], b[3][1])          # positions / velocities [B, T, dof]
        assert float(a[3][0].abs().max()) > 0.1
