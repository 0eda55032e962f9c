"""Link counts the reacher step kernels are not instantiated for (1 and 8; `_lib.STEP_LINKS` = 2..7).  The envs can be made
and reset at every count 1..FG_MAX_DOF, and their stand-alone trajectories are generated; a step is refused with
NotImplementedError before anything changes, so the env stays usable."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.blackbox import make_oracle  # noqa: E402
from tests.golden.make_golden import n_params_of  # noqa: E402

DEV = "cuda:0"
NAMES = ("HoleReacher-v0", "ViaPointReacher-v0", "SimpleReacher-v0")
OUTSIDE = (1, 8)
_CTX_OBS = {"HoleReacher-v0": 4, "ViaPointReacher-v0": 5, "SimpleReacher-v0": 3}       # task entries + step counter


def _fg():
    import fancy_gym_b200 as fancy_gym
    return fancy_gym


def _bb_state(env):
    base = env.unwrapped
    return dict(plan_steps=env.plan_steps, current_traj_steps=env.current_traj_steps, out_i=env._out_i,
                ret=env._ret.data_ptr(), q=base.q.clone(), v=base.v.clone(), steps=base.steps.clone(), done=base.done.clone())


def _env_state(env):
    ring = [s["obs"].data_ptr() for s in env._step_sets] if env._step_sets is not None else None
    return dict(ring=ring, q=env.q.clone(), v=env.v.clone(), steps=env.steps.clone(), done=env.done.clone(),
                dtype=env._last_action_dtype)


def _assert_same(before, after):
    for k, x in before.items():
        y = after[k]
        assert (torch.equal(x, y) if torch.is_tensor(x) else x == y), k


@pytest.mark.parametrize("n", OUTSIDE)
@pytest.mark.parametrize("name", NAMES)
def test_make_and_reset(name, n):
    fancy_gym = _fg()
    B = 300
    env = fancy_gym.make(f"fancy/{name}", num_envs=B, device=DEV, n_links=n)
    obs, _ = env.reset(seed=3)
    assert obs.shape == (B, 3 * n + _CTX_OBS[name]) and env.q.shape == (B, n)
    assert int(env.steps.abs().max()) == 0 and bool((env.q[:, 1:] == 0).all())
    for mp in ("ProMP", "DMP", "ProDMP"):
        bb = fancy_gym.make(f"fancy_{mp}/{name}", num_envs=B, device=DEV, n_links=n)
        obs, _ = bb.reset(seed=3)
        assert obs.shape == (B, bb.observation_space.shape[0])
        assert bb.action_space.shape[0] == n_params_of(f"fancy_{mp}/{name}", {"env": dict(n_links=n)})


@pytest.mark.parametrize("n", OUTSIDE)
@pytest.mark.parametrize("name", NAMES)
def test_refused_step_changes_nothing(name, n):
    """black-box step(), step_plans() and the step-based step() raise NotImplementedError naming the instantiated range and
    leave the plan counters, the env state and the result buffers as they were; another env steps afterwards"""
    fancy_gym = _fg()
    B = 64
    over = {"black_box_kwargs": dict(replanning_schedule=lambda p, v, o, a, t: t % 50 == 0)}
    for mp_over, call in (({}, "step"), (over, "step_plans")):
        bb = fancy_gym.make(f"fancy_ProMP/{name}", num_envs=B, device=DEV, n_links=n, mp_config_override=mp_over)
        bb.reset(seed=1)
        P = bb.action_space.shape[0]
        before = _bb_state(bb)
        with pytest.raises(NotImplementedError, match=r"2\.\.7"):
            if call == "step":
                bb.step(torch.zeros(B, P, device=DEV))
            else:
                bb.step_plans(torch.zeros(B, 2, P, device=DEV))
        _assert_same(before, _bb_state(bb))
    env = fancy_gym.make(f"fancy/{name}", num_envs=B, device=DEV, n_links=n)
    env.reset(seed=1)
    before = _env_state(env)
    with pytest.raises(NotImplementedError, match=r"2\.\.7"):
        env.step(torch.zeros(B, n, device=DEV))
    _assert_same(before, _env_state(env))
    torch.cuda.synchronize()

    # the next valid calls, on envs of an instantiated link count
    ok = fancy_gym.make(f"fancy_ProMP/{name}", num_envs=B, device=DEV)
    ok.reset(seed=1)
    obs, ret, te, tr, info = ok.step(torch.zeros(B, ok.action_space.shape[0], device=DEV))
    assert bool((info["trajectory_length"] == 200).all()) and bool(tr.all()) and not bool(torch.isnan(ret).any())
    step_env = fancy_gym.make(f"fancy/{name}", num_envs=B, device=DEV)
    step_env.reset(seed=1)
    step_env.step(torch.zeros(B, step_env.n_links, device=DEV))
    assert int(step_env.steps.min()) == 1
    torch.cuda.synchronize()


@pytest.mark.parametrize("n", OUTSIDE)
@pytest.mark.parametrize("mp", ["ProMP", "DMP", "ProDMP"])
def test_trajectory_matches_the_oracle(mp, n):
    """fg_trajgen takes 1..FG_MAX_DOF links: bit for bit the oracle's mirror mode (the kernel's specification)"""
    fancy_gym = _fg()
    env_id = f"fancy_{mp}/HoleReacher-v0"
    B = 257
    env = fancy_gym.make(env_id, num_envs=B, device=DEV, n_links=n)
    env.reset(seed=0)
    params = (0.7 * np.random.default_rng(3).standard_normal((B, env.action_space.shape[0]))).astype(np.float32)
    pos, vel = env.get_trajectory(torch.as_tensor(params, device=DEV))
    orc = make_oracle(env_id, mode="mirror", mp_overrides={"env": dict(n_links=n)})
    orc.reset(seeds=range(B))
    o_pos, o_vel = orc.get_trajectory(params)
    assert pos.shape == (B, 200, n)
    assert np.array_equal(pos.cpu().numpy(), o_pos), np.abs(pos.cpu().numpy() - o_pos).max()
    assert np.array_equal(vel.cpu().numpy(), o_vel), np.abs(vel.cpu().numpy() - o_vel).max()
