"""GPU tests of the decisions that end an episode (joint limits, self collision, wall) at constructed boundaries
(tests/boundary_cases.py), and of non-finite joint angles, actions and ProMP weights against the oracle.

State injection: reset the env, overwrite q and ctx with a constructed state (v = 0, steps = 0), then take one step that
does not move the arm: env.step with a float64 zero action (q + dt * 0 == q), or a fused ProMP rollout with all-zero
weights (a zero action on every step: length 1 means the first step collided, 200 that no step did).

Error bands.  Wall (fg_device.cuh wall_collision): every sample coordinate the device compares is float32.  A link's
c, s come from the float64-reduced angle within 2 * 2^-24 each (N links: 2N * 2^-24 on a joint's coordinate); the joint
coordinate k is a float32 running sum, k additions of values <= k, each rounded by <= 1/2 ulp (sum over k <= N:
N(N+1)/2 * 2^-24 at most); the sample is one fma per coordinate (1/2 ulp of a value <= N: N * 2^-24); s_m is float32(linspace)
(|c| * 2^-25 * 2 for both coordinates: 2^-24); the hole edge / floor is rounded to float32 once (1/2 ulp of a value
<= 4: 2 * 2^-24, + 1 for the base).  Collected with the rounding of the float64 reference itself (< 2^-40):
    beta_wall(N) = 2^-24 * (N^2 / 2 + 4.5 N + 4)        (0.9e-6 at N = 2, 3.6e-6 at N = 7)
in the oracle's absolute margin unit.  Self collision (links_intersect): an orientation value is a float32 sum of <= N
sines of relative link angles, each within 2 * 2^-24 relative (accurate path) or formed as sn cs - cs sn from values
within 2^-24 (fast path, taken only when every value is farther than 8e-6 from zero), plus <= N roundings of the sum:
    beta_self(N) = 4 (N + 1) * 2^-24
relative to sum |sin|, the oracle's margin unit.  Where the oracle margin exceeds beta the device must take the oracle's
decision; inside beta it may take either (the resolution is printed).  Joint limits compare the float64 q itself, which is
bit-identical on both sides: exact, no band.
"""
import numpy as np
import pytest
import torch

from tests import boundary_cases as bc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CTX = {"HoleReacher-v0": np.array([2.0, 0.5, 1.0, 0.0]), "ViaPointReacher-v0": np.array([1.0, 1.0, 2.0, 2.0])}


def _fg():
    import fancy_gym_b200 as fancy_gym
    return fancy_gym


def _inject(base, q, ctx):
    base.q.copy_(torch.as_tensor(q, device=DEV))
    base.ctx.copy_(torch.as_tensor(ctx, device=DEV))
    base.v.zero_()
    base.steps.zero_()


def step_env_collided(name, n, q, ctx, **over):
    """is_collided of one env.step with a float64 zero action from the injected state; q must come back unchanged"""
    fg = _fg()
    B = len(q)
    env = fg.make(f"fancy/{name}", num_envs=B, device=DEV, n_links=n, **over)
    env.reset(seed=0)
    _inject(env, q, ctx)
    _, _, te, _, info = env.step(torch.zeros(B, n, dtype=torch.float64, device=DEV))
    got_q = env.q.cpu().numpy()
    assert np.array_equal(got_q, q, equal_nan=True)
    col = info["is_collided"].cpu().numpy()
    assert np.array_equal(te.cpu().numpy(), col)
    return col


def rollout_collided(name, n, q, ctx, wall_mode=0, **over):
    """(collided on the first step, all outputs) of a fused ProMP rollout with all-zero weights from the injected state"""
    fg = _fg()
    B = len(q)
    env = fg.make(f"fancy_ProMP/{name}", num_envs=B, device=DEV, n_links=n,
                  mp_config_override={"black_box_kwargs": {"wall_mode": wall_mode}}, **over)
    env.reset(seed=0)
    _inject(env.unwrapped, q, ctx)
    obs, ret, te, tr, info = env.step(torch.zeros(B, env.action_space.shape[0], device=DEV))
    length = info["trajectory_length"].cpu().numpy()
    te, tr = te.cpu().numpy(), tr.cpu().numpy()
    assert np.isin(length, (1, 200)).all() and np.array_equal(te, length == 1) and np.array_equal(tr, length == 200)
    return length == 1, [x.cpu().numpy() for x in (obs, ret, info["trajectory_length"])] + [te, tr]


def _oracle_decision(q):
    from oracle.reacher import forward_kinematics, self_collision
    with np.errstate(all="ignore"):
        return self_collision(q, forward_kinematics(q), margins=False)[0]


def _report(what, kernel, hit, m, beta):
    """decisions must agree where |margin| > beta; print how the cases inside the band were resolved"""
    out = np.abs(m) > beta
    bad = out & (kernel != hit)
    inside = ~out
    print(f"{what}: {int(out.sum())} cases outside beta={beta:.3g}, {int(inside.sum())} inside: "
          f"{int((kernel == hit)[inside].sum())} as the oracle, {int((kernel != hit)[inside].sum())} the other way")
    return bad


# --------------------------------------------------------------------------------------------
# joint limits: exact
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["HoleReacher-v0", "ViaPointReacher-v0"])
@pytest.mark.parametrize("n", range(2, 8))
def test_joint_limits_are_exact(name, n):
    """any(q > pi) | any(q < -pi) of numpy (NaN is not a limit; +-inf and |q| >= 2^1017 are) combined with the oracle's
    pair decision, with no tie window, on both the step env and the fused rollout"""
    over = dict(allow_wall_collision=True) if name == "HoleReacher-v0" else {}
    c = bc.joint_limit_cases(n, CTX[name])
    want = _oracle_decision(c["q"])
    assert np.array_equal(want & ~bc.joint_limit_decision(c["q"]), np.zeros_like(want))    # the pairs never decide here
    got_step = step_env_collided(name, n, c["q"], c["ctx"], **over)
    got_roll, _ = rollout_collided(name, n, c["q"], c["ctx"], **over)
    for path, got in (("step", got_step), ("rollout", got_roll)):
        bad = got != want
        assert not bad.any(), (path, list(c["label"][bad]))


# --------------------------------------------------------------------------------------------
# wall: the four modes bit-identical, the float64 decision outside beta
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", range(2, 8))
def test_wall_decisions_at_constructed_boundaries(n):
    c = bc.wall_cases(n)
    q, ctx = c["q"], c["ctx"]
    over = dict(allow_self_collision=True)
    outs = [rollout_collided("HoleReacher-v0", n, q, ctx, wall_mode=mode, **over) for mode in (0, 1, 2, 3)]
    for mode, (col, o) in zip((1, 2, 3), outs[1:]):
        bad = col != outs[0][0]
        assert not bad.any(), (mode, list(c["label"][bad]))
        for a, b in zip(outs[0][1], o):
            assert np.array_equal(a, b, equal_nan=True), mode
    kernel = outs[0][0]
    assert np.array_equal(step_env_collided("HoleReacher-v0", n, q, ctx, **over), kernel)
    hit, m = bc.wall_signed(q, ctx)
    beta = bc.beta_wall(n)
    assert ((np.abs(m) > beta) & (np.abs(m) <= 4 * beta)).sum() >= 50
    bad = _report(f"wall n={n}", kernel, hit, m, beta)
    assert not bad.any(), [(lbl, d) for lbl, d in zip(c["label"][bad], m[bad])]


# --------------------------------------------------------------------------------------------
# self collision: the float64 decision outside beta, on both paths
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["HoleReacher-v0", "ViaPointReacher-v0"])
@pytest.mark.parametrize("n", range(3, 8))
def test_self_collision_at_constructed_boundaries(name, n):
    from oracle.reacher import CCW_EPS, _cross, forward_kinematics
    over = dict(allow_wall_collision=True) if name == "HoleReacher-v0" else {}
    c = bc.self_cases(n, CTX[name])
    q = c["q"]
    hit, m = bc.self_signed(q)
    # where the reference's own float64 noise decides (an orientation value within 2^-44 of 1e-12): a tie by construction
    J = forward_kinematics(q)
    noise = np.zeros(len(q), bool)
    for i in range(n):
        for j in range(i + 2, n):
            for cv in (_cross(J[:, i], J[:, j], J[:, j + 1]), _cross(J[:, i + 1], J[:, j], J[:, j + 1]),
                       _cross(J[:, i], J[:, i + 1], J[:, j]), _cross(J[:, i], J[:, i + 1], J[:, j + 1])):
                noise |= np.abs(cv - CCW_EPS) < 2.0 ** -44
    fold = np.char.startswith(c["label"].astype(str), "self fold")     # margin | |q| - pi | = 0: exact by construction
    m = np.where(noise & ~fold, 0.0, np.where(fold, np.inf, m))
    beta = bc.beta_self(n)
    assert ((np.abs(m) > beta) & (np.abs(m) <= 4 * beta)).sum() >= 20
    for path, got in (("step", step_env_collided(name, n, q, c["ctx"], **over)),
                      ("rollout", rollout_collided(name, n, q, c["ctx"], **over)[0])):
        bad = _report(f"self {name} n={n} {path}", got, hit, m, beta)
        assert not bad.any(), [(lbl, d) for lbl, d in zip(c["label"][bad], m[bad])]


# --------------------------------------------------------------------------------------------
# non-finite actions (step env) and ProMP weights (fused rollout) against the oracle
# --------------------------------------------------------------------------------------------
def _same(a, b, rtol):
    """equal within rtol, NaN == NaN, +-inf exactly"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    fin = np.isfinite(b)
    ok = np.where(fin, np.abs(a - b) <= rtol * np.maximum(1.0, np.abs(b)), (a == b) | (np.isnan(a) & np.isnan(b)))
    return ok


def _nonfinite_rows(B, n, rng, sigma):
    a = sigma * rng.standard_normal((B, n))
    vals = (np.inf, -np.inf, np.nan)
    for b in range(B):
        a[b, b % n] = vals[(b // n) % 3]
    return a


@pytest.mark.parametrize("name", ["HoleReacher-v0", "ViaPointReacher-v0", "SimpleReacher-v0"])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_step_env_non_finite_actions_match_oracle(name, dtype):
    from tests.test_gpu_step_env import _oracle_for
    fg = _fg()
    B = 96
    env = fg.make(f"fancy/{name}", num_envs=B, device=DEV)
    env.reset(seed=3)
    orc = _oracle_for(env, name, {})
    n = env.n_links
    rng = np.random.default_rng(0)
    acts = [(0.3 * rng.standard_normal((B, n))).astype(dtype), _nonfinite_rows(B, n, rng, 0.3).astype(dtype),
            (0.3 * rng.standard_normal((B, n))).astype(dtype)]
    for t, a in enumerate(acts):
        ob, r, te, tr, info = env.step(a)
        with np.errstate(all="ignore"):
            o_ob, o_r, o_te, o_info = orc.step(a)
        assert _same(ob.cpu().numpy(), o_ob, 1e-5).all(), t
        assert _same(r.cpu().numpy(), o_r, 1e-5).all(), (t, np.nonzero(~_same(r.cpu().numpy(), o_r, 1e-5))[0][:8])
        assert np.array_equal(te.cpu().numpy(), o_te), (t, np.nonzero(te.cpu().numpy() != o_te)[0][:8])
        if "is_collided" in info:
            assert np.array_equal(info["is_collided"].cpu().numpy(), o_info["is_collided"]), t
        assert np.array_equal(env.q.cpu().numpy(), orc.q, equal_nan=True), t


_POS = {"controller_kwargs": {"controller_type": "position"}}
NONFINITE_ROLLOUTS = [("fancy_ProMP/HoleReacher-v0", {}), ("fancy_ProMP/ViaPointReacher-v0", _POS),
                      ("fancy_ProMP/SimpleReacher-v0", {})]


@pytest.mark.parametrize("env_id,mp_over", NONFINITE_ROLLOUTS, ids=["velocity", "position", "pd"])
def test_rollout_non_finite_weights_match_oracle(env_id, mp_over):
    """NaN / +-inf ProMP weights: the controller's clip keeps a NaN (np.clip does), so a diverged search sees NaN returns"""
    from oracle.blackbox import make_oracle
    fg = _fg()
    B = 150
    env = fg.make(env_id, num_envs=B, device=DEV, mp_config_override=mp_over)
    env.reset(seed=100)
    P = env.action_space.shape[0]
    rng = np.random.default_rng(5)
    params = _nonfinite_rows(B, P, rng, 0.5).astype(np.float32)
    params[-6:] = (0.5 * rng.standard_normal((6, P))).astype(np.float32)        # finite rows next to them
    obs, ret, te, tr, info = env.step(torch.as_tensor(params, device=DEV))
    ret, te, tr = ret.cpu().numpy(), te.cpu().numpy(), tr.cpu().numpy()
    length = info["trajectory_length"].cpu().numpy()
    orc = make_oracle(env_id, mode="mirror", mp_overrides={"ctrl": mp_over.get("controller_kwargs", {})})
    orc.reset(seeds=100 + np.arange(B))
    with np.errstate(all="ignore"):
        o_obs, o_ret, o_te, o_tr, o_info = orc.step(params)
    tie = o_info["min_margin"] < 1e-5             # (NaN margins are not ties)
    agree = (length == o_info["trajectory_length"]) & (te == o_te) & (tr == o_tr)
    assert (agree | tie).all(), np.nonzero(~(agree | tie))[0][:10]
    same = _same(ret, o_ret, 1e-5)
    assert (same | ~agree).all(), [(b, ret[b], o_ret[b]) for b in np.nonzero(~same & agree)[0][:8]]
    assert np.isnan(o_ret).sum() >= B // 4 and np.array_equal(np.isnan(ret)[agree], np.isnan(o_ret)[agree])
