"""GPU tests of the step-based envs (`fancy/<Name>-v0`: BaseReacherEnv.step, fg_env_step) and of their vector env:
against the reference's own per-step records, bit for bit against the fused rollout's per-step outputs, against the oracle
at scale, and for what graph capture needs (no host synchronisation, identical replays)."""
import json
import os

import numpy as np
import pytest
import torch

from tests.golden.make_golden import ENV_CASES

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TIE_EPS = 1e-5


def _fg():
    import fancy_gym_b200 as fancy_gym
    return fancy_gym


def rel_err(a, b, scale=1.0):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), scale)


# --------------------------------------------------------------------------------------------
# 1. the reference's env classes, step by step (tests/golden/env_kat.npz)
# --------------------------------------------------------------------------------------------
# 2x the largest errors measured on a B200 (profiles/step_env_golden_errors.json, written by this test with
# FG_STEP_GOLDEN_ERRORS_JSON=<file>).  The joint angles are bit-identical to the reference's (the dynamics are float
# additions and products in the reference's dtypes); what is left is CUDA's float64 sin / cos against glibc's in the end
# effector.  Measured: every observation bit-identical, rewards within 3.7e-16 relative (two float64 ulps of a distance
# term).
STEP_GOLDEN_TOL = dict(obs=0.0, reward=7.5e-16)
_golden_err = {}


@pytest.mark.parametrize("case", ENV_CASES, ids=[c[0] for c in ENV_CASES])
def test_step_env_matches_reference_env_records(case, golden_dir):
    fg = _fg()
    key, name, kind, kw, seeds, amps, over = case
    g = np.load(os.path.join(golden_dir, "env_kat.npz"))
    k = key.replace("-", "_")
    n, B, T = kw["n_links"], len(seeds), 200
    env = fg.make(f"fancy/{name}", num_envs=B, device=DEV, **over)
    obs0, _ = env.reset(seed=seeds)
    assert np.array_equal(obs0.cpu().numpy(), g[f"{k}/obs0"])
    outs = []
    for t in range(T):       # the action schedule of test_oracle_golden.py, float32
        a = np.stack([(A * np.sin(0.05 * t + np.arange(n))).astype(np.float32) for A in amps])
        ob, r, te, tr, _ = env.step(a)
        outs.append((ob.clone(), r.clone(), te.clone(), tr.clone()))
    obs = torch.stack([o[0] for o in outs], 1).cpu().numpy()
    rew = torch.stack([o[1] for o in outs], 1).cpu().numpy()
    term = torch.stack([o[2] for o in outs], 1).cpu().numpy()
    trunc = torch.stack([o[3] for o in outs], 1).cpu().numpy()
    length = g[f"{k}/length"]
    err = dict(obs=0.0, reward=0.0)
    for i in range(B):
        L = length[i]
        assert np.array_equal(term[i, :L], g[f"{k}/term"][i, :L]), (i, L)
        ends = np.nonzero(term[i])[0]
        assert (ends[0] + 1 if len(ends) else T) == L, (i, L)          # the episode ends where the reference's does
        ref_o, ref_r = g[f"{k}/obs"][i, :L], g[f"{k}/rew"][i, :L]
        err["obs"] = max(err["obs"], float(rel_err(obs[i, :L], ref_o).max()))
        fin = np.isfinite(ref_r)
        assert np.array_equal(rew[i, :L][~fin], ref_r[~fin])
        if fin.any():
            err["reward"] = max(err["reward"], float(rel_err(rew[i, :L][fin], ref_r[fin]).max()))
    # gymnasium's TimeLimit of the registration (200 steps): truncated on the 200th step and not before
    assert not trunc[:, :T - 1].any() and trunc[:, T - 1].all()
    _golden_err[key] = err
    record = os.environ.get("FG_STEP_GOLDEN_ERRORS_JSON")
    if record:
        with open(record, "w") as f:
            worst = {m: max(e[m] for e in _golden_err.values()) for m in STEP_GOLDEN_TOL}
            json.dump({"tolerance": STEP_GOLDEN_TOL, "measured_max_over_cases": worst, "per_case": _golden_err}, f, indent=1)
    for m, tol in STEP_GOLDEN_TOL.items():
        assert err[m] <= tol, (key, m, err[m], tol)


# --------------------------------------------------------------------------------------------
# 2. the fused rollout's per-step outputs (verbose=2), replayed one step() per control step
# --------------------------------------------------------------------------------------------
BB_IDS = [f"fancy_{mp}/{name}" for name in ("HoleReacher-v0", "ViaPointReacher-v0", "SimpleReacher-v0", "LongSimpleReacher-v0")
          for mp in ("ProMP", "DMP", "ProDMP")]
_POS = {"controller_kwargs": {"controller_type": "position"}}
REPLAY_CASES = [(i, {}, {}) for i in BB_IDS]
REPLAY_CASES += [("fancy_ProMP/HoleReacher-v0", dict(rew_fct="vel_acc"), {}),
                 ("fancy_ProMP/HoleReacher-v0", dict(rew_fct="unbounded"), {}),
                 ("fancy_ProDMP/HoleReacher-v0", dict(rew_fct="unbounded"), {}),
                 ("fancy_ProMP/HoleReacher-v0", dict(allow_self_collision=True), {}),
                 ("fancy_ProMP/HoleReacher-v0", dict(allow_wall_collision=True), {}),
                 ("fancy_DMP/ViaPointReacher-v0", dict(allow_self_collision=True), {}),
                 ("fancy_ProMP/HoleReacher-v0", {}, _POS), ("fancy_DMP/ViaPointReacher-v0", {}, _POS),
                 ("fancy_ProDMP/SimpleReacher-v0", {}, _POS)]
# every k_env_step instantiation against the verbose=2 instantiation of k_rollout at the same link count, under every MP
_REGISTERED_LINKS = {"HoleReacher-v0": 5, "ViaPointReacher-v0": 5, "SimpleReacher-v0": 2}
REPLAY_CASES += [(f"fancy_{mp}/{name}", dict(n_links=n), {}) for name in _REGISTERED_LINKS for n in range(2, 8)
                 for mp in ("ProMP", "DMP", "ProDMP") if n != _REGISTERED_LINKS[name]]


@pytest.mark.parametrize("env_id,env_over,mp_over", REPLAY_CASES,
                         ids=[c[0] + "".join(f"-{k}={v}" for k, v in c[1].items()) + ("-position" if c[2] else "")
                              for c in REPLAY_CASES])
def test_step_env_replays_the_fused_rollout_bit_for_bit(env_id, env_over, mp_over):
    fg = _fg()
    from fancy_gym_b200 import _lib
    B = 1000                 # not a multiple of the block size: a ragged last block
    bb = fg.make(env_id, num_envs=B, device=DEV, mp_config_override=dict(mp_over, black_box_kwargs={"verbose": 2}),
                 **env_over)
    bb.reset(seed=5)
    gen = torch.Generator(device=DEV).manual_seed(3)
    params = 0.7 * torch.randn(B, bb.action_space.shape[0], generator=gen, device=DEV)
    _, _, te_bb, tr_bb, info = bb.step(params)
    acts, s_obs, s_rew = info["step_actions"].clone(), info["step_observations"].clone(), info["step_rewards"].clone()
    L = info["trajectory_length"].clone().long()
    te_bb, tr_bb = te_bb.clone(), tr_bb.clone()
    # the controller's action reaches env.step as float32 (velocity / position control: the clipped float32 trajectory)
    # or float64 (PD control)
    dtype = torch.float64 if bb.tracking_controller.abi_code == _lib.CTRL_MOTOR else torch.float32
    env = fg.make("fancy/" + env_id.split("/")[1], num_envs=B, device=DEV, **env_over)
    env.reset(seed=5)
    O = env.observation_space.shape[0]
    bad_obs = torch.zeros(B, dtype=torch.bool, device=DEV)
    bad_rew = torch.zeros_like(bad_obs)
    first_term = torch.full((B,), -1, dtype=torch.long, device=DEV)
    tr_last = torch.zeros_like(bad_obs)
    for t in range(acts.shape[1]):
        ob, r, te, tr, _ = env.step(acts[:, t].to(dtype).contiguous())
        live = t < L
        bad_obs |= live & (ob != s_obs[:, t, :O]).any(1)
        bad_rew |= live & (r != s_rew[:, t])                 # (-inf == -inf)
        first_term = torch.where((first_term < 0) & te, t, first_term)
        tr_last = torch.where(L - 1 == t, tr, tr_last)
    assert int(bad_obs.sum()) == 0 and int(bad_rew.sum()) == 0, (int(bad_obs.sum()), int(bad_rew.sum()))
    ended = torch.where(first_term >= 0, first_term + 1, torch.full_like(first_term, 10 ** 6))
    assert torch.equal(te_bb, ended == L)                      # terminated on the rollout's last step ...
    assert bool((ended >= L).all())                            # ... and never before it
    assert torch.equal(tr_last, tr_bb)
    assert int(te_bb.sum()) + int(tr_bb.sum()) > 0


# --------------------------------------------------------------------------------------------
# 3. the oracle (oracle/reacher.py) at scale: random actions of both dtypes, past truncation
# --------------------------------------------------------------------------------------------
# (the oracle's wall test with its margins costs ~0.25 s per HoleReacher step at this size on the host: the HoleReacher
# options run with one action dtype each; the dtype rule itself is the same code for every option)
ORACLE_CASES = [("HoleReacher-v0", 2.0, {}, "float32"), ("HoleReacher-v0", 2.0, {}, "float64"),
                ("HoleReacher-v0", 2.0, dict(rew_fct="vel_acc"), "float32"),
                ("HoleReacher-v0", 2.0, dict(rew_fct="unbounded"), "float64"),
                ("HoleReacher-v0", 2.0, dict(allow_wall_collision=True, hole_x=1.0, hole_width=0.4, hole_depth=0.7), "float32"),
                ("HoleReacher-v0", 3.0, dict(allow_self_collision=True, allow_wall_collision=True), "float64"),
                ("ViaPointReacher-v0", 2.0, {}, "float32"), ("ViaPointReacher-v0", 2.0, {}, "float64"),
                ("ViaPointReacher-v0", 2.0, dict(allow_self_collision=True, random_start=True), "float32"),
                ("SimpleReacher-v0", 30.0, {}, "float32"), ("SimpleReacher-v0", 30.0, {}, "float64"),
                ("LongSimpleReacher-v0", 30.0, dict(random_start=False), "float64")]
# every link count k_env_step is instantiated for; the action dtype alternates with it, so both run for every env
_SIGMA = {"HoleReacher-v0": 2.0, "ViaPointReacher-v0": 2.0, "SimpleReacher-v0": 30.0}
ORACLE_CASES += [(name, _SIGMA[name], dict(n_links=n), ("float32", "float64")[n % 2])
                 for name in _REGISTERED_LINKS for n in range(2, 8) if n != _REGISTERED_LINKS[name]]
_KIND = {"HoleReacher-v0": "hole", "ViaPointReacher-v0": "viapoint", "SimpleReacher-v0": "simple", "LongSimpleReacher-v0": "simple"}


def _oracle_for(env, name, over):
    from oracle.reacher import BatchedReacher
    kind = _KIND[name]
    kw = dict(n_links=env.n_links, random_start=env.random_start, allow_self_collision=env.allow_self_collision)
    if kind == "hole":
        kw.update(allow_wall_collision=env.allow_wall_collision, collision_penalty=env.collision_penalty, rew_fct=env.rew_fct)
    elif kind == "viapoint":
        kw.update(collision_penalty=env.collision_penalty)
    o = BatchedReacher(kind, **kw)
    ctx, q0 = env.ctx.cpu().numpy(), env.q[:, 0].cpu().numpy()
    if kind == "hole":
        contexts = [dict(x=c[0], width=c[1], depth=c[2], q0=q) for c, q in zip(ctx, q0)]
    elif kind == "viapoint":
        contexts = [dict(via=c[0:2], goal=c[2:4], q0=q) for c, q in zip(ctx, q0)]
    else:
        contexts = [dict(goal=c[0:2], q0=q) for c, q in zip(ctx, q0)]
    o.reset(contexts=contexts)
    return o


@pytest.mark.parametrize("name,sigma,over,dtype", ORACLE_CASES,
                         ids=[c[0] + "".join(f"-{k}={v}" for k, v in c[2].items()) + "-" + c[3] for c in ORACLE_CASES])
def test_step_env_matches_oracle_at_scale(name, sigma, over, dtype):
    fg = _fg()
    B, T = 4096 + 37, 230
    env = fg.make(f"fancy/{name}", num_envs=B, device=DEV, **over)
    env.reset(seed=21)
    orc = _oracle_for(env, name, over)
    assert np.allclose(env.get_obs().cpu().numpy(), orc.get_obs(), rtol=0, atol=1e-6)
    rng = np.random.default_rng(4)
    tie_env = np.zeros(B, bool)            # envs in which a decision at an oracle margin below TIE_EPS came out differently
    for t in range(T):
        a = (sigma * rng.standard_normal((B, env.n_links))).astype(dtype)
        ob, r, te, tr, info = env.step(a)
        o_ob, o_r, o_te, o_info = orc.step(a)
        ob, r, te, tr = ob.cpu().numpy(), r.cpu().numpy(), te.cpu().numpy(), tr.cpu().numpy()
        assert (np.abs(ob - o_ob) <= 1e-5 * np.maximum(1.0, np.abs(o_ob))).all(), t
        # without the oracle (pinned against the reference at the registered link counts only): the observation's joint
        # entries and the end effector follow from the env's own float64 state
        n, q = env.n_links, env.q.cpu().numpy()
        trig = np.concatenate([np.cos(q), np.sin(q)], axis=1).astype(np.float32)
        assert (np.abs(ob[:, :2 * n] - trig) <= np.spacing(np.abs(trig))).all(), t          # within one float32 ulp
        assert np.array_equal(ob[:, 2 * n:3 * n], env.v.cpu().numpy().astype(np.float32)), t
        if "end_effector" in info:
            th = np.cumsum(q, axis=1)
            ee = np.stack([np.cos(th).sum(axis=1), np.sin(th).sum(axis=1)], axis=1)
            assert rel_err(info["end_effector"].cpu().numpy(), ee).max() <= 1e-12, t
        assert (tr == (t + 1 >= 200)).all(), t
        agree = te == o_te
        for k_ in ("is_success", "is_collided"):
            if k_ in info:
                agree &= info[k_].cpu().numpy() == o_info[k_]
        tie = o_info["margin"] < TIE_EPS
        assert (agree | tie).all(), (t, np.nonzero(~(agree | tie))[0][:10])
        tie_env |= ~agree
        ok = ~tie_env                       # (a tie resolved differently changes the "unbounded" latch from there on)
        fin = ok & np.isfinite(o_r)             # (ViaPointReacher: -inf except on steps 100 and 199 and on collisions)
        assert not fin.any() or rel_err(r[fin], o_r[fin]).max() < 1e-5, t
        assert np.array_equal(r[ok & ~np.isfinite(o_r)], o_r[ok & ~np.isfinite(o_r)]), t
        if "reward_dist" in info:
            assert rel_err(info["reward_dist"].cpu().numpy(), o_info["reward_dist"]).max() < 1e-5
            assert rel_err(info["reward_ctrl"].cpu().numpy(), o_info["reward_ctrl"]).max() < 1e-5
        if "end_effector" in info:
            assert rel_err(info["end_effector"].cpu().numpy(), o_info["end_effector"], scale=5.0).max() < 1e-5
        if "joints" in info:
            assert rel_err(info["joints"].cpu().numpy(), o_info["joints"], scale=np.pi).max() < 1e-12
    assert tie_env.sum() <= max(2, B // 500), int(tie_env.sum())


# --------------------------------------------------------------------------------------------
# 4. the vector env: auto-reset of the finished sub-envs only
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,sigma,T", [("HoleReacher-v0", 3.0, 230), ("SimpleReacher-v0", 20.0, 205)])
def test_step_vector_env_autoreset(name, sigma, T):
    fg = _fg()
    N, seed = 64, 7
    vec = fg.make_vec(f"fancy/{name}", N, device=DEV, tensors=True)
    twin = fg.make(f"fancy/{name}", num_envs=N, device=DEV)        # the same env without the adapter
    obs, _ = vec.reset(seed=seed)
    twin.reset(seed=seed)
    refs = {}                                                      # sub-env i: the reference env reset with seed + i

    def ref(i):
        if i not in refs:
            refs[i] = fg.make(f"fancy/{name}", num_envs=1, device=DEV, context_sampler="numpy")
            refs[i].reset(seed=seed + i)
        return refs[i]

    gen = torch.Generator(device=DEV).manual_seed(0)
    n_done = 0
    for t in range(T):
        a = sigma * torch.randn(N, vec.env.n_links, generator=gen, device=DEV)
        ctx0 = vec.env.ctx.clone()
        obs, rew, te, tr, info = vec.step(a)
        t_ob, t_r, t_te, t_tr, _ = twin.step(a)
        done = info["_final_observation"]
        assert torch.equal(done, t_te | t_tr) and torch.equal(rew, t_r)
        assert torch.equal(info["final_observation"], t_ob)          # the finished envs' last observation
        keep = ~done
        assert torch.equal(obs[keep], t_ob[keep]) and torch.equal(vec.env.ctx[keep], ctx0[keep])   # untouched rows
        twin.device_reset(None, mask=twin.done)
        for i in torch.nonzero(done).flatten().tolist():
            r_obs, _ = ref(i).reset()                              # the reference's unseeded follow-up reset
            assert torch.equal(vec.env.ctx[i], ref(i).ctx[0]) and torch.equal(vec.env.q[i], ref(i).q[0])
            assert torch.allclose(obs[i], r_obs[0], atol=1e-6), (t, i)
            assert obs[i, -1] == 0 and info["final_observation"][i, -1] > 0
        n_done += int(done.sum())
    assert n_done >= N
    if name == "SimpleReacher-v0":
        assert n_done == N             # never terminates: every sub-env is truncated once, on its 200th step
    vec.close()


# --------------------------------------------------------------------------------------------
# 5. no host synchronisation; a captured step() replays the eager steps bit for bit
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,dtype", [("HoleReacher-v0", torch.float32), ("ViaPointReacher-v0", torch.float64),
                                        ("SimpleReacher-v0", torch.float32)])
def test_step_without_sync_and_under_graph_capture(name, dtype):
    fg = _fg()
    B, T = 4096, 200
    kw = dict(rew_fct="unbounded") if name == "HoleReacher-v0" else {}
    eager = fg.make(f"fancy/{name}", num_envs=B, device=DEV, **kw)
    graphed = fg.make(f"fancy/{name}", num_envs=B, device=DEV, **kw)
    eager.reset(seed=2)
    graphed.reset(seed=2)
    gen = torch.Generator(device=DEV).manual_seed(9)
    acts = (1.5 * torch.randn(T, B, eager.n_links, generator=gen, device=DEV)).to(dtype)

    def keep(out):
        ob, r, te, tr, info = out
        return [ob.clone(), r.clone(), te.clone(), tr.clone()] + [v.clone() for v in info.values()]

    want = []
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for t in range(T):
            want.append(keep(eager.step(acts[t])))
    finally:
        torch.cuda.set_sync_debug_mode(0)

    got = [keep(graphed.step(acts[0]))]            # one eager step first: the output ring and the latch are allocated
    static_a = acts[1].clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = graphed.step(static_a)
    for t in range(1, T):
        static_a.copy_(acts[t])
        g.replay()
        got.append(keep(out))
    torch.cuda.synchronize()
    for t in range(T):
        for x, y in zip(got[t], want[t]):
            assert torch.equal(x, y), t
