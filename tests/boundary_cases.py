"""States placed at a chosen signed distance from one collision or joint-limit decision (plain numpy, no GPU).

Every builder returns a batch dict: q [B, n] float64 joint angles, ctx [B, 4] float64 env context (HoleReacher: hole x, width,
depth, 0), delta [B] (the oracle's signed margin the state was built for, NaN for exact / path cases whose margin is not
set), label [B] (what the case is).  The signed margin is the oracle's decision margin (oracle/reacher.py) with the sign of
the decision: positive for a free state, negative for a colliding one.  Wall margins are absolute (L-inf distance of the
nearest sample to the forbidden region, or the depth of the deepest sample inside it); self-collision margins are relative
to sum |sin| of the orientation test (the oracle's unit).  A state is found by varying one scalar of a family (a hole edge,
the depth, a rotation of the arm, one joint angle) with brentq until the oracle's signed margin equals delta.
"""
import numpy as np
from scipy.optimize import brentq

from oracle.reacher import forward_kinematics, line_points, self_collision, wall_collision

PI = np.pi
ULP24 = 2.0 ** -24


def beta_wall(n):
    """float32 error bound of the device's wall test at n links (derivation: tests/test_gpu_boundaries.py)"""
    return ULP24 * (n * n / 2 + 4.5 * n + 4)


def beta_self(n):
    """float32 error bound of the device's orientation tests, relative to sum |sin| (tests/test_gpu_boundaries.py)"""
    return 4 * (n + 1) * ULP24


def offsets(beta):
    d = [beta / 4, beta, 2 * beta, 4 * beta, 1e-5, 1e-4]
    return [0.0] + [s * x for x in d for s in (1.0, -1.0)]


# ----------------------------------------------------------------------------------------------------------------------
# oracle decisions with signed margins
# ----------------------------------------------------------------------------------------------------------------------
def wall_signed(q, ctx):
    """(collided [B], signed margin [B]) of the oracle's wall test alone"""
    q, ctx = np.atleast_2d(q), np.atleast_2d(ctx)
    hit, m = wall_collision(q, ctx[:, 0], ctx[:, 1], ctx[:, 2])
    return hit, np.where(hit, -m, m)


def self_signed(q):
    """(collided [B], signed margin [B]) of the oracle's pair tests alone (no joint limits: |q| <= pi is asserted)"""
    q = np.atleast_2d(q)
    assert (np.abs(q) <= PI).all()
    hit, m = self_collision(q, forward_kinematics(q))
    return hit, np.where(hit, -m, m)


def _solve(f, t0, delta, h0=1e-3):
    """t near t0 with f(t) == delta; the bracket grows until f - delta changes sign"""
    g = lambda t: f(t) - delta      # noqa: E731
    h = h0
    for _ in range(12):
        lo, hi = t0 - h, t0 + h
        glo, ghi = g(lo), g(hi)
        if glo == 0:
            return lo
        if ghi == 0:
            return hi
        if np.sign(glo) != np.sign(ghi):
            return brentq(g, lo, hi, xtol=1e-16, rtol=4 * np.finfo(float).eps, maxiter=400)
        h *= 4
    raise ValueError("no sign change around t0")


def _batch(rows):
    q = np.array([r[0] for r in rows], dtype=np.float64)
    ctx = np.array([r[1] for r in rows], dtype=np.float64)
    return dict(q=q, ctx=ctx, delta=np.array([r[2] for r in rows], dtype=np.float64), label=np.array([r[3] for r in rows]))


# ----------------------------------------------------------------------------------------------------------------------
# joint limits
# ----------------------------------------------------------------------------------------------------------------------
def _hi_edge():
    """pi's high word with the low word 0, and the largest double below it (the two edges of the device's high-word screen)"""
    pi_bits = np.array([PI]).view(np.uint64)[0]
    edge = np.array([pi_bits & np.uint64(0xFFFFFFFF00000000)], dtype=np.uint64).view(np.float64)[0]
    return edge, np.nextafter(edge, 0.0)


def joint_limit_values():
    e0, e1 = _hi_edge()
    v = [PI, np.nextafter(PI, 4.0), np.nextafter(PI, 0.0), e0, e1, 4.0, 1e300, 2.0 ** 1017, 1e308, np.inf, np.nan]
    return v + [-x for x in v[:-1]]


def joint_limit_cases(n, ctx_row):
    """each value of joint_limit_values() in joint 0, in joint n-1 and in a middle joint, the other joints 0 (a straight
    arm: a fold at exactly pi retraces the arm, so every orientation test is exactly collinear); NaN also together with a
    second joint at pi or nextafter(pi, 0).  delta is NaN: the decision is numpy's any(|q| > pi) | oracle pairs."""
    rows = []
    joints = sorted({0, n // 2, n - 1})
    for j in joints:
        for x in joint_limit_values():
            q = np.zeros(n)
            q[j] = x
            rows.append((q, ctx_row, np.nan, f"limit j{j}={x!r}"))
    for j in joints:
        for k in joints:
            if k == j:
                continue
            for p in (PI, np.nextafter(PI, 0.0), -PI):
                q = np.zeros(n)
                q[j], q[k] = np.nan, p
                rows.append((q, ctx_row, np.nan, f"limit j{j}=nan j{k}={p!r}"))
    return _batch(rows)


def joint_limit_decision(q):
    """numpy's any(q > pi) | any(q < -pi): NaN compares False"""
    with np.errstate(invalid="ignore"):
        return np.any(q > PI, axis=1) | np.any(q < -PI, axis=1)


# ----------------------------------------------------------------------------------------------------------------------
# wall (HoleReacher, run with allow_self_collision=True so the wall test alone decides)
# ----------------------------------------------------------------------------------------------------------------------
def _wall_shapes(n):
    """arm shapes (name, q): links at exactly 0 (c = 1, s = 0), within 1e-7 of vertical / horizontal, +-pi/4, downward, a
    link that crosses the ground line inside the link (an interior sample decides), absolute angles near 1e6 rad"""
    big = 2 * PI * 159155           # ~1e6 rad
    z = [0.0] * (n - 1)
    retrace = [PI if k % 2 == 0 else -PI for k in range(n - 2)]      # later links fold back along the previous one
    shapes = [("dive", [-PI / 2] + z), ("dive+1e-7", [-PI / 2 + 1e-7] + z), ("dive-1e-7", [-PI / 2 - 1e-7] + z),
              ("diag-right", [-PI / 4] + z), ("diag-left", [-3 * PI / 4] + z),
              ("dive-big", [-PI / 2 + big] + z), ("diag-big", [-PI / 4 - big] + z)]
    if n >= 2:
        shapes += [("bend-flat", [-PI / 2, PI / 2] + retrace), ("bend-flat+1e-7", [-PI / 2, PI / 2 + 1e-7] + retrace),
                   ("bend-pi-1e-7", [-PI / 2, -PI / 2 + 1e-7] + retrace),
                   ("cross-right", [0.5, -1.7] + retrace), ("cross-left", [PI - 0.5, 1.7] + [-x for x in retrace])]
    return [(name, np.array(q, dtype=np.float64)) for name, q in shapes]


def _ctx(xl, xr, d):
    return np.array([(xl + xr) / 2, xr - xl, d, 0.0])


def _wall_families(q):
    """(feature, build(t) -> ctx, t0) for one arm: t0 puts the feature on its boundary"""
    P = line_points(q[None])[0].reshape(-1, 2)[1:]      # sample 0 of link 0 is the base
    px, py = P[:, 0], P[:, 1]
    below = py < 0
    fam = []
    far = 4.0 + np.abs(P).max()
    if below.any():
        xmin, xmax, ymin = px[below].min(), px[below].max(), py.min()
        # left / right edge at the extreme below-ground sample (a ground-crossing link: an interior sample)
        fam.append(("edge-left", lambda t: _ctx(t, t + 2 * far, 2 * far), xmin))
        fam.append(("edge-right", lambda t: _ctx(t - 2 * far, t, 2 * far), xmax))
        # floor under the lowest sample, the column around the whole arm
        fam.append(("floor", lambda t: _ctx(-far, far, t), -ymin))
    return fam


def _rot(q, t):
    r = q.copy()
    r[0] += t
    return r


def wall_cases(n):
    rows = []
    beta = beta_wall(n)
    deltas = offsets(beta)
    for name, q in _wall_shapes(n):
        for feat, build, t0 in _wall_families(q):
            for d in deltas:
                t = _solve(lambda t: wall_signed(q, build(t))[1][0], t0, d)
                rows.append((q, build(t), d, f"wall {name} {feat}"))
    # the ground line, away from the hole: a straight arm rotated about the base (every joint on y = 0 at t = 0), and a
    # zigzag whose even joints touch the ground
    hole_far = np.array([50.0, 1.0, 1.0, 0.0])
    fams = [("ground-straight", np.zeros(n))]
    if n >= 2:
        fams.append(("ground-zigzag", np.array([0.3] + [(-0.6 if k % 2 == 0 else 0.6) for k in range(n - 1)])))
    for name, q in fams:
        for d in deltas:
            t = _solve(lambda t: wall_signed(_rot(q, t), hole_far)[1][0], 0.0, d)
            rows.append((_rot(q, t), hole_far, d, f"wall {name}"))
    # a floor above the ground line (negative depth): an arm reaching over a column that does not hold the base
    q = np.array([0.4] + [0.0] * (n - 1))
    P = line_points(q[None])[0].reshape(-1, 2)
    xl = 0.5 * (P[149, 0] + P[150, 0])     # midway between two samples of link 1
    inside = (P[:, 0] > xl)
    for d in deltas:
        build = lambda t: _ctx(xl, 50.0, t)      # noqa: E731
        t = _solve(lambda t: wall_signed(q, build(t))[1][0], -P[inside, 1].min(), d)
        rows.append((q, build(t), d, "wall floor-above-ground"))
    # exact cases (no offset): the base joint on an edge, edges at the float32 samples, depth 0, negative depth
    for w in (1.0, 0.5):
        for sgn in (1.0, -1.0):
            for name, q in _wall_shapes(n)[:5]:
                rows.append((q, np.array([sgn * w / 2, w, 2.0, 0.0]), np.nan, f"wall exact base-on-edge {name}"))
    s32 = np.linspace(0, 1, 100).astype(np.float32)
    flat = [sh for sh in _wall_shapes(n) if sh[0] == "bend-flat"]
    for name, q in flat:
        for k in (1, 33, 50, 98, 99):
            for e in (s32[k], np.nextafter(s32[k], np.float32(0)), np.nextafter(s32[k], np.float32(2))):
                e = float(e)
                rows.append((q, _ctx(-1.0, e, 2.0), np.nan, f"wall exact xr=s32[{k}] {name}"))
                rows.append((q, _ctx(e - 1.0, e, 2.0), np.nan, f"wall exact xr=s32[{k}] narrow {name}"))
    for name, q in _wall_shapes(n)[:5] + [("flat", np.zeros(n))]:
        rows.append((q, np.array([0.0, 4.0, 0.0, 0.0]), np.nan, f"wall exact depth0 {name}"))
        rows.append((q, np.array([0.0, 4.0, -0.5, 0.0]), np.nan, f"wall exact depth<0 {name}"))
        rows.append((q, np.array([3.0, 2.0, -0.5, 0.0]), np.nan, f"wall exact depth<0 off-base {name}"))
    return _batch(rows)


# ----------------------------------------------------------------------------------------------------------------------
# self collision (pair tests; |q| <= pi everywhere)
# ----------------------------------------------------------------------------------------------------------------------
def self_cases(n, ctx_row):
    assert n >= 3
    rows = []
    beta = beta_self(n)
    deltas = offsets(beta)
    # the last joint folds onto the straight part of the arm: q_{n-2} = a, q_{n-1} = 2 pi - 2 a puts joint n on the line of
    # link n-3 at 1 + 2 cos a from joint n-3 (a = 2.0: inside link n-3; 2.08: 0.024 from its start, two links crossing
    # near an end; 2.5: inside link n-4)
    for a in (2.0, 2.08, 2.5):
        if a == 2.5 and n < 4:
            continue
        for q0, s in ((0.3, 1.0), (-2.0, 1.0), (1.1, 1.0), (0.3, -1.0), (-2.0, -1.0), (1.1, -1.0)):   # s: mirrored
            base = s * np.array([q0] + [0.0] * (n - 3) + [a, 2 * PI - 2 * a])
            for d in deltas:
                def f(t):
                    qq = base.copy()
                    qq[-1] += t
                    return self_signed(qq)[1][0]
                t = _solve(f, 0.0, d, h0=1e-4)
                qq = base.copy()
                qq[-1] += t
                rows.append((qq, ctx_row, d, f"self touch a={s * a} q0={s * q0}"))
    # path cases (decision far from its boundary, orientation values near the fast / accurate switch at 8e-6): links 0 and
    # 1 at relative angle eps, a bend of 3.05 further on so the pair tests run
    for eps in (1e-7, 1e-6, 7e-6, 9e-6, 1e-5):
        for s in (1.0, -1.0):
            q = np.array([0.3, s * eps, 3.05] + [0.1] * (n - 3))
            rows.append((q, ctx_row, np.nan, f"self eps={s * eps:g}"))
            q = np.array([0.3, 0.5] + [s * eps] * (n - 3) + [3.05])
            rows.append((q, ctx_row, np.nan, f"self eps-tail={s * eps:g}"))
    # folds at exactly +-pi (collinear overlap, not a limit)
    for j in range(1, n):
        for p in (PI, -PI):
            q = np.zeros(n)
            q[0], q[j] = 0.7, p
            rows.append((q, ctx_row, np.nan, f"self fold j{j}={p:+.3f}"))
    # the curl (equal turns) at the edge of the turn screen: sum_{l>=1} |q_l| around 3.0 (float32) and pi
    t3 = np.float32(3.0)
    for total in (float(np.nextafter(t3, np.float32(0))), 3.0, float(np.nextafter(t3, np.float32(4))), PI - 1e-6,
                  PI + 1e-6):
        for s in (1.0, -1.0):
            q = np.array([0.2] + [s * total / (n - 1)] * (n - 1))
            rows.append((q, ctx_row, np.nan, f"self curl {s * total!r}"))
    return _batch(rows)
