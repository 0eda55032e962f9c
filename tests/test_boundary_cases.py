"""The constructed boundary states (tests/boundary_cases.py) are what they claim to be, by the oracle alone: no GPU.  A
construction bug shows up here, apart from any kernel bug in tests/test_gpu_boundaries.py."""
import numpy as np
import pytest

from tests import boundary_cases as bc

CTX_VIA = np.array([1.0, 1.0, 2.0, 2.0])


@pytest.mark.parametrize("n", range(2, 8))
def test_wall_cases_sit_at_their_offsets(n):
    c = bc.wall_cases(n)
    hit, m = bc.wall_signed(c["q"], c["ctx"])
    off = np.isfinite(c["delta"])
    assert np.abs(m[off] - c["delta"][off]).max() <= 1e-12
    nz = off & (c["delta"] != 0)
    assert np.array_equal(hit[nz], c["delta"][nz] < 0)          # negative offset: collided; positive: free
    beta = bc.beta_wall(n)
    assert ((np.abs(m) > beta) & (np.abs(m) <= 4 * beta)).sum() >= 50
    # every shape and feature at every offset
    labels = set(c["label"][off])
    assert {"wall cross-right edge-left", "wall dive-big floor", "wall ground-zigzag", "wall floor-above-ground"} <= labels
    # the exact cases cover both decisions
    assert hit[~off].any() and not hit[~off].all()


@pytest.mark.parametrize("n", range(3, 8))
def test_self_cases_sit_at_their_offsets(n):
    c = bc.self_cases(n, CTX_VIA)
    hit, m = bc.self_signed(c["q"])
    off = np.isfinite(c["delta"])
    assert np.abs(m[off] - c["delta"][off]).max() <= 1e-12
    nz = off & (c["delta"] != 0)
    assert np.array_equal(hit[nz], c["delta"][nz] < 0)
    beta = bc.beta_self(n)
    assert ((np.abs(m) > beta) & (np.abs(m) <= 4 * beta)).sum() >= 20
    # the path cases (relative angle eps, curls) are far from their decision boundary; the folds at exactly +-pi (whose
    # oracle margin is the | |q| - pi | = 0 of the joint-limit term) retrace a straight arm: every test exactly collinear
    fold = np.char.startswith(c["label"].astype(str), "self fold")
    path = ~off & ~fold
    assert (np.abs(m[path]) > 1e-3).all(), c["label"][path][np.abs(m[path]) <= 1e-3]
    assert fold.sum() == 2 * (n - 1) and not hit[fold].any()
    assert not bc.joint_limit_decision(c["q"]).any()
    eps = np.char.startswith(c["label"].astype(str), "self eps")
    assert eps.sum() == 20 and (np.abs(c["q"][eps]).sum(axis=1) - np.abs(c["q"][eps, 0]) > 3.0).all()   # past the screen


@pytest.mark.parametrize("n", range(2, 8))
def test_joint_limit_cases(n):
    c = bc.joint_limit_cases(n, CTX_VIA)
    q = c["q"]
    want = bc.joint_limit_decision(q)
    # the values the device screens on their high words: +-inf and |q| >= 2^1017 are limits, NaN and pi itself are not
    for x, lim in ((np.inf, True), (-np.inf, True), (1e308, True), (2.0 ** 1017, True), (np.nextafter(np.pi, 4), True),
                   (np.pi, False), (-np.pi, False), (np.nextafter(np.pi, 0), False), (bc._hi_edge()[0], False)):
        rows = (q == x).any(axis=1) & ~np.isnan(q).any(axis=1)
        assert rows.sum() == len({0, n // 2, n - 1}) and (want[rows] == lim).all(), x
    nan_rows = np.isnan(q).any(axis=1)
    assert nan_rows.sum() > 3 and not want[nan_rows].any()
    # a straight arm folded at one joint: no pair of links intersects (the oracle's margin there is | |q| - pi |, not a
    # distance of the pair tests)
    fin = np.isfinite(q).all(axis=1) & ~want
    hit, _ = bc.self_signed(q[fin])
    assert fin.sum() > 10 and not hit.any()
