"""Trajectory covariance (K5, fg_traj_cov) on every tiling path of both kernels.

1. Arithmetic: path 1 (k_cov_simt) and path 2 (k_cov_umma) against the float64 product oracle.mp.traj_pos_cov of the
   kernel's own float32 basis, element by element within k * 2^-24 * (M + reg * max_i M_ii * I), where
   M = |Psi| |L| |L|^T |Psi|^T is the magnitude the float32 sums run over.  The shapes reach the SIMT template and run-time
   Kc, its scalar fallback and both column-quad passes, and the UMMA kernel's N-tile counts (1..6, so the "empty" barrier
   reaches its second phase), ragged and single M tiles, TMA boxes larger than the matrix, K' = 8..48, operand plans near
   the shared-memory limit and two CTAs per SM sharing TMEM.
2. Invariances, bit for bit: rows per block, path 0 vs 1, sharding, the strict upper triangle of L, unbatched input.
3. Limits: what the kernels cannot do raises NotImplementedError; B = 0; std at more than 65 535 envs.
4. Semantics: the covariance is that of the trajectories the env generates, under either placement of the weight / goal
   scales (switch scale_on_library_side)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import mp as omp  # noqa: E402
from oracle.blackbox import RESOLVED, make_oracle  # noqa: E402
from oracle.mp import traj_pos_cov  # noqa: E402

DEV = "cuda:0"
EPS = 2.0 ** -24
REG = 1e-4
# error bound in units of 2^-24 * M.  A float32 emulation of the operation order on the CPU reached 5.4 (SIMT) and 18
# (3xTF32: the dropped A_lo * B_lo term and TF32-rounded operands) at dof 5, Kc 5, T 200.  On a B200 (1000 W power limit)
# the kernels reached at most 5.6 (path 1), 30.7 (path 2) and 7.4 (std) over the cases below.
K_BOUND = {1: 32, 2: 64}

PROMP_S, PROMP_H = "fancy_ProMP/SimpleReacher-v0", "fancy_ProMP/HoleReacher-v0"
PRODMP_S, PRODMP_H = "fancy_ProDMP/SimpleReacher-v0", "fancy_ProDMP/HoleReacher-v0"

# id (dof-Kc-T), env id, n_links, num_basis, T, B, path 2 accepts it
CASES = [("2-5-8", PROMP_S, None, None, 8, 3, True),             # TMA boxes larger than the matrix; row_lanes 64
         ("2-5-100-B400", PROMP_S, None, None, 100, 400, True),  # one N tile, ragged M tile, 2 UMMA CTAs / SM, many waves
         ("2-5-128", PROMP_S, None, None, 128, 3, True),         # exactly one full M and N tile
         ("2-5-129", PROMP_S, None, None, 129, 3, False),        # dof*T % 4 != 0: SIMT scalar fallback
         ("5-5-129", PROMP_H, None, None, 129, 3, False),
         ("2-5-640", PROMP_S, None, None, 640, 3, True),         # 5 N tiles, 5 M tiles; two column-quad passes
         ("5-5-300-B17", PROMP_H, None, None, 300, 17, True),    # 6 N tiles, last M tile 44 rows, > 148 CTAs
         ("7-5-200", PROMP_H, 7, None, 200, 3, True),            # 6 N tiles, D = 35, ~204 KB shared memory
         ("2-1-50", PROMP_S, None, 1, 50, 3, True),              # K' = 8 (one MMA), k_cov_simt<0>
         ("5-3-64", PROMP_H, None, 3, 64, 3, True),              # run-time Kc, one M tile
         ("7-13-40", PROMP_H, 7, 13, 40, 3, True),               # D = 91, K' = 40, last N tile 24 columns
         ("6-16-100", PROMP_H, 6, 16, 100, 3, False),            # D = 96 (the limit), Kc = 16; path 2: shared memory
         ("5-8-200", PRODMP_H, None, 7, 200, 3, True),           # run-time Kc with c0 = 2, K' = 24, ~217 KB
         ("2-6-8", PRODMP_S, None, None, 8, 3, True)]            # k_cov_simt<6> at the smallest shape
CASE = {c[0]: c for c in CASES}


def _fg():
    import fancy_gym_b200 as fancy_gym
    return fancy_gym


def _traj_gen(env_id, T, n_links=None, num_basis=None):
    """the env's trajectory generator with a T-point plan over the same 2 s (the phase still spans [0, 1]).  The ProDMP
    tables are looked up at the nearest pre-integrated point, so every T down to 8 is accepted."""
    over = {"basis_generator_kwargs": dict(RESOLVED[env_id]["basis"], num_basis=num_basis)} if num_basis else {}
    env_kw = {"n_links": n_links} if n_links else {}
    tg = _fg().make(env_id, num_envs=1, device=DEV, mp_config_override=over, **env_kw).traj_gen
    tg.set_duration(2.0, 2.0 / T)
    assert tg.n_steps == T
    return tg


def _kernel_basis(tg, env_id, T, n_links=None, num_basis=None):
    """Psi's diagonal block [T, Kc]: the float32 table the kernels read, checked bit for bit against the oracle's
    mirror-mode table (the float64 reference is only a reference of the kernels' arithmetic if both start from it)"""
    c0 = 2 if "ProDMP" in env_id else 0
    psi = np.asarray(tg.tables().tab_a[:T, c0:], dtype=np.float32)
    over = {}
    if num_basis:
        over["basis"] = dict(num_basis=num_basis)
    if n_links:
        over["env"] = dict(n_links=n_links)
    otg = make_oracle(env_id, mode="mirror", mp_overrides=over).traj_gen
    n = otg.num_dof
    otg.set_params(np.zeros((1, otg.num_params), np.float32))
    otg.set_initial_conditions(np.array(0.0), np.zeros((1, n)), np.zeros((1, n)))
    otg.set_duration(2.0, 2.0 / T)
    mirror = otg.cov_basis().astype(np.float32)
    assert psi.shape == mirror.shape and np.array_equal(psi, mirror), "the kernel's basis table is not the oracle's"
    return psi


def _draw_L(B, D, seed=0, big=None, factor=1e3):
    """as tests/test_gpu_cov.py (BASELINE config 4), one env optionally scaled so per-env and batch maxima differ"""
    rng = np.random.default_rng(seed)
    L = np.tril(0.1 * rng.standard_normal((B, D, D))) + 0.5 * np.eye(D)
    if big is not None:
        L[big] *= factor
    return L.astype(np.float32)


def _blockdiag(psi, N):
    T, Kc = psi.shape
    P = np.zeros((N * T, N * Kc))
    for d in range(N):
        P[d * T:(d + 1) * T, d * Kc:(d + 1) * Kc] = psi
    return P


def _magnitude(psi, L, N, batch_scope):
    """M = |Psi| |L| |L|^T |Psi|^T in float64, the max of its diagonal over the regulariser's scope, and the absolute
    error float32 allows where terms fall below its smallest normal number 2^-126 (the wider bases have denormal entries;
    a product of two of them vanishes): 2^-126 * max(1, max |Psi|)"""
    P = np.abs(_blockdiag(np.asarray(psi, np.float64), N))
    La = np.abs(np.tril(L.astype(np.float64)))
    M = P[None] @ (La @ np.swapaxes(La, 1, 2)) @ P.T[None]
    Md = np.einsum("bii->bi", M)
    mx = Md.max() if batch_scope else Md.max(axis=1)[:, None, None]
    return M, Md, mx, 2.0 ** -126 * max(1.0, float(P.max()))


def _cov_ratio(cov, ref, M, mx, tiny):
    """max over elements of |cov - ref| / (2^-24 (M + reg max M_ii I) + tiny)"""
    denom = EPS * (M + REG * mx * np.eye(M.shape[1])[None]) + tiny
    return float(np.max(np.abs(cov.astype(np.float64) - ref) / denom))


def _std_ratio(std, ref_std, Md, mx, tiny, T, N):
    """the same bound on the variance: |std^2 - ref^2| / (2^-24 (M_ii + reg max M_ii) + tiny)"""
    B = std.shape[0]
    Mii = Md.reshape(B, N, T).transpose(0, 2, 1)
    denom = EPS * (Mii + REG * (mx if np.ndim(mx) == 0 else mx.reshape(B, 1, 1))) + tiny
    return float(np.max(np.abs(std.astype(np.float64) ** 2 - ref_std ** 2) / denom))


def _cov(tg, L, batch_scope, path):
    tg.set_mp_params_variances(torch.as_tensor(L, device=DEV))
    return tg.get_traj_pos_cov(reg=REG, batch_scope=batch_scope, path=path).cpu().numpy()


def _std(tg, L, batch_scope):
    tg.set_mp_params_variances(torch.as_tensor(L, device=DEV))
    return tg.get_traj_pos_std(reg=REG, batch_scope=batch_scope).cpu().numpy()


# ---- 1. arithmetic against float64 ------------------------------------------------------------------------------------
ARITH = [(c[0], False) for c in CASES] + [("5-5-300-B17", True), ("7-13-40", True)]


@pytest.mark.parametrize("case,batch_scope", ARITH, ids=[f"{c}-{'batch' if s else 'env'}" for c, s in ARITH])
def test_cov_paths_within_float32_bound(case, batch_scope):
    _, env_id, n_links, num_basis, T, B, umma_ok = CASE[case]
    tg = _traj_gen(env_id, T, n_links, num_basis)
    psi = _kernel_basis(tg, env_id, T, n_links, num_basis)
    N, D = tg.num_dof, tg._num_local_params
    assert D == N * psi.shape[1]
    L = _draw_L(B, D, seed=1, big=1)
    ref, ref_std = traj_pos_cov(psi.astype(np.float64), L, N, REG, batch_scope)
    M, Md, mx, tiny = _magnitude(psi, L, N, batch_scope)
    ratios = {}
    for path in (1, 2):
        if path == 2 and not umma_ok:
            with pytest.raises(NotImplementedError):
                _cov(tg, L, batch_scope, path)
            continue
        cov = _cov(tg, L, batch_scope, path)
        assert cov.shape == (B, N * T, N * T)
        ratios[path] = _cov_ratio(cov, ref, M, mx, tiny)
    ratios["std"] = _std_ratio(_std(tg, L, batch_scope), ref_std, Md, mx, tiny, T, N)
    print(f"cov {case} batch_scope={batch_scope}: max err / (2^-24 M) " + ", ".join(f"{k}: {v:.2f}" for k, v in ratios.items()))
    msg = f"max err / (2^-24 M) per path: {ratios}, bounds {K_BOUND}"
    assert all(ratios[p] <= K_BOUND[p] for p in (1, 2) if p in ratios), msg
    assert ratios["std"] <= K_BOUND[1], msg


# ---- 2. invariances, bit for bit ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["5-5-300-B17", "2-5-100-B400"])
def test_rows_per_block_does_not_change_bits(case, monkeypatch):
    _, env_id, n_links, num_basis, T, _, _ = CASE[case]
    tg = _traj_gen(env_id, T, n_links, num_basis)
    L = _draw_L(3, tg._num_local_params, seed=2, big=1)
    base = _cov(tg, L, False, 1)
    assert np.array_equal(_cov(tg, L, False, 0), base)          # path 0 selects path 1
    for rows in (1, 3, 7, 64, T):
        monkeypatch.setenv("FG_COV_ROWS", str(rows))            # read by every launch
        assert np.array_equal(_cov(tg, L, False, 1), base), rows


@pytest.mark.parametrize("case", ["5-5-300-B17", "2-5-100-B400", "7-13-40"])
def test_shards_upper_triangle_and_unbatched_do_not_change_bits(case):
    _, env_id, n_links, num_basis, T, _, _ = CASE[case]
    tg = _traj_gen(env_id, T, n_links, num_basis)
    D = tg._num_local_params
    L = _draw_L(5, D, seed=3, big=2)
    L_nan = L.copy()
    L_nan[:, np.triu_indices(D, 1)[0], np.triu_indices(D, 1)[1]] = np.nan
    for path in (1, 2):
        whole = _cov(tg, L, False, path)
        shards = np.concatenate([_cov(tg, L[a:b], False, path) for a, b in ((0, 1), (1, 4), (4, 5))])
        assert np.array_equal(whole, shards), path
        assert np.array_equal(_cov(tg, L[0], False, path), whole[0]), path
        for scope in (False, True):
            assert np.array_equal(_cov(tg, L_nan, scope, path), _cov(tg, L, scope, path)), (path, scope)
    for scope in (False, True):
        assert np.array_equal(_std(tg, L_nan, scope), _std(tg, L, scope)), scope
    assert np.array_equal(_std(tg, L[0], False), _std(tg, L, False)[0])


# ---- 3. limits and refusals ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env_id,n_links,num_basis,T,B,paths,std", [
    (PROMP_S, None, 17, 100, 2, (1, 2), True),      # Kc = 17
    (PROMP_H, 7, 14, 100, 2, (1, 2), True),         # D = 98
    (PROMP_H, None, None, 400, 2, (2,), False),     # path 2: operands exceed shared memory
    (PROMP_S, None, None, 8, 65536, (1, 2), False),  # one launch covers at most 65 535 envs (output 64 MB)
], ids=["Kc17", "D98", "umma-smem", "B65536"])
def test_refusals(env_id, n_links, num_basis, T, B, paths, std):
    tg = _traj_gen(env_id, T, n_links, num_basis)
    L = torch.as_tensor(_draw_L(1, tg._num_local_params)).expand(B, -1, -1).contiguous()
    for path in paths:
        with pytest.raises(NotImplementedError):
            _cov(tg, L, False, path)
    if std:
        with pytest.raises(NotImplementedError):
            _std(tg, L, False)


@pytest.mark.parametrize("flip", [False, True], ids=["defaults", "scale_on_parameters"])
def test_empty_batch(flip):
    from fancy_gym_b200.mp import assumptions as pa
    with pa.assume(**(dict(scale_on_library_side=False) if flip else {})):
        tg = _traj_gen(PROMP_H, 200)
    D, N = tg._num_local_params, tg.num_dof
    L = np.zeros((0, D, D), np.float32)
    for path in (1, 2):
        assert _cov(tg, L, False, path).shape == (0, N * 200, N * 200)
    assert _std(tg, L, False).shape == (0, 200, N)


@pytest.mark.parametrize("batch_scope", [False, True])
def test_std_beyond_65535_envs(batch_scope):
    """the std needs no covariance launch, so it has no batch limit: 70 000 envs, checked on a seeded sample of 64 incl.
    indices above 65 535.  With batch scope one planted env above 65 535 holds the batch's largest variance."""
    T, B = 200, 70000
    tg = _traj_gen(PROMP_H, T)
    psi = _kernel_basis(tg, PROMP_H, T)
    N, D = tg.num_dof, tg._num_local_params
    rng = np.random.default_rng(4)
    L = _draw_L(B, D, seed=5)
    planted = 68000
    if batch_scope:
        L[planted] *= 10
    sample = np.sort(np.concatenate([rng.choice(65536, 48, replace=False), rng.choice(np.arange(65536, B), 16, replace=False)]))
    std = _std(tg, L, batch_scope)
    assert std.shape == (B, T, N)
    worst = 0.0
    for chunk in np.array_split(sample, 8):
        sub = np.concatenate([L[[planted]], L[chunk]]) if batch_scope else L[chunk]
        _, ref_std = traj_pos_cov(psi.astype(np.float64), sub, N, REG, batch_scope)
        _, Md, mx, tiny = _magnitude(psi, sub, N, batch_scope)
        got = np.concatenate([std[[planted]], std[chunk]]) if batch_scope else std[chunk]
        worst = max(worst, _std_ratio(got, ref_std, Md, mx, tiny, T, N))
    assert worst <= K_BOUND[1], worst


# ---- 4. semantics: the covariance of the trajectories the env generates -------------------------------------------------
SEMANTIC = [(PROMP_H, {}), (PRODMP_S, dict(weights_scale=3.0, goal_scale=0.5))]


def _effective_basis(env_id, traj, D):
    """Psi_eff [dof*T, D] of the gold oracle: column k = pos(e_k) - pos(0) of get_traj_pos, every scale included wherever
    the switch puts it"""
    otg = make_oracle(env_id, mode="gold", mp_overrides={"traj": traj} if traj else None).traj_gen
    n = otg.num_dof
    assert otg.num_params == D
    params = np.concatenate([np.zeros((1, D)), np.eye(D)])
    otg.set_params(params)
    otg.set_initial_conditions(np.array(0.0), np.zeros((D + 1, n)), np.zeros((D + 1, n)))
    otg.set_duration(2.0, 0.01)
    pos = np.asarray(otg.get_traj_pos(), dtype=np.float64)            # [D+1, T, dof]
    eff = (pos[1:] - pos[:1]).transpose(2, 1, 0).reshape(-1, D)      # rows d * T + t
    return eff, np.asarray(otg.cov_basis(), dtype=np.float64)


@pytest.mark.parametrize("flip", [False, True], ids=["defaults", "scale_on_parameters"])
@pytest.mark.parametrize("env_id,traj", SEMANTIC, ids=[s[0] for s in SEMANTIC])
def test_cov_is_that_of_the_generated_trajectories(env_id, traj, flip):
    from fancy_gym_b200.mp import assumptions as pa
    flips = dict(scale_on_library_side=False) if flip else {}
    with pa.assume(**flips):
        env = _fg().make(env_id, num_envs=1, device=DEV,
                         mp_config_override={"trajectory_generator_kwargs": traj} if traj else {})
    with omp.assume(**flips):
        eff, o_basis = _effective_basis(env_id, traj, env.traj_gen._num_local_params)
    tg = env.traj_gen
    tg.set_duration(2.0, 0.01)
    N, D = tg.num_dof, tg._num_local_params
    L = _draw_L(3, D, seed=6)
    Lt = np.tril(L.astype(np.float64))
    ref = eff[None] @ (Lt @ np.swapaxes(Lt, 1, 2)) @ eff.T[None]
    ref = ref + REG * np.einsum("bii->bi", ref).max(axis=1)[:, None, None] * np.eye(ref.shape[1])[None]
    scale = np.abs(ref).max(axis=(1, 2), keepdims=True)
    got = {f"path {p}": _cov(tg, L, False, p) for p in (1, 2)}
    got["oracle"] = traj_pos_cov(o_basis, L, N, REG, False)[0]
    for name, cov in got.items():
        err = float((np.abs(cov - ref) / scale).max())
        assert err <= 1e-5, f"{name}: error {err:.2e} of the largest entry, largest entries {np.abs(cov).max() / scale.max():.3f}x the reference's"
