"""Trajectory covariance (fg_traj_cov, SURVEY.md §8 row a20 / BASELINE config 4) against the float64 oracle
(oracle/mp.py traj_pos_cov; PARITY UNPINNED: mp_pytorch is absent and fancy_gym never calls this path).
Tolerance: 1e-5 of the largest covariance entry of the env (entries far off the diagonal cancel to ~0)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.blackbox import make_oracle  # noqa: E402
from oracle.mp import traj_pos_cov  # noqa: E402


def _setup(env_id, B, seed=0):
    import fancy_gym_b200 as fancy_gym
    env = fancy_gym.make(env_id, num_envs=B, device="cuda:0")
    env.reset(seed=0)
    tg = env.traj_gen
    tg.set_initial_conditions(0.0, env.unwrapped.q, env.unwrapped.v)
    tg.set_duration(2.0, 0.01)
    D = tg._num_local_params
    rng = np.random.default_rng(seed)
    L = np.tril(0.1 * rng.standard_normal((B, D, D))) + 0.5 * np.eye(D)        # BASELINE config 4
    return env, tg, L.astype(np.float32), _oracle_basis(env_id, D)


def _oracle_basis(env_id, D):
    """Psi's diagonal block [T, Kc] from the ORACLE (float64 definition, oracle/mp.py), not from the product's own tables:
    ProMP weights_scale * Phi (learnable columns), ProDMP the bracketed H = [H_w | H_g] of App. B.7"""
    orc = make_oracle(env_id, mode="gold")
    orc.reset(seeds=[0])
    otg = orc.traj_gen
    otg.set_params(np.zeros((1, D)))
    otg.set_initial_conditions(np.array(0.0), orc.env.current_pos, orc.env.current_vel)
    otg.set_duration(2.0, 0.01)
    return np.asarray(otg.cov_basis(), dtype=np.float64)


@pytest.mark.parametrize("env_id,B", [("fancy_ProMP/HoleReacher-v0", 3), ("fancy_ProDMP/SimpleReacher-v0", 17),
                                      ("fancy_ProMP/SimpleReacher-v0", 5), ("fancy_ProDMP/HoleReacher-v0", 2)])
@pytest.mark.parametrize("batch_scope", [False, True])
@pytest.mark.parametrize("path", [1, 2])
def test_traj_cov_matches_oracle(env_id, B, batch_scope, path):
    env, tg, L, basis = _setup(env_id, B)
    tg.set_mp_params_variances(torch.as_tensor(L))
    cov = tg.get_traj_pos_cov(batch_scope=batch_scope, path=path).cpu().numpy()
    std = tg.get_traj_pos_std(batch_scope=batch_scope).cpu().numpy()
    o_cov, o_std = traj_pos_cov(basis, L, tg.num_dof, 1e-4, batch_scope)
    scale = np.abs(o_cov).max(axis=(1, 2), keepdims=True)
    assert (np.abs(cov - o_cov) <= 1e-5 * scale).all(), float((np.abs(cov - o_cov) / scale).max())
    assert np.allclose(std, o_std, rtol=1e-5, atol=0)
    assert np.array_equal(cov, np.swapaxes(cov, 1, 2)) or np.abs(cov - np.swapaxes(cov, 1, 2)).max() <= 2e-6 * scale.max()
    # positive definite thanks to the regulariser (what it is there for): Cholesky succeeds in float64
    np.linalg.cholesky(cov[0].astype(np.float64) + 1e-7 * scale[0] * np.eye(cov.shape[1]))


def test_traj_cov_unbatched_and_errors():
    env, tg, L, basis = _setup("fancy_ProMP/HoleReacher-v0", 1)
    tg.set_mp_params_variances(torch.as_tensor(L[0]))
    cov = tg.get_traj_pos_cov()
    assert cov.shape == (1000, 1000)
    with pytest.raises(ValueError):
        tg.set_mp_params_variances(torch.zeros(3, 3))
        tg.get_traj_pos_cov()
    import fancy_gym_b200 as fancy_gym
    dmp = fancy_gym.make("fancy_DMP/ViaPointReacher-v0", num_envs=1, device="cuda:0").traj_gen
    with pytest.raises(NotImplementedError):
        dmp.set_mp_params_variances(torch.zeros(30, 30))
