"""Parity at BASELINE.json's full sizes (configs 2, 3, 5 and the divergent sigma = 1.0 regime): a random 4 096-env subset of
the full batch is checked against the oracle (the envs are seeded individually, env i == seed s + i, so any subset can be
re-run on the CPU), and the WHOLE batch against shard equivalence — the same envs run as four separate batches must
give bit-identical results (what the multi-GPU sharding of SURVEY.md §8e relies on)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle.blackbox import make_oracle  # noqa: E402

TIE_EPS = 1e-5
SUBSET = 4096

CASES = [("fancy_ProMP/HoleReacher-v0", 65536, 0.25, "config2", {}),
         ("fancy_ProMP/HoleReacher-v0", 65536, 1.0, "config2-sigma1", {}),
         ("fancy_DMP/ViaPointReacher-v0", 262144, 1.0, "config3", {}),
         ("fancy_ProMP/HoleReacher-v0", 1 << 20, 0.25, "config5-per-gpu", {})]
# the persistent grid and its work queue (B above twice the resident blocks; the B / 4 shards run without it) at link counts
# whose slot layout and shared-memory budget, hence occupancy, differ from the registered 5
CASES += [("fancy_ProMP/HoleReacher-v0", 1 << 18, 1.0, f"sigma1-{n}links", dict(n_links=n)) for n in (3, 7)]


def rel_err(a, b, scale=1.0):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), scale)


@pytest.mark.parametrize("env_id,B,sigma,name,env_kw", CASES, ids=[c[3] for c in CASES])
def test_full_size_subset_against_oracle_and_shard_equivalence(env_id, B, sigma, name, env_kw):
    import fancy_gym_b200 as fancy_gym
    dev = "cuda:0"
    seed = 1000
    env = fancy_gym.make(env_id, num_envs=B, device=dev, context_sampler="device", **env_kw)
    P = env.action_space.shape[0]
    gen = torch.Generator(device=dev).manual_seed(5)
    params = sigma * torch.randn(B, P, generator=gen, device=dev)
    env.reset(seed=seed)
    obs, ret, te, tr, info = env.step(params)
    full = [x.clone() for x in (obs, ret, te, tr, info["trajectory_length"])]
    steps_total = int(full[4].sum())
    assert steps_total > 0

    # ---- the whole batch: four shards, each its own env object and launch ----
    n_sh = 4
    shard = fancy_gym.make(env_id, num_envs=B // n_sh, device=dev, context_sampler="device", **env_kw)
    for k in range(n_sh):
        lo = k * (B // n_sh)
        sl = slice(lo, lo + B // n_sh)
        shard.reset(seed=seed + lo)
        s_obs, s_ret, s_te, s_tr, s_info = shard.step(params[sl])
        assert torch.equal(s_info["trajectory_length"], full[4][sl]) and torch.equal(s_te, full[2][sl])
        assert torch.equal(s_tr, full[3][sl]) and torch.equal(s_obs, full[0][sl])
        assert torch.equal(torch.nan_to_num(s_ret, neginf=-1e300), torch.nan_to_num(full[1][sl], neginf=-1e300))

    # ---- a random subset against the oracle ----
    idx = np.sort(np.random.default_rng(0).choice(B, size=SUBSET, replace=False))
    it = torch.as_tensor(idx, device=dev)
    sub = [x[it].cpu().numpy() for x in full]
    orc = make_oracle(env_id, mode="mirror", mp_overrides={"env": env_kw})
    orc.reset(seeds=seed + idx)
    o_obs, o_ret, o_te, o_tr, o_info = orc.step(params[it].cpu().numpy())
    tie = o_info["min_margin"] < TIE_EPS
    agree = (sub[4] == o_info["trajectory_length"]) & (sub[2] == o_te) & (sub[3] == o_tr)
    assert (agree | tie).all(), f"{name}: {(~(agree | tie)).sum()} flag / length mismatches outside boundary ties"
    assert (~agree).sum() <= max(2, SUBSET // 500), f"{name}: {(~agree).sum()} boundary ties resolved differently"
    fin = agree & np.isfinite(o_ret)
    assert not fin.any() or rel_err(sub[1][fin], o_ret[fin]).max() < 1e-5
    assert np.array_equal(sub[1][agree & ~np.isfinite(o_ret)], o_ret[agree & ~np.isfinite(o_ret)])
    assert (np.abs(sub[0][agree] - o_obs[agree]) <= 1e-5 * np.maximum(1.0, np.abs(o_obs[agree]))).all()
    if sigma >= 1.0 and "HoleReacher" in env_id:
        assert sub[2].mean() > 0.5           # the divergent regime: most episodes end in a collision
