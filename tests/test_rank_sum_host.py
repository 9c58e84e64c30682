"""Host checks of the data-parallel trainer's arithmetic (rl_rocket_6dof_b200.ppo): the rank-order Chan combination of
per-rank (count, mean, M2) against numpy in float64, the stratified minibatch slices, the rank-order sum that
r6_rank_sum states (restated in numpy, with a case where the order matters), and the construction-time consistency
verdict."""
import numpy as np
import pytest
import torch

from rl_rocket_6dof_b200 import ppo
from rl_rocket_6dof_b200.sharding import shard_batch_kwargs


def _sets(seed, sizes):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal(k) * 10.0 ** rng.uniform(-2, 2) + rng.uniform(-50, 50) for k in sizes]


@pytest.mark.parametrize("sizes", [[7], [1, 1], [5, 9, 2], [1000, 3, 250, 17, 1, 64, 9, 500]])
def test_combine_moments_matches_numpy(sizes):
    """Unequal counts, means and spreads per rank: the combined mean and unbiased variance are those of the concatenated
    float64 data within float64 round-off."""
    xs = _sets(len(sizes), sizes)
    rows = torch.stack([ppo.local_moments(torch.from_numpy(x)) for x in xs])
    for x, r in zip(xs, rows.numpy()):
        assert r[0] == len(x) and abs(r[1] - x.mean()) <= 1e-14 * np.abs(x).max()
        assert abs(r[2] - ((x - x.mean()) ** 2).sum()) <= 1e-12 * ((x - x.mean()) ** 2).sum() + 1e-300
    n, mean, m2 = ppo.combine_moments(rows).numpy()
    allx = np.concatenate(xs)
    assert n == len(allx)
    assert abs(mean - allx.mean()) <= 1e-13 * np.abs(allx).max()
    if len(allx) > 1:
        var = allx.var(ddof=1)
        assert abs(m2 / (n - 1) - var) <= 1e-12 * var


def test_combine_moments_one_rank_is_the_row():
    x = torch.from_numpy(_sets(3, [33])[0])
    row = ppo.local_moments(x)
    assert torch.equal(ppo.combine_moments(row[None]), row)


def test_combine_moments_is_rank_ordered():
    """The result is a function of the rows in their order: the same rows in another order may give other bits, and
    the same rows always give the same bits."""
    rows = torch.stack([ppo.local_moments(torch.from_numpy(x)) for x in _sets(5, [3, 1000, 7])])
    a, b = ppo.combine_moments(rows), ppo.combine_moments(rows.clone())
    assert torch.equal(a, b)
    n, mean, m2 = ppo.combine_moments(rows.flip(0))
    assert n == a[0] and abs(mean - a[1]) <= 1e-13 * abs(a[1]) and abs(m2 - a[2]) <= 1e-12 * a[2]


@pytest.mark.parametrize("T,n,bs,world", [(4, 6, 8, 2), (4, 6, 24, 1), (3, 5, 6, 3), (8, 16, 64, 8), (2, 3, 4, 2),
                                          (5, 7, 35, 1)])
def test_minibatch_slices_are_a_stratified_partition(T, n, bs, world):
    """Every rank's slices partition its T n samples in order; each global minibatch takes bs / world from every rank
    (the last one possibly short, equally on every rank); W = 1 is the single-GPU split range(0, T n, bs)."""
    total = T * n
    sl = ppo.minibatch_slices(total, bs, world)
    b = bs // world
    assert [s for s, _ in sl] == list(range(0, total, b))
    assert sl[-1][1] == total and all(e - s == b for s, e in sl[:-1]) and 0 < sl[-1][1] - sl[-1][0] <= b
    if world == 1:
        assert sl == [(s, min(s + bs, total)) for s in range(0, total, bs)]
    # global sample ids of minibatch k (rank r's local sample t n + i is t (W n) + r n + i): disjoint, and their union
    # over the epoch is the whole W n-env rollout
    rng = np.random.default_rng(T * n + bs)
    perms = [rng.permutation(total) for _ in range(world)]
    glob = lambda r, s: (s // n) * (world * n) + r * n + s % n
    seen = []
    for s, e in sl:
        mb = np.concatenate([glob(r, perms[r][s:e]) for r in range(world)])
        assert len(mb) == world * (e - s) and len(np.unique(mb)) == len(mb)
        seen.append(mb)
    assert np.array_equal(np.sort(np.concatenate(seen)), np.arange(world * total))


def test_minibatch_slices_refuse_a_non_multiple():
    with pytest.raises(ValueError):
        ppo.minibatch_slices(100, 10, 3)
    with pytest.raises(ValueError):
        ppo.minibatch_slices(100, 0, 1)


def rank_sum_ref(rows):
    """r6_rank_sum's statement in numpy: float64 accumulation in rank order from 0, one rounding to float32."""
    acc = np.zeros(rows.shape[1])
    for r in rows:
        acc = acc + r.astype(np.float64)
    return acc


def test_rank_sum_order_matters_on_crafted_rows():
    """1 + 1e30 - 1e30 in rank order is 0 and in reverse order 1: what a GPU check of r6_rank_sum uses as teeth."""
    g = np.array([[1.0], [1e30], [-1e30]], np.float32)
    assert rank_sum_ref(g).astype(np.float32)[0] == 0.0
    assert rank_sum_ref(g[::-1]).astype(np.float32)[0] == 1.0


def _row(**kw):
    v = dict(num_envs=8, env_offset=0, num_envs_global=16, nparams=10311, use_sde=0, separate=0, env_seed_hi=0,
             env_seed_lo=5, local_error=0, learning_rate=3e-4, n_steps=4, batch_size=np.inf, n_epochs=2, gamma=0.99,
             gae_lambda=0.95, clip_range=0.2, normalize_advantage=1, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5,
             target_kl=np.inf, tensor_cores=3, cfg_use_sde=0, sde_sample_freq=-1, clip_range_vf=np.inf)
    v.update(kw)
    return [float(v[k]) for k in ppo._DP_FIELDS]


def test_group_errors():
    ok = np.array([_row(), _row(env_offset=8)])
    assert ppo._group_errors(ok, 2) == []
    assert ppo._group_errors(np.array([_row(num_envs_global=8)]), 1) == []
    bad = ppo._group_errors(np.array([_row(), _row(env_offset=0)]), 2)
    assert len(bad) == 1 and "env_offset" in bad[0]
    assert any("gamma" in e for e in ppo._group_errors(np.array([_row(), _row(env_offset=8, gamma=0.9)]), 2))
    assert any("batch_size" in e for e in ppo._group_errors(np.array([_row(batch_size=9), _row(env_offset=8, batch_size=9)]), 2))
    assert any("num_envs_global" in e for e in ppo._group_errors(np.array([_row(num_envs_global=24),
                                                                           _row(env_offset=8, num_envs_global=24)]), 2))
    assert any("rank 1" in e for e in ppo._group_errors(np.array([_row(), _row(env_offset=8, local_error=2)]), 2))


def test_shard_batch_kwargs():
    assert shard_batch_kwargs(8, 0, 1) == dict(env_offset=0, num_envs_global=8)
    assert shard_batch_kwargs(1 << 20, 7, 8) == dict(env_offset=7 << 20, num_envs_global=8 << 20)
    for bad in ((0, 0, 1), (8, 2, 2), (8, -1, 2), (8, 0, 0)):
        with pytest.raises(ValueError):
            shard_batch_kwargs(*bad)
