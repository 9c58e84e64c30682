"""VecNormalize without a GPU: the numpy restatement of SB3 1.6's RunningMeanStd / VecNormalize (tests/vecnorm_ref.py)
checked against itself, the vectorised rank-order combination the data-parallel VecNormalize uses, its construction
verdict, and the r6_vn_* argument checks that return R6_EINVAL before any CUDA call."""
import numpy as np
import pytest
import torch

import vecnorm_ref as vr


def test_two_halves_equal_one_update():
    """update(a); update(b) equals update(a ∪ b) to a stated bound: the two paths differ only in rounding, a few float64
    roundings of values no larger than the data's second moment (mean) and its square (var), so 64 u of that scale."""
    rng = np.random.default_rng(0)
    x = rng.normal(3.0, 2.0, (4097, 13)) * rng.uniform(0.1, 10, 13)
    one, two = vr.RunningMeanStd(shape=(13,)), vr.RunningMeanStd(shape=(13,))
    one.update(x)
    two.update(x[:2000])
    two.update(x[2000:])
    u = 2.0 ** -53
    s = np.max(np.abs(x), axis=0) + 1
    assert np.all(np.abs(one.mean - two.mean) <= 64 * u * s)
    assert np.all(np.abs(one.var - two.var) <= 64 * u * s * s)
    assert one.count == two.count == 4097 + 1e-4
    assert not np.array_equal(one.var, two.var) or not np.array_equal(one.mean, two.mean)   # really two paths


def test_initial_statistics_and_first_update():
    """RunningMeanStd(1e-4): mean 0, var 1, count 1e-4; the first update weighs them by 1e-4."""
    r = vr.RunningMeanStd(shape=(2,))
    assert np.array_equal(r.as_row(), [0, 0, 1, 1, 1e-4])
    r.update(np.array([[1.0, 2.0], [3.0, 2.0]]))
    tot = 1e-4 + 2
    assert np.allclose(r.mean, np.array([2.0, 2.0]) * 2 / tot, rtol=1e-15)
    assert np.allclose(r.var, (1e-4 + np.array([1.0, 0.0]) * 2 + np.array([4.0, 4.0]) * 1e-4 * 2 / tot) / tot, rtol=1e-15)


def test_returns_reset_at_dones():
    ref = vr.VecNormalizeRef(3, gamma=0.5)
    obs = np.zeros((3, 13), np.float32)
    ref.reset(obs)
    ref.step_wait(obs, np.float32([1, 2, 4]), [False, True, False])
    assert np.array_equal(ref.returns, [1.0, 0.0, 4.0])
    ref.step_wait(obs, np.float32([1, 1, 1]), [False, False, True])
    assert np.array_equal(ref.returns, [1.5, 1.0, 0.0])
    # ret_rms saw the returns before the reset: (1, 2, 4), then (1.5, 1, 3)
    want = vr.RunningMeanStd()
    want.update(np.array([1.0, 2.0, 4.0]))
    want.update(np.array([1.5, 1.0, 3.0]))
    assert np.array_equal(ref.ret_rms.as_row(), want.as_row())


def test_clipping_at_both_signs():
    mean, var = np.zeros(13), np.full(13, 1e-6)
    obs = np.zeros((2, 13), np.float32)
    obs[0, :3] = [1.0, -1.0, 1e-6]
    out = vr.normalize_obs(obs, mean, var, 1e-8, 10.0)
    assert out[0, 0] == 10.0 and out[0, 1] == -10.0 and 0 < out[0, 2] < 10.0 and out[1, 0] == 0.0
    r = vr.normalize_reward(np.float32([100.0, -100.0, 0.5]), 1.0, 1e-8, 5.0)
    assert r[0] == 5.0 and r[1] == -5.0 and r[2] == np.float32(0.5 / np.sqrt(1.0 + 1e-8))
    assert out.dtype == np.float32 and r.dtype == np.float32


def test_norm_reward_off_still_updates_ret_rms():
    """SB3 updates ret_rms whenever training, with or without norm_reward; without training neither statistic moves."""
    obs = np.ones((2, 13), np.float32)
    a = vr.VecNormalizeRef(2, norm_reward=False)
    a.reset(obs)
    _, rew, _ = a.step_wait(obs, np.float32([1, 3]), [False, False])
    assert np.array_equal(rew, np.float32([1, 3])) and a.ret_rms.count > 1
    b = vr.VecNormalizeRef(2, training=False)
    b.reset(obs)
    b.step_wait(obs, np.float32([1, 3]), [False, False])
    assert b.obs_rms.count == b.ret_rms.count == 1e-4


def test_vectorised_rank_order_combination():
    """VecNormalize.combine passes gathered rows [W, 3, R] to ppo.combine_moments: the result per row is the numpy
    twin's rank-order combination of that row's [W, 3], bit for bit."""
    from rl_rocket_6dof_b200.ppo import combine_moments
    rng = np.random.default_rng(1)
    for W in (1, 2, 3, 8):
        rows = np.stack([np.stack([np.full(13, float(rng.integers(1, 1000))), rng.normal(0, 5, 13),
                                   rng.uniform(0, 100, 13)], 1) for _ in range(W)])          # [W, 13, 3]
        got = combine_moments(torch.from_numpy(rows).permute(0, 2, 1)).t().numpy()
        want = np.stack([vr.combine_moments(rows[:, r]) for r in range(13)])
        assert np.array_equal(got, want), W


def test_group_verdict_on_crafted_rows():
    from rl_rocket_6dof_b200.vec_normalize import GROUP_FIELDS, group_errors
    good = np.array([[1, 1, 1, 10.0, 10.0, 0.99, 1e-8, 4096]] * 3, np.float64)
    assert len(GROUP_FIELDS) == good.shape[1] and group_errors(good) == []
    bad = good.copy()
    bad[1, GROUP_FIELDS.index("clip_obs")] = 5.0
    bad[2, GROUP_FIELDS.index("num_envs")] = 2048
    errs = group_errors(bad)
    assert len(errs) == 2 and "clip_obs" in errs[0] and "num_envs" in errs[1]
    # a function of the rows only: every rank holding the gathered rows reaches the same verdict
    assert all(group_errors(bad.copy()) == errs for _ in range(3))


def test_invalid_arguments_without_a_gpu():
    """Every r6_vn_* entry point returns R6_EINVAL before any CUDA call (the pointers below are never dereferenced)."""
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    p = 256                                      # a non-null address: only the argument checks may look at it
    cases = [
        L.r6_vn_moments(None, 8, 13, 0, 8, p, p, None), L.r6_vn_moments(p, 8, 13, 0, 8, None, p, None),
        L.r6_vn_moments(p, 8, 13, 0, 8, p, None, None), L.r6_vn_moments(p, 0, 13, 0, 0, p, p, None),
        L.r6_vn_moments(p, 8, 0, 0, 8, p, p, None), L.r6_vn_moments(p, 8, 13, 4, 5, p, p, None),
        L.r6_vn_moments(p, 8, 13, -1, 4, p, p, None), L.r6_vn_moments(p, 8, 13, 0, 0, p, p, None),
        L.r6_vn_update(None, 13, p, 1, 1e-8, p, None), L.r6_vn_update(p, 13, None, 1, 1e-8, p, None),
        L.r6_vn_update(p, 0, p, 1, 1e-8, p, None), L.r6_vn_update(p, 1025, p, 1, 1e-8, p, None),
        L.r6_vn_update(p, 13, p, -1, 1e-8, p, None), L.r6_vn_update(p, 13, p, 1, -1e-8, p, None),
        L.r6_vn_update(p, 13, p, 1, float("nan"), p, None), L.r6_vn_update(p, 13, p, 1, float("inf"), p, None),
        L.r6_vn_normalize(None, p, 8, 0, 8, p, 0, None, 1, 10.0, None),
        L.r6_vn_normalize(p, None, 8, 0, 8, p, 0, None, 1, 10.0, None),
        L.r6_vn_normalize(p, p, 8, 0, 8, None, 0, None, 1, 10.0, None),
        L.r6_vn_normalize(p, p, -1, 0, 0, p, 0, None, 1, 10.0, None),
        L.r6_vn_normalize(p, p, 8, 4, 5, p, 0, None, 1, 10.0, None),
        L.r6_vn_normalize(p, p, 8, 0, 8, p, 1, None, 1, 10.0, None),
        L.r6_vn_normalize(p, p, 8, 0, 8, p, 0, None, 0, 10.0, None),
        L.r6_vn_normalize(p, p, 8, 0, 8, p, 0, None, 1, 0.0, None),
        L.r6_vn_normalize(p, p, 8, 0, 8, p, 0, None, 1, -1.0, None),
        L.r6_vn_normalize(p, p, 8, 0, 8, p, 0, None, 1, float("nan"), None),
        L.r6_vn_ret_moments(None, p, 4, 8, p, 0.99, p, p, None), L.r6_vn_ret_moments(p, None, 4, 8, p, 0.99, p, p, None),
        L.r6_vn_ret_moments(p, p, 4, 8, None, 0.99, p, p, None), L.r6_vn_ret_moments(p, p, 4, 8, p, 0.99, None, p, None),
        L.r6_vn_ret_moments(p, p, 4, 8, p, 0.99, p, None, None), L.r6_vn_ret_moments(p, p, 0, 8, p, 0.99, p, p, None),
        L.r6_vn_ret_moments(p, p, 4, 0, p, 0.99, p, p, None), L.r6_vn_ret_moments(p, p, 4, 8, p, -0.5, p, p, None),
        L.r6_vn_ret_moments(p, p, 4, 8, p, float("nan"), p, p, None),
        L.r6_vn_scale_rewards(None, 4, 8, p, 10.0, None), L.r6_vn_scale_rewards(p, 4, 8, None, 10.0, None),
        L.r6_vn_scale_rewards(p, 0, 8, p, 10.0, None), L.r6_vn_scale_rewards(p, 4, 0, p, 10.0, None),
        L.r6_vn_scale_rewards(p, 4, 8, p, 0.0, None), L.r6_vn_scale_rewards(p, 4, 8, p, float("nan"), None),
    ]
    assert all(rc == -1 for rc in cases), cases
    assert L.r6_vn_moments_work_bytes(4097, 13) == 3 * 13 * 3 * 8 and L.r6_vn_moments_work_bytes(0, 13) == 0
    assert L.r6_vn_ret_work_bytes(32, 257) == 2 * 8 * 32 * 3 * 8


def test_vec_normalize_refuses_bad_settings():
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    for kw in (dict(clip_obs=0.0), dict(clip_reward=-1.0), dict(epsilon=-1e-8), dict(gamma=float("nan"))):
        with pytest.raises(ValueError):
            VecNormalize(None, **kw)
