"""VecNormalize on the device (r6_vn_*, vec_normalize.VecNormalize, collect_rollout / step_policy / run_montecarlo with
vec_normalize, PPOTrainer(vec_normalize=...)) against the numpy restatement of SB3 1.6 in tests/vecnorm_ref.py.

The collection check drives the restatement with a TWIN batch (same seed, weights and params) stepped by step() with
the collection's clipped env actions; its observations, rewards, dones and terminal observations are raw and never
touch a r6_vn_* kernel.  The restatement is fed the device's batch moments of the twin's raw data (checked against
numpy's float64 two-pass moments by the first tests), so everything downstream of the moments is compared bit for bit."""
import datetime
import os
import time

import numpy as np
import pytest
import torch

import policy_ref as pr
import timeout_ref as tr
import vecnorm_ref as vr
from oracle import gae_oracle
from parity_utils import env_params

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
G, LAM = 0.99, 0.95
F_TRUNC = 0x04
SEP = [dict(pi=[64, 64], vf=[64, 64])]


def _L():
    from rl_rocket_6dof_b200 import _lib
    return _lib, _lib.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dev_moments(x: torch.Tensor, first=0, count=None) -> np.ndarray:
    """r6_vn_moments of rows of the component-major float32 x [rows, n] over [first, first + count): [rows, 3]."""
    _lib, L = _L()
    rows, n = x.shape
    count = n - first if count is None else count
    out = torch.empty(rows, 3, dtype=torch.float64, device=DEV)
    work = torch.empty(max(int(L.r6_vn_moments_work_bytes(count, rows)), 8), dtype=torch.uint8, device=DEV)
    _lib.check(L.r6_vn_moments(x.data_ptr(), n, rows, first, count, out.data_ptr(), work.data_ptr(), _stream()), L)
    return out.cpu().numpy()


def _as_sb3(m):
    """(count, mean, M2) rows [R, 3] -> SB3's (batch_mean, batch_var, batch_count)."""
    return m[:, 1], m[:, 2] / m[0, 0], m[0, 0]


# ----------------------------------------------------------------------------------------------------- 1. moments
@pytest.mark.parametrize("n", [1, 31, 32, 33, 4097, (1 << 20) + 5])
def test_moments_against_float64_two_pass(n):
    rng = np.random.default_rng(n)
    x = (rng.normal(0, 1, (13, n)) * rng.uniform(0.01, 100, (13, 1)) + rng.uniform(-50, 50, (13, 1))).astype(np.float32)
    x[3] = 0.25                                    # a constant row: M2 exactly 0
    x[4] = np.float32(1e6) + x[4] * np.float32(1e-3)   # a large offset against a small spread
    xd = torch.from_numpy(x).to(DEV)
    ranges = [(0, n)] + ([(1, n - 1), (n // 3, n - n // 3 - 1)] if n > 2 else [])
    for first, count in ranges:
        got = _dev_moments(xd, first, count)
        sl = x[:, first:first + count].astype(np.float64)
        mean = sl.mean(1)
        m2 = ((sl - mean[:, None]) ** 2).sum(1)
        parts = -(-count // 2048)
        assert np.all(got[:, 0] == count)
        for r in range(13):
            bm, bm2 = vr.moments_bound(sl[r], parts, 8)
            assert abs(got[r, 1] - mean[r]) <= bm, (first, count, r)
            assert abs(got[r, 2] - m2[r]) <= bm2, (first, count, r)
        assert got[3, 1] == 0.25 and got[3, 2] == 0.0
        # bit-reproducible: a rerun, and a run on another stream
        assert np.array_equal(got, _dev_moments(xd, first, count))
        with torch.cuda.stream(torch.cuda.Stream()):
            again = _dev_moments(xd, first, count)
        torch.cuda.synchronize()
        assert np.array_equal(got, again)


@pytest.mark.parametrize("n", [1, 33, 4097, (1 << 18) + 3])
def test_return_scan_against_numpy(n):
    """r6_vn_ret_moments: returns bit-exact against numpy's float64 scan, per-step moments within the bound."""
    _lib, L = _L()
    T = 9
    rng = np.random.default_rng(n)
    rew = rng.normal(0, 3, (T, n)).astype(np.float32)
    rew[4, ::7] = 100.0
    done = (rng.random((T, n)) < 0.2).astype(np.uint8)
    ret0 = rng.normal(0, 5, n)
    ret = torch.from_numpy(ret0).to(DEV)
    out = torch.empty(T, 3, dtype=torch.float64, device=DEV)
    work = torch.empty(int(L.r6_vn_ret_work_bytes(T, n)), dtype=torch.uint8, device=DEV)
    rd, dd = torch.from_numpy(rew).to(DEV), torch.from_numpy(done).to(DEV)
    _lib.check(L.r6_vn_ret_moments(rd.data_ptr(), dd.data_ptr(), T, n, ret.data_ptr(), G, out.data_ptr(), work.data_ptr(),
                                   _stream()), L)
    got = out.cpu().numpy()
    r = ret0.copy()
    for t in range(T):
        r = r * G + rew[t].astype(np.float64)
        mean = r.mean()
        bm, bm2 = vr.moments_bound(r, 8 * -(-n // 256), 1)
        assert got[t, 0] == n and abs(got[t, 1] - mean) <= bm and abs(got[t, 2] - ((r - mean) ** 2).sum()) <= bm2, t
        r[done[t] != 0] = 0
    assert np.array_equal(ret.cpu().numpy(), r)


# ------------------------------------------------------------------------------------------------------ 2. update
def test_update_is_update_from_moments_bit_for_bit():
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    _lib, L = _L()
    rng = np.random.default_rng(2)
    env = _mk(64)
    vn = VecNormalize(env)
    ref = vr.RunningMeanStd(shape=(13,))
    assert np.array_equal(vn.obs_rms.cpu().numpy(), ref.as_row())
    hist = torch.empty(2, 2, 13, dtype=torch.float64, device=DEV)
    for step in range(60):
        m = int(rng.integers(1, 5000))
        x = (rng.normal(0, 1, (13, m)) * rng.uniform(0.1, 10, (13, 1)) + step * 0.1).astype(np.float32)
        mom = torch.from_numpy(_dev_moments(torch.from_numpy(x).to(DEV))).to(DEV)
        vn.update(vn.obs_rms, mom, 1, hist)
        ref.update_from_moments(*_as_sb3(mom.cpu().numpy()))
        h = hist.cpu().numpy()
        assert np.array_equal(vn.obs_rms.cpu().numpy(), ref.as_row()), step
        assert np.array_equal(h[1, 0], ref.mean) and np.array_equal(h[1, 1], np.sqrt(ref.var + 1e-8)), step
    # T sequential updates in one launch (the reward pass) equal T single ones
    a, b = vr.RunningMeanStd(), torch.tensor([0.0, 1.0, 1e-4], dtype=torch.float64, device=DEV)
    moms = np.stack([[[float(rng.integers(1, 99)), rng.normal(), rng.uniform(0, 9)]] for _ in range(50)])
    for mm in moms:
        a.update_from_moments(*_as_sb3(mm))
    vn.update(b, torch.from_numpy(moms).to(DEV), 50)
    assert np.array_equal(b.cpu().numpy(), a.as_row())


# --------------------------------------------------------------------------------------------------- 3. normalize
def test_normalize_bit_exact():
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    n = 5000
    env = _mk(n)
    env.reset()
    vn = VecNormalize(env, clip_obs=3.0)
    obs = env.obs.clone()
    for _ in range(5):                                    # rows z and vz start at 0 (ICRange 0): their var tends to 0
        vn.observe(obs)
    o = obs.cpu().numpy()
    const = [r for r in range(13) if np.all(o[r] == o[r, 0])]
    assert const, "the reset observations have a constant row (an IC range of 0)"
    o[0, :50] = 1e4
    o[0, 50:100] = -1e4                                   # beyond +-clip at both signs
    src = torch.from_numpy(o).to(DEV)
    hist = vn.obs_hist(1)
    rms = vn.obs_rms.cpu().numpy()
    want = vr.normalize_obs(o[:13].T, rms[:13], rms[13:26], 1e-8, 3.0).T
    out = torch.full_like(src, 7.0)
    vn.normalize(src, out, hist)
    got = out.cpu().numpy()
    assert np.array_equal(got[:13], want) and np.all(got[13] == 7.0)
    assert np.any(got[:13] == 3.0) and np.any(got[:13] == -3.0)
    # an env range, in place: the rest untouched
    ip = src.clone()
    vn.normalize(ip, ip, hist, 0, 1234, 2000)
    g = ip.cpu().numpy()
    assert np.array_equal(g[:13, 1234:3234], want[:, 1234:3234]) and np.array_equal(g[:, :1234], o[:, :1234])
    assert np.array_equal(g[:, 3234:], o[:, 3234:]) and np.array_equal(g[13], o[13])
    # per-column history rows (a truncation slot layer): step -1 and rows past the history are not written
    h3 = torch.stack([hist[0], hist[0] * 0.5 + 1, hist[0] * 2.0 + 0.5])      # 3 rows
    step = torch.from_numpy(np.arange(n) % 4 - 1).to(torch.int32).to(DEV)   # -1, 0, 1, 2
    sl = src[:13].clone()
    vn.normalize(sl, sl, h3, step=step)
    g, hh = sl.cpu().numpy(), h3.cpu().numpy()
    s = step.cpu().numpy()
    for v in (0, 1):
        cols = s == v
        m_, sd = hh[v + 1, 0], hh[v + 1, 1]
        w = np.clip((o[:13, cols].astype(np.float64) - m_[:, None]) / sd[:, None], -3.0, 3.0).astype(np.float32)
        assert np.array_equal(g[:, cols], w), v
    for v in (-1, 2):
        assert np.array_equal(g[:, s == v], o[:13, s == v]), v


# ------------------------------------------------------------------------------------------------- 4. collection
def _weights(family="sb3_init"):
    w = pr.weights(family)
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(DEV) for k, v in w.items()}


def _mk(n, limit=None, seed=21, **kw):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    ep = env_params()
    if limit is not None:
        ep.max_episode_steps = limit
    return Rocket6DOFBatch(n, params=ep, device=DEV, seed=seed, **kw)


def _values(env, wd, obs_cm: np.ndarray, tc):
    """V of the component-major normalized observations [13, c]: one deterministic policy launch in mode tc."""
    from rl_rocket_6dof_b200 import _lib
    x = torch.from_numpy(np.ascontiguousarray(obs_cm, np.float32)).to(DEV)
    c = x.shape[1]
    act = torch.empty(c, 3, dtype=torch.float32, device=DEV)
    val = torch.empty(c, dtype=torch.float32, device=DEV)
    env._policy(_lib.make_mlp(wd), x.data_ptr(), 0, c, tc, False, 0, act.data_ptr(), None, val.data_ptr(), None,
                torch.cuda.current_stream(env.device))
    return val.cpu().numpy()


def _collect_and_check(n, k, limit, tc, lanes, vkw, seed=71):
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    _lib, L = _L()
    wd = _weights()
    a, b = _mk(n, limit, seed, lanes=lanes, split_step=True), _mk(n, limit, seed, lanes=lanes, split_step=True)
    a.reset(); b.reset()
    vn = VecNormalize(a, gamma=0.9, clip_obs=5.0, clip_reward=4.0, **vkw)
    vn.reset()
    a.reset_stats(); b.reset_stats()
    ro = a.collect_rollout(k, wd, gamma=G, gae_lambda=LAM, tensor_cores=tc, bootstrap_truncated=True, vec_normalize=vn)
    torch.cuda.synchronize()
    # the twin: raw steps with the collection's clipped actions
    ref = vr.VecNormalizeRef(n, gamma=0.9, clip_obs=5.0, clip_reward=4.0, **vkw)
    moments = lambda o: _as_sb3(_dev_moments(torch.from_numpy(np.ascontiguousarray(o.T)).to(DEV)))
    raw0 = b.obs[:13].t().cpu().numpy()
    obs0 = ref.reset(raw0, moments)
    raw = dict(rew=[], done=[], flags=[], obs=[], tobs=[])
    for j in range(k):
        b.step(ro["actions"][j].clamp(-1.0, 1.0).contiguous())
        raw["rew"].append(b.reward_f32.cpu().numpy().copy())
        raw["done"].append(b.done.cpu().numpy().copy())
        raw["flags"].append(b.flags.cpu().numpy().copy())
        raw["obs"].append(b.obs[:13].t().cpu().numpy().copy())
        raw["tobs"].append(b.terminal_obs[:13].t().cpu().numpy().copy())
    rews, dns = np.stack(raw["rew"]), np.stack(raw["done"])
    # the device's per-step return moments of the twin's raw rewards (the scan is checked against numpy above)
    out = torch.empty(k, 3, dtype=torch.float64, device=DEV)
    ret0 = torch.zeros(n, dtype=torch.float64, device=DEV)
    work = torch.empty(int(L.r6_vn_ret_work_bytes(k, n)), dtype=torch.uint8, device=DEV)
    _lib.check(L.r6_vn_ret_moments(torch.from_numpy(rews).to(DEV).data_ptr(), torch.from_numpy(dns).to(DEV).data_ptr(), k, n,
                                   ret0.data_ptr(), 0.9, out.data_ptr(), work.data_ptr(), _stream()), L)
    rmom = out.cpu().numpy()
    obs_n, rew_n, tob_n = [obs0], [], []
    trunc = (np.stack(raw["flags"]) & F_TRUNC) != 0
    for j in range(k):
        tdict = {int(i): raw["tobs"][j][i] for i in np.nonzero(trunc[j])[0]}
        o, r, t = ref.step_wait(raw["obs"][j], raw["rew"][j], raw["done"][j], tdict, moments,
                                lambda _ret, j=j: _as_sb3(rmom[j:j + 1]))
        obs_n.append(o); rew_n.append(r); tob_n.append(t)
    got_obs = ro["obs"].cpu().numpy()                           # [k, n, 13]
    for j in range(k):
        assert np.array_equal(got_obs[j], obs_n[j]), j
    # rewards: SB3's bootstrap of the normalized rewards with V(normalized terminal obs), fl32 at each step
    vals = np.zeros((k, n), np.float32)
    for j in range(k):
        if tob_n[j]:
            idx = np.array(sorted(tob_n[j]))
            vals[j, idx] = _values(a, wd, np.stack([tob_n[j][i] for i in idx]).T, tc)
    want_rew = tr.bootstrap_timeouts(np.stack(rew_n), trunc, vals, G)
    got_rew = ro["rewards"].cpu().numpy()
    assert np.array_equal(got_rew, want_rew), int((got_rew != want_rew).sum())
    assert np.array_equal(ro["dones"].cpu().numpy(), dns)
    last_v = _values(a, wd, ref.normalize_obs(raw["obs"][k - 1]).T, tc)
    assert np.array_equal(ro["last_values"].cpu().numpy(), last_v)
    c = lambda t: t.cpu().numpy()
    adv, ret = gae_oracle.compute_returns_and_advantage(got_rew, c(ro["values"]), c(ro["dones"]) != 0, c(ro["last_values"]),
                                                        G, LAM)
    assert np.array_equal(adv, c(ro["advantages"])) and np.array_equal(ret, c(ro["returns"]))
    # statistics bit-exact given the device moments; within the moments bound of numpy's own two-pass restatement
    assert np.array_equal(c(vn.obs_rms), ref.obs_rms.as_row()) and np.array_equal(c(vn.ret_rms), ref.ret_rms.as_row())
    assert np.array_equal(c(vn.returns), ref.returns)
    # raw state: the batch's obs is the twin's, its episode statistics are the raw rewards' (return_sum is accumulated
    # with atomics, so its last bits depend on the order the CTAs finish in)
    assert torch.equal(a.obs, b.obs)
    sa, sb = a.stats_dict(), b.stats_dict()
    assert sa["return_sum"] == pytest.approx(sb["return_sum"], rel=1e-12, abs=0)
    assert sa["episodes"] == sb["episodes"] and sa["truncated"] > 0
    return ro, vn, trunc, (raw0, raw)


@pytest.mark.parametrize("vkw", [dict(norm_reward=False), dict(norm_obs=False), {}], ids=["obs", "reward", "both"])
@pytest.mark.parametrize("tc", [0, 3])
def test_collection_against_the_restatement(vkw, tc):
    """L = 5, k = 12 from reset(): truncations at steps 4 and 9 inside the window; one and two lanes are checked against
    the twin and are bit-identical to each other."""
    ro1, vn1, trunc, _ = _collect_and_check(3001, 12, 5, tc, 1, vkw)
    ro2, vn2, _, _ = _collect_and_check(3001, 12, 5, tc, 2, vkw)
    assert trunc[4].any() and trunc[9].any()
    for key in ro1:
        assert torch.equal(ro1[key], ro2[key]), key
    for t in ("obs_rms", "ret_rms", "returns"):
        assert torch.equal(getattr(vn1, t), getattr(vn2, t)), t


def test_collection_statistics_against_float64_moments():
    """Both normalizations, 2^16 + 7 envs: the running statistics against the restatement with numpy's own float64
    two-pass moments.  An update is a weighted mean of the old statistics and the batch's, so it does not amplify a
    moment's error: the statistics stay within the per-step moments bound (test_moments_against_float64_two_pass; about
    1e-13 relative at this size), asserted here as a relative 1e-12."""
    n, k = (1 << 16) + 7, 6
    ro, vn, _, (raw0, raw) = _collect_and_check(n, k, 4, 3, 2, {})
    pure = vr.VecNormalizeRef(n, gamma=0.9, clip_obs=5.0, clip_reward=4.0)
    pure.reset(raw0)
    for j in range(k):
        pure.step_wait(raw["obs"][j], raw["rew"][j], raw["done"][j])
    for got, want in ((vn.obs_rms, pure.obs_rms.as_row()), (vn.ret_rms, pure.ret_rms.as_row())):
        g = got.cpu().numpy()
        assert np.all(np.abs(g - want) <= 1e-12 * (np.abs(want) + 1e-3)), np.max(np.abs(g - want) / (np.abs(want) + 1e-3))
    assert np.array_equal(vn.returns.cpu().numpy(), pure.returns)


def test_collection_refuses_one_episode_batches():
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    env = _mk(64, auto_reset=False)
    env.reset()
    with pytest.raises(ValueError):
        env.collect_rollout(2, _weights(), vec_normalize=VecNormalize(env))
    other = _mk(64)
    with pytest.raises(ValueError):
        _mk(64).collect_rollout(2, _weights(), vec_normalize=VecNormalize(other))


# ---------------------------------------------------------------------------------------------------- 5. trainer
ATOMIC_LOGS = ("rollout/return_sum", "rollout/mean_return")     # episode sums accumulated with atomics


def _logs_equal(l1: dict, l2: dict) -> bool:
    """Bit-equal logs, except the episode return sums, whose last bits depend on the atomics' order: relative 1e-12."""
    return l1.keys() == l2.keys() and all(l1[k] == l2[k] if k not in ATOMIC_LOGS else l1[k] == pytest.approx(l2[k], rel=1e-12)
                                          for k in l1)


LAYOUTS = {"shared": ({}, {}), "sde": (dict(use_sde=True), dict(use_sde=True)), "sep": (dict(net_arch=SEP), {}),
           "sepsde": (dict(use_sde=True, net_arch=SEP), dict(use_sde=True, sde_sample_freq=4))}


def _train(layout, vf, tmp=None):
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    pk, ck = LAYOUTS[layout]
    env = _mk(512, 6, 13, lanes=2, split_step=True)
    params = ActorCriticParams.sb3_init(seed=3, device=DEV, **pk)
    vn = VecNormalize(env)
    cfg = PPOConfig(n_steps=8, n_epochs=2, clip_range_vf=0.2 if vf else None, **ck)
    tr_ = PPOTrainer(env, params, cfg, seed=5, vec_normalize=vn)
    logs = tr_.learn(3 * 8 * 512)
    return logs, params, vn


@pytest.mark.parametrize("vf", [False, True])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_learn_on_every_layout(layout, vf, tmp_path):
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    logs, params, vn = _train(layout, vf)
    assert len(logs) == 3
    for log in logs:
        assert all(np.isfinite(v) for k, v in log.items() if k != "train/explained_variance"), log
        assert log["rollout/episodes"] > 0
    assert float(vn.obs_rms[-1]) == pytest.approx(1e-4 + 512 * (1 + 3 * 8))      # reset + every collected step
    assert float(vn.ret_rms[-1]) == pytest.approx(1e-4 + 512 * 3 * 8)
    logs2, params2, vn2 = _train(layout, vf)
    assert torch.equal(params.flat, params2.flat) and torch.equal(vn.obs_rms, vn2.obs_rms)       # reproducible
    for l1, l2 in zip(logs, logs2):
        assert _logs_equal(l1, l2)
    p = str(tmp_path / "vn.npz")
    vn.save(p)
    z = np.load(p)
    assert "returns" not in z.files and {"obs_rms.mean", "obs_rms.var", "obs_rms.count", "ret_rms.var"} <= set(z.files)
    back = VecNormalize(_mk(512), training=False, clip_obs=1.0).load(p)
    assert torch.equal(back.obs_rms, vn.obs_rms) and torch.equal(back.ret_rms, vn.ret_rms)
    assert back.clip_obs == vn.clip_obs and back.training == vn.training and back.gamma == vn.gamma


def test_trainer_checks_its_vec_normalize():
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOTrainer
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    env = _mk(64)
    with pytest.raises(ValueError):
        PPOTrainer(env, ActorCriticParams.sb3_init(device=DEV), vec_normalize=VecNormalize(_mk(64)))


# --------------------------------------------------------------------------------------------- 6. frozen statistics
@pytest.mark.parametrize("tc,lanes", [(0, 1), (3, 2)])
def test_step_policy_with_frozen_statistics(tc, lanes):
    from rl_rocket_6dof_b200 import _lib
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    wd = _weights("golden")
    n, k = 4099, 5
    a, b = _mk(n, seed=81, lanes=lanes, split_step=True), _mk(n, seed=81, lanes=lanes, split_step=True)
    a.reset(); b.reset()
    vn = VecNormalize(a, training=False, clip_obs=2.0)
    vn.obs_rms[:13] = torch.linspace(-0.5, 0.5, 13, dtype=torch.float64)
    vn.obs_rms[13:26] = torch.linspace(0.01, 4.0, 13, dtype=torch.float64)
    before = vn.obs_rms.clone(), vn.ret_rms.clone()
    a.step_policy(k, wd, tensor_cores=tc, vec_normalize=vn)
    rms = vn.obs_rms.cpu().numpy()
    act = torch.empty(n, 3, dtype=torch.float32, device=DEV)
    for j in range(k):
        x = vr.normalize_obs(b.obs[:13].t().cpu().numpy(), rms[:13], rms[13:26], 1e-8, 2.0).T
        xd = torch.from_numpy(np.ascontiguousarray(x)).to(DEV)
        b._policy(_lib.make_mlp(wd), xd.data_ptr(), 0, n, tc, False, b.steps_done, act.data_ptr(), None, None, None,
                  torch.cuda.current_stream(b.device))
        b.step(act)
    torch.cuda.synchronize()
    assert torch.equal(a._policy_act, act) and torch.equal(a.obs, b.obs) and torch.equal(a.state, b.state)
    assert torch.equal(vn.obs_rms, before[0]) and torch.equal(vn.ret_rms, before[1])


def test_montecarlo_with_frozen_statistics(tmp_path):
    """Identity statistics (mean 0, var 1, eps 0, a wide clip) reproduce the run without them bit for bit; real
    statistics change the actions; a .npz path works as the CLI passes it; the fused kernel is refused."""
    from rl_rocket_6dof_b200 import montecarlo, policy
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    w = pr.weights("golden")
    kw = dict(seed=5, two_kernel=True, tensor_cores=True, chunk_steps=32)
    base = montecarlo.run_montecarlo(300, w, **kw)
    ident = VecNormalize(_mk(8), training=False, clip_obs=1e30, epsilon=0.0)
    same = montecarlo.run_montecarlo(300, w, vec_normalize=ident, **kw)
    assert np.array_equal(base["terminal_state"], same["terminal_state"])
    real = VecNormalize(_mk(8), training=False)
    real.obs_rms[:13] = 0.1
    real.obs_rms[13:26] = 0.5
    p = str(tmp_path / "stats.npz")
    real.save(p)
    other = montecarlo.run_montecarlo(300, w, vec_normalize=p, **kw)
    assert not np.array_equal(base["terminal_state"], other["terminal_state"])
    assert np.array_equal(other["terminal_state"], montecarlo.run_montecarlo(300, w, vec_normalize=real, **kw)["terminal_state"])
    with pytest.raises(ValueError):
        montecarlo.run_montecarlo(300, w, vec_normalize=p, two_kernel=False)


# ---------------------------------------------------------------------------------------------- 7. data-parallel
N_DP = 256


def _dp_learn(rank, world, dev, group, clip_obs=10.0):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    from rl_rocket_6dof_b200.sharding import shard_batch_kwargs
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    ep = env_params()
    ep.max_episode_steps = 6
    env = Rocket6DOFBatch(N_DP, params=ep, device=dev, seed=31, **shard_batch_kwargs(N_DP, rank, world))
    vn = VecNormalize(env, group=group, clip_obs=clip_obs)
    params = ActorCriticParams.sb3_init(seed=7, device=dev)
    trainer = PPOTrainer(env, params, PPOConfig(n_steps=8, n_epochs=2), seed=9, group=group, vec_normalize=vn)
    logs = trainer.learn(2 * 8 * N_DP * world)
    keys = sorted(logs[0])
    return dict(flat=params.flat.cpu().numpy(), obs_rms=vn.obs_rms.cpu().numpy(), ret_rms=vn.ret_rms.cpu().numpy(),
                logs=np.array([[float(l[k]) for k in keys] for l in logs]), keys=np.array(keys))


def _dp_worker(rank, world, store_path, out_path):
    import torch.distributed as dist
    dev = torch.device(DEV)
    torch.cuda.set_device(dev)
    store = dist.FileStore(store_path, world)
    dist.init_process_group("gloo", store=store, rank=rank, world_size=world, timeout=datetime.timedelta(seconds=240))
    try:
        res = {}
        for rep in range(2):
            for k, v in _dp_learn(rank, world, dev, dist.group.WORLD).items():
                res[f"dp{rep}/{k}"] = v
        singles = [dist.new_group([r]) for r in range(world)]
        for tag, grp in (("one", singles[rank]), ("none", None)):
            for k, v in _dp_learn(0, 1, dev, grp).items():
                res[f"{tag}/{k}"] = v
        # the per-step combination is combine_moments of the gathered rows
        from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
        from rl_rocket_6dof_b200.ppo import combine_moments
        from rl_rocket_6dof_b200.sharding import shard_batch_kwargs
        from rl_rocket_6dof_b200.vec_normalize import VecNormalize
        env = Rocket6DOFBatch(N_DP, device=dev, seed=31, **shard_batch_kwargs(N_DP, rank, world))
        env.reset()
        vn = VecNormalize(env, group=dist.group.WORLD)
        local = vn.obs_moments(env.obs).clone()
        rows = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(rows, local)
        want = torch.stack([combine_moments(torch.stack([r[c] for r in rows])) for c in range(13)])
        res["combine_ok"] = np.array(torch.equal(vn.combine(local), want))
        try:
            _dp_learn(rank, world, dev, dist.group.WORLD, clip_obs=10.0 if rank == 0 else 5.0)
            res["bad_error"] = np.array("")
        except ValueError as e:
            res["bad_error"] = np.array(str(e))
        dist.barrier()
        np.savez(out_path, **res)
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module")
def dp_runs(tmp_path_factory):
    import torch.multiprocessing as mp
    tmp = str(tmp_path_factory.mktemp("vn_gloo"))
    ctx = mp.get_context("spawn")
    outs = [os.path.join(tmp, f"rank{r}.npz") for r in range(2)]
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, os.path.join(tmp, "store"), outs[r])) for r in range(2)]
    for p in procs:
        p.start()
    deadline = time.monotonic() + 900
    try:
        for p in procs:
            p.join(timeout=max(1.0, deadline - time.monotonic()))
    finally:
        survivors = [p for p in procs if p.is_alive()]
        for p in survivors:
            p.terminate()
            p.join(timeout=30)
            if p.is_alive():
                p.kill()
                p.join()
    assert not survivors and [p.exitcode for p in procs] == [0, 0]
    return [dict(np.load(o)) for o in outs]


def _dp_same(r, a, b):
    """Runs a and b of result r: parameters and statistics bit-identical, logs as _logs_equal."""
    for k in ("flat", "obs_rms", "ret_rms"):
        assert np.array_equal(r[0][f"{a}/{k}"], r[1][f"{b}/{k}"]), (a, b, k)
    keys = list(r[0][f"{a}/keys"])
    assert keys == list(r[1][f"{b}/keys"])
    for la, lb in zip(r[0][f"{a}/logs"], r[1][f"{b}/logs"]):
        assert _logs_equal(dict(zip(keys, la)), dict(zip(keys, lb))), (a, b)


def test_dp_ranks_bit_identical(dp_runs):
    r0, r1 = dp_runs
    for k in ("flat", "obs_rms", "ret_rms", "logs"):                # the group's statistics and logs: same on both ranks
        assert np.array_equal(r0[f"dp0/{k}"], r1[f"dp0/{k}"]), k
    _dp_same((r0, r0), "dp0", "dp1")                                # a rerun
    assert r0["dp0/obs_rms"][-1] == pytest.approx(1e-4 + 2 * N_DP * (1 + 2 * 8))
    assert not np.array_equal(r0["dp0/obs_rms"], r0["none/obs_rms"])
    for r in dp_runs:
        _dp_same((r, r), "one", "none")
        assert bool(r["combine_ok"])
    msgs = [str(r["bad_error"]) for r in dp_runs]
    assert all("clip_obs" in m for m in msgs) and msgs[0] == msgs[1], msgs


# ------------------------------------------------------------------------------------------- 8. argument checks
def test_einval_writes_nothing():
    _lib, L = _L()
    n = 64
    x = torch.ones(14, n, dtype=torch.float32, device=DEV)
    out = torch.full((13, 3), 7.0, dtype=torch.float64, device=DEV)
    work = torch.zeros(4096, dtype=torch.uint8, device=DEV)
    rms = torch.full((27,), 3.0, dtype=torch.float64, device=DEV)
    hist = torch.full((2, 2, 13), 5.0, dtype=torch.float64, device=DEV)
    y = torch.full((14, n), 9.0, dtype=torch.float32, device=DEV)
    rew = torch.full((4, n), 2.0, dtype=torch.float32, device=DEV)
    dn = torch.zeros(4, n, dtype=torch.uint8, device=DEV)
    ret = torch.full((n,), 4.0, dtype=torch.float64, device=DEV)
    rh = torch.full((5, 2, 1), 6.0, dtype=torch.float64, device=DEV)
    snaps = [t.clone() for t in (out, work, rms, hist, y, rew, ret, rh)]
    P = lambda t: t.data_ptr()
    s = _stream()
    cases = [
        L.r6_vn_moments(P(x), n, 13, 0, 0, P(out), P(work), s), L.r6_vn_moments(P(x), n, 13, 10, n, P(out), P(work), s),
        L.r6_vn_moments(P(x), n, 0, 0, n, P(out), P(work), s), L.r6_vn_moments(P(x), n, 13, 0, n, P(out), None, s),
        L.r6_vn_update(P(rms), 13, P(out), 1, -1.0, P(hist), s), L.r6_vn_update(P(rms), 0, P(out), 1, 1e-8, P(hist), s),
        L.r6_vn_update(P(rms), 13, None, 1, 1e-8, P(hist), s), L.r6_vn_update(P(rms), 13, P(out), -2, 1e-8, P(hist), s),
        L.r6_vn_normalize(P(x), P(y), n, 0, n, P(hist), 0, None, 2, 0.0, s),
        L.r6_vn_normalize(P(x), P(y), n, 0, n, P(hist), 2, None, 2, 10.0, s),
        L.r6_vn_normalize(P(x), P(y), n, 1, n, P(hist), 0, None, 2, 10.0, s),
        L.r6_vn_normalize(P(x), P(y), n, 0, n, None, 0, None, 2, 10.0, s),
        L.r6_vn_ret_moments(P(rew), P(dn), 4, n, P(ret), 0.99, P(out), None, s),
        L.r6_vn_ret_moments(P(rew), P(dn), 0, n, P(ret), 0.99, P(out), P(work), s),
        L.r6_vn_ret_moments(P(rew), P(dn), 4, n, P(ret), float("inf"), P(out), P(work), s),
        L.r6_vn_scale_rewards(P(rew), 4, n, P(rh), -1.0, s), L.r6_vn_scale_rewards(P(rew), 4, 0, P(rh), 10.0, s),
        L.r6_vn_scale_rewards(P(rew), 4, n, None, 10.0, s),
    ]
    torch.cuda.synchronize()
    assert all(rc == -1 for rc in cases), cases
    for a, b in zip((out, work, rms, hist, y, rew, ret, rh), snaps):
        assert torch.equal(a, b)
