"""Bootstrapping of TimeLimit truncations during collection (collect_rollout(..., bootstrap_truncated=True),
r6_trunc_record / r6_trunc_bootstrap) against SB3's timeout handling (tests/timeout_ref.py).

The independent expectation is a TWIN batch (same seed, weights and env params) stepped by policy_forward(stochastic)
+ step(): after each step its reward_f32, flags and terminal observations are read and V(terminal observation) is one
r6_policy_range launch in the collection's mode.  None of that path uses the new kernels."""
import numpy as np
import pytest
import torch

import policy_ref as pr
import timeout_ref as tr
from oracle import gae_oracle
from parity_utils import env_params

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
G, LAM = 0.99, 0.95
F_OOB, F_TRUNC = 0x02, 0x04


def _weights(family):
    w = pr.weights(family)
    return w, {k: torch.from_numpy(np.ascontiguousarray(v)).to(DEV) for k, v in w.items()}


def _mk(n, limit=None, seed=21, **kw):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    ep = env_params()
    if limit is not None:
        ep.max_episode_steps = limit
    return Rocket6DOFBatch(n, params=ep, device=DEV, seed=seed, **kw)


def _values(env, wd, obs, tc):
    """V of the component-major observations obs [>= 13, n]: one r6_policy_range launch, mode tc, deterministic."""
    from rl_rocket_6dof_b200 import _lib
    n = obs.shape[1]
    act = torch.empty(n, 3, dtype=torch.float32, device=DEV)
    val = torch.empty(n, dtype=torch.float32, device=DEV)
    env._policy(_lib.make_mlp(wd), obs.data_ptr(), 0, n, tc, False, 0, act.data_ptr(), None, val.data_ptr(), None,
                torch.cuda.current_stream(env.device))
    return val


def _twin(env, wd, k, tc, cols=None):
    """k steps of policy_forward(stochastic=True, step_index) + step(); per step (columns `cols`, default all): rew, flags,
    val = V(terminal_obs), val_reset = V(obs after the step, the reset observation of a finished env), tobs = terminal
    observation rows 0..12 [k, 13, c]."""
    out = {key: [] for key in ("rew", "flags", "val", "val_reset", "tobs")}
    sel = (lambda t: t) if cols is None else (lambda t: t[..., cols])
    for _ in range(k):
        a, _, _, _ = env.policy_forward(wd, stochastic=True, tensor_cores=tc, step_index=env.steps_done)
        env.step(a)
        out["rew"].append(sel(env.reward_f32).clone())
        out["flags"].append(sel(env.flags).clone())
        out["val"].append(sel(_values(env, wd, env.terminal_obs, tc)))
        out["val_reset"].append(sel(_values(env, wd, env.obs, tc)))
        out["tobs"].append(sel(env.terminal_obs[:13]).clone())
    return {key: torch.stack(v).cpu().numpy() for key, v in out.items()}


def _check(ro, tw, cols=None):
    """The collection's rewards bit for bit against SB3's bootstrap of the twin's, the bootstrapped set = the twin's
    F_TRUNCATED set, and advantages / returns bit-exact against the GAE restatement on those rewards.  Returns
    (rewards, truncated mask) of the columns."""
    c = (lambda t: t.cpu().numpy()) if cols is None else (lambda t: t[..., cols].cpu().numpy())
    rew = c(ro["rewards"])
    trunc = (tw["flags"] & F_TRUNC) != 0
    want = tr.bootstrap_timeouts(tw["rew"], trunc, tw["val"], G)
    assert np.array_equal(rew[~trunc], tw["rew"][~trunc])                 # every other reward is the twin's
    assert np.array_equal(rew, want), int((rew != want).sum())
    assert np.array_equal(rew != tw["rew"], trunc)                        # bootstrapped exactly where truncated
    adv, ret = gae_oracle.compute_returns_and_advantage(rew, c(ro["values"]), c(ro["dones"]) != 0, c(ro["last_values"]),
                                                        G, LAM)
    assert np.array_equal(adv, c(ro["advantages"])) and np.array_equal(ret, c(ro["returns"]))
    return rew, trunc


def _wrong(tw, mask, vals):
    return tr.bootstrap_timeouts(tw["rew"], mask, vals, G)


@pytest.mark.parametrize("family,tc", [("sb3_init", 0), ("sb3_init", 3), ("golden", 0), ("golden", 3)])
def test_synchronised_truncations(family, tc):
    """L = 5 from reset(): every env truncates at steps 4, 9 and 14 of a 16-step rollout (4 slots, 3 used)."""
    w, wd = _weights(family)
    n, k = 4096, 16
    a, b = _mk(n, 5), _mk(n, 5)
    a.reset(); b.reset()
    ro = a.collect_rollout(k, wd, gamma=G, gae_lambda=LAM, tensor_cores=tc, bootstrap_truncated=True)
    tw = _twin(b, wd, k, tc)
    rew, trunc = _check(ro, tw)
    assert np.array_equal(np.nonzero(trunc.any(1))[0], [4, 9, 14]) and trunc[[4, 9, 14]].all()
    # V of the terminal observations against the float64 network, within the bound of the mode
    x = tw["tobs"][[4, 9, 14]].transpose(0, 2, 1).reshape(-1, 13)
    v = tw["val"][[4, 9, 14]].reshape(-1).astype(np.float64)
    _, v64 = pr.forward64(w, x)
    r = np.abs(v - v64) / pr.bound(w, x, tc)[:, 3]
    print(f"{family} tensor_cores={tc}: worst |V - forward64| / bound {r.max():.3g} over {len(v)} terminal observations")
    assert r.max() <= pr.C_BAR
    # teeth: V of the reset observation obs[j + 1] instead of the terminal one, and one fused rounding instead of two
    assert (rew != _wrong(tw, trunc, tw["val_reset"]))[trunc].mean() > 0.99
    fma = tw["rew"].copy()
    fma[trunc] = tr.fma_f32(tw["rew"][trunc], np.float32(G), tw["val"][trunc])
    miss = int((rew != fma).sum())
    print(f"{family} tensor_cores={tc}: an FMA-rounded expectation misses {miss} of {int(trunc.sum())} rewards")
    assert miss >= 1


def _place(env, n, limit, phase):
    """Starts every env from its reset state with step_count = phase[i] (so it truncates first at step limit - 1 -
    phase[i]); envs with phase < 0 instead sit just below the upper altitude bound, climbing, with step_count = limit - 1:
    they leave the bounds on step 0, exactly when their count reaches the limit."""
    ic = env.state.t().to(torch.float32).clone()
    oob = torch.from_numpy(np.nonzero(phase < 0)[0]).to(DEV)
    ic[oob, 0] = float(env.params.bounds_high[0]) - 0.1
    ic[oob, 3] = 100.0                      # m/s upwards: out of bounds within the 0.1 s step
    for p in np.unique(phase):
        idx = torch.from_numpy(np.nonzero(phase == p)[0]).to(DEV)
        env.set_state(ic[idx], idx, step_count=int(p) if p >= 0 else limit - 1)


def test_scattered_truncations_and_edges():
    """L = 8, k = 17 (3 slots): envs with step_count 0..7 truncate at every step; those at 7 truncate at steps 0, 8 and 16
    (the first step, the last and the slot maximum ceil(17 / 8)).  Envs that go out of bounds on the step their count
    reaches L are not truncated (gym: TimeLimit.truncated = not done) and must not be bootstrapped."""
    w, wd = _weights("golden")
    n, k, L = 2048, 17, 8
    phase = np.arange(n) % L
    phase[::97] = -1
    a, b = _mk(n, L, 31), _mk(n, L, 31)
    for e in (a, b):
        e.reset()
        _place(e, n, L, phase)
    ro = a.collect_rollout(k, wd, gamma=G, gae_lambda=LAM, bootstrap_truncated=True)
    tw = _twin(b, wd, k, 3)
    rew, trunc = _check(ro, tw)
    last = phase == L - 1
    assert trunc[0].any() and trunc[k - 1].any() and np.all(trunc[:, last].sum(0) == 3)
    assert np.array_equal(np.nonzero(trunc[:, last].all(1))[0], [0, 8, 16])
    oob = phase < 0
    assert np.all(tw["flags"][0, oob] & F_OOB) and not trunc[0, oob].any() and ro["dones"][0].cpu().numpy()[oob].all()
    assert np.array_equal(rew[0, oob], tw["rew"][0, oob])
    # teeth: bootstrapping the out-of-bounds-at-the-limit envs too breaks the bit-exact check on each of them
    wrong_mask = trunc.copy()
    wrong_mask[0, oob] = True
    assert np.all(rew[0, oob] != _wrong(tw, wrong_mask, tw["val"])[0, oob])


def test_lanes_bit_identical():
    """1, 2 and 3 lanes give the same rollout; blocks of 500 envs share a phase, so the seams (1001, 1501, 2001) sit inside
    runs of envs that truncate on the same steps."""
    _, wd = _weights("sb3_init")
    n, k, L = 3001, 17, 8
    phase = (np.arange(n) // 500) % L
    ros = []
    for lanes in (1, 2, 3):
        e = _mk(n, L, 41, split_step=True, lanes=lanes)
        e.reset()
        _place(e, n, L, phase)
        ros.append(e.collect_rollout(k, wd, bootstrap_truncated=True))
    twin = _mk(n, L, 41, split_step=True, lanes=2)
    twin.reset()
    _place(twin, n, L, phase)
    _, trunc = _check(ros[1], _twin(twin, wd, k, 3))
    for seam in (1001, 1501, 2001):
        assert trunc[:, seam - 1:seam + 2].all(1).any()                 # a step where both sides of the seam truncate
    for ro in ros[1:]:
        for key in ros[0]:
            assert torch.equal(ros[0][key], ro[key]), key


def test_full_mask_at_scale():
    """2^20 envs, L = 16, k = 32, two lanes, from reset(): every env truncates at steps 15 and 31.  8192 random envs plus
    both ends and the lane seam are checked against the twin."""
    _, wd = _weights("sb3_init")
    n, k = 1 << 20, 32
    a, b = _mk(n, 16, 51, lanes=2), _mk(n, 16, 51, lanes=2)
    a.reset(); b.reset()
    a.reset_stats()
    ro = a.collect_rollout(k, wd, bootstrap_truncated=True)
    assert a.stats_dict()["truncated"] == 2 * n
    seam = a._lane_ranges[1][0]
    rng = np.random.default_rng(0)
    cols = np.unique(np.concatenate([rng.choice(n, 8192, replace=False), [0, 1, 2, n - 3, n - 2, n - 1],
                                     np.arange(seam - 3, seam + 3)]))
    cols_d = torch.from_numpy(cols).to(DEV)
    _, trunc = _check(ro, _twin(b, wd, k, 3, cols=cols_d), cols=cols_d)
    assert np.array_equal(np.nonzero(trunc.any(1))[0], [15, 31]) and trunc[[15, 31]].all()


@pytest.mark.parametrize("limit", ["default", "off"])
def test_no_truncation_is_a_noop(limit):
    """No truncation in the rollout (the default 1500-step limit from reset(), or no TimeLimit at all): True gives the same
    dict as False, bit for bit."""
    _, wd = _weights("golden")
    kw = dict(time_limit=False) if limit == "off" else {}
    a, b = _mk(4096, seed=61, **kw), _mk(4096, seed=61, **kw)
    a.reset(); b.reset()
    r0 = a.collect_rollout(16, wd)
    r1 = b.collect_rollout(16, wd, bootstrap_truncated=True)
    assert set(r0) == set(r1)
    for key in r0:
        assert torch.equal(r0[key], r1[key]), key
    assert torch.equal(a.state, b.state)


def test_one_episode_batches_are_refused():
    _, wd = _weights("golden")
    e = _mk(256, auto_reset=False)
    e.reset()
    with pytest.raises(ValueError, match="auto_reset"):
        e.collect_rollout(4, wd, bootstrap_truncated=True)
    e.collect_rollout(4, wd)                # the default still collects


def test_record_and_bootstrap_kernels_directly():
    """r6_trunc_record fills the first free slot of each truncating env of its range and never a slot past `slots - 1`;
    r6_trunc_bootstrap adds fl32(fl32(gamma) V) where a slot holds a step in [0, T) and nothing elsewhere."""
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    n, first, count, slots = 300, 10, 250, 2
    g = torch.Generator(device=DEV).manual_seed(0)
    flags = torch.full((n,), F_TRUNC, dtype=torch.uint8, device=DEV)
    flags[::5] = F_OOB                                          # done but not truncated
    tobs = torch.randn(14, n, generator=g, device=DEV)
    slot_step = torch.full((slots + 1, n), -1, dtype=torch.int32, device=DEV)      # one guard layer after the slots
    slot_obs = torch.full((slots + 1, 13, n), 7.0, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    for step in range(3):                                       # the third truncation finds no free slot
        _lib.check(L.r6_trunc_record(flags.data_ptr(), tobs.data_ptr(), n, first, count, step, slots, slot_step.data_ptr(),
                                     slot_obs.data_ptr(), s), L)
    inr = torch.zeros(n, dtype=torch.bool, device=DEV)
    inr[first:first + count] = True
    hit = inr & (flags == F_TRUNC)
    for sl in range(slots):
        assert torch.equal(slot_step[sl], torch.where(hit, sl, -1).to(torch.int32))
        assert torch.equal(slot_obs[sl][:, hit], tobs[:13, hit]) and bool((slot_obs[sl][:, ~hit] == 7.0).all())
    assert bool((slot_step[slots] == -1).all()) and bool((slot_obs[slots] == 7.0).all())
    T, j = 2, first + 1                                         # slot 0 holds step 0, slot 1 step 1; move one past T
    assert bool(hit[j])
    slot_step[1, j] = 5
    rew = torch.randn(T, n, generator=g, device=DEV)
    vals = torch.randn(slots, n, generator=g, device=DEV)
    out = rew.clone()
    _lib.check(L.r6_trunc_bootstrap(out.data_ptr(), T, n, slots, slot_step.data_ptr(), vals.data_ptr(), G, s), L)
    st, r, v = slot_step[:slots].cpu().numpy(), rew.cpu().numpy(), vals.cpu().numpy()
    mask = np.zeros((T, n), bool)
    tv = np.zeros((T, n), np.float32)
    for sl in range(slots):
        ok = (st[sl] >= 0) & (st[sl] < T)
        mask[st[sl, ok], np.nonzero(ok)[0]] = True
        tv[st[sl, ok], np.nonzero(ok)[0]] = v[sl, ok]
    assert not mask[1, j] and mask.sum() == 2 * int(hit.sum()) - 1
    assert np.array_equal(out.cpu().numpy(), tr.bootstrap_timeouts(r, mask, tv, G))


def test_trainer_trains_on_bootstrapped_rewards():
    """PPOTrainer.learn collects with bootstrap_truncated=True: the rollout handed to train() equals a twin collection
    with the bootstrap, bit for bit, on a batch that truncates (L = 5); a batch without auto-reset is refused."""
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    n, k = 2048, 16
    p0 = ActorCriticParams.sb3_init(7, DEV)
    params = ActorCriticParams(p0.flat.clone())
    env = _mk(n, 5, 71)
    trainer = PPOTrainer(env, params, PPOConfig(n_steps=k, n_epochs=1), seed=7)
    seen = []
    real_train = trainer.train
    trainer.train = lambda ro: (seen.append({key: v.clone() for key, v in ro.items()}), real_train(ro))[1]
    logs = trainer.learn(k * n)
    assert len(seen) == 1 and logs[0]["rollout/truncated"] > 0
    twin = _mk(n, 5, 71)
    twin.reset()
    want = twin.collect_rollout(k, p0.mlp(), gamma=G, gae_lambda=LAM, tensor_cores=3, bootstrap_truncated=True)
    plain = _mk(n, 5, 71)
    plain.reset()
    unboot = plain.collect_rollout(k, p0.mlp(), gamma=G, gae_lambda=LAM, tensor_cores=3)
    for key in want:
        assert torch.equal(seen[0][key], want[key]), key
    assert not torch.equal(seen[0]["rewards"], unboot["rewards"])
    frozen = _mk(256, 5, 71, auto_reset=False)
    with pytest.raises(ValueError, match="auto_reset"):
        PPOTrainer(frozen, ActorCriticParams(p0.flat.clone()), PPOConfig(n_steps=4, n_epochs=1), seed=7).learn(4 * 256)
