"""rl_rocket_6dof_b200.evaluation's host logic against tests/evalcb_ref.py (SB3 1.6's evaluate_policy and
EvalCallback._on_step restated): the evaluation schedule, the result order, mean / std, the best-model decisions and
evaluations.npz, on synthetic episodes; the construction errors, and the data-parallel consistency row on two gloo
ranks (the same message on every rank).  No GPU: the episodes come from a stub in place of the device loop."""
import datetime
import math
import os
import sys
import types

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import evalcb_ref as ref  # noqa: E402


def _batch(n=8, offset=0, n_global=None, auto_reset=False, time_limit=True, seed=7):
    return types.SimpleNamespace(num_envs=n, env_offset=offset, num_envs_global=n if n_global is None else n_global,
                                 seed_value=seed, auto_reset=auto_reset, time_limit=time_limit, device="cpu")


class _Params:
    def __init__(self):
        self.version = 0

    def save_npz(self, path):
        np.savez(path, version=self.version)


def _trainer(n_steps):
    return types.SimpleNamespace(group=None, cfg=types.SimpleNamespace(n_steps=n_steps, tensor_cores=3),
                                 params=_Params(), vec_normalize=None, num_timesteps=0)


def _episodes(rng, n, max_len=40):
    """One (return, length) per env with many ties in length and returns of all magnitudes."""
    lengths = rng.integers(1, max_len, n)
    returns = rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, n)
    return returns, lengths


# ------------------------------------------------------------------------------------------------------ schedule

@pytest.mark.parametrize("n_steps", [4, 8])
@pytest.mark.parametrize("eval_freq", [1, 3, 4, 5, 8, 12, 16, 20, 33])
def test_schedule_matches_sb3(n_steps, eval_freq):
    """An iteration evaluates when SB3 would evaluate at least once during its n_steps calls; when eval_freq is a
    multiple of n_steps the evaluations are SB3's one for one, at SB3's timesteps."""
    from rl_rocket_6dof_b200.evaluation import evaluation_due
    iters, n_envs = 30, 5
    cb = ref.EvalCallbackRef(eval_freq)
    sb3_iters, sb3_timesteps = [], []
    for i in range(iters):
        for j in range(n_steps):
            ts = (i * n_steps + j + 1) * n_envs
            if cb.on_step(ts, lambda: ([0.0], [1])) is not None:
                sb3_iters.append(i)
                sb3_timesteps.append(ts)
    mine = [i for i in range(iters) if evaluation_due((i + 1) * n_steps, n_steps, eval_freq)]
    assert mine == sorted(set(sb3_iters))
    if eval_freq % n_steps == 0:
        assert mine == sb3_iters
        assert [(i + 1) * n_steps * n_envs for i in mine] == sb3_timesteps
    if eval_freq < n_steps:
        assert mine == list(range(iters))           # several SB3 evaluations in one collection: one here


# ---------------------------------------------------------------------------------------- order, statistics

@pytest.mark.parametrize("seed", range(6))
def test_result_order_and_statistics_match_evaluate_policy(seed):
    from rl_rocket_6dof_b200.evaluation import monitor_rewards, result_order, summarize
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 200))
    returns, lengths = _episodes(rng, n)
    # the SB3 eval env auto-resets: later episodes of an env must not be counted
    eps = [[(returns[i], lengths[i]), (rng.standard_normal(), int(rng.integers(1, 5)))] for i in range(n)]
    want_r, want_l = ref.evaluate_policy(eps, n)
    rewards = monitor_rewards(returns)
    order = result_order(lengths)
    assert rewards[order].tolist() == want_r and lengths[order].tolist() == want_l
    logs = summarize(rewards[order], lengths[order], np.zeros(n, bool))
    assert logs["eval/mean_reward"] == float(np.mean(want_r)) and logs["eval/std_reward"] == float(np.std(want_r))
    assert logs["eval/mean_ep_length"] == float(np.mean(want_l))
    assert logs["eval/std_ep_length"] == float(np.std(want_l))
    assert logs["eval/landing_rate"] == 0.0


def test_monitor_rounding_is_pythons_round():
    from rl_rocket_6dof_b200.evaluation import monitor_rewards
    x = np.array([0.0000005, 2.6749995, -1.0000015, 123.4567895, 1e-7, -3.5e-7, 1e12 + 0.3])
    assert monitor_rewards(x).tolist() == [round(float(v), 6) for v in x]
    # the two roundings part ways somewhere on a fine grid: the module must follow Python's
    grid = np.arange(1, 200001) * 1e-7 + 0.1234565
    assert monitor_rewards(grid).tolist() == [round(float(v), 6) for v in grid]


# -------------------------------------------------------------------------------- callback: best model, npz

def _same(a, b):
    return a == b or (math.isnan(a) and math.isnan(b))


def _drive(tmp_path, eval_freq, n_steps, means, n=6, seed=0):
    """Runs the callback and the reference over len(means) collections whose evaluation k has mean reward means[k]
    (an evaluation per collection: eval_freq == n_steps, or one every few); returns both and the saved versions."""
    from rl_rocket_6dof_b200.evaluation import EvalCallback
    rng = np.random.default_rng(seed)
    cb = EvalCallback(_batch(n), eval_freq=eval_freq, log_path=str(tmp_path), best_model_save_path=str(tmp_path))
    tr = _trainer(n_steps)
    rcb = ref.EvalCallbackRef(eval_freq)
    k = [0]
    plays = []

    def play():
        m = means[min(k[0], len(means) - 1)]
        lengths = _episodes(rng, n)[1]
        returns = np.full(n, m)          # equal returns: equal means are ties, whatever the rounding of the mean
        plays.append((returns.copy(), lengths.copy()))
        k[0] += 1
        return plays[-1]

    saved, logs_all = [], []
    for i in range(len(means) * eval_freq // n_steps):
        tr.params.version = i
        tr.num_timesteps = (i + 1) * n_steps * n
        before = len(plays)
        cb.run = lambda trainer: (lambda r, l: {"episode_return": r, "episode_length": l,
                                                "flags": np.where(l % 2 == 0, 0xF8, 0).astype(np.uint8)})(*play())
        logs = cb.on_rollout_end(tr)
        for j in range(n_steps):
            def sb3_eval():
                r, l = plays[before]
                return ref.evaluate_policy([[(r[e], l[e])] for e in range(n)], n)
            rl = rcb.on_step((i * n_steps + j + 1) * n, sb3_eval)
            if rl is not None:
                for key in ("mean_reward", "std_reward", "mean_ep_length", "std_ep_length"):
                    assert _same(logs["eval/" + key], rl[key]), key
                assert _same(logs["eval/best_mean_reward"], rcb.best_mean_reward)
                r, l = plays[before]
                assert logs["eval/landing_rate"] == float(np.mean(l % 2 == 0))
        if logs:
            logs_all.append(logs)
            p = tmp_path / "best_model.npz"
            saved.append(int(np.load(p)["version"]) if p.exists() else None)
    return cb, rcb, saved, logs_all


@pytest.mark.parametrize("means", [[1.0, 2.0, 2.0, 0.5, 3.0], [-5.0, -5.0, -4.0, float("nan"), -3.0],
                                   [float("nan"), float("nan"), 1.0], [0.0, -0.0, 1e-12]])
def test_best_model_and_npz_match_eval_callback(tmp_path, means):
    n_steps = 4
    cb, rcb, saved, logs = _drive(tmp_path, n_steps, n_steps, means)
    # best_model.npz holds the parameters of the last strict improvement so far (NaN never improves, ties do not)
    best, last_saved, want = -math.inf, None, []
    for i, lg in enumerate(logs):
        if lg["eval/mean_reward"] > best:
            best, last_saved = lg["eval/mean_reward"], i
        want.append(last_saved)
    assert saved == want
    assert [c // n_steps - 1 for c in rcb.saved] == sorted(set(x for x in want if x is not None))
    got, exp = np.load(tmp_path / "evaluations.npz"), rcb.npz()
    assert sorted(got.files) == ["ep_lengths", "results", "timesteps"]
    assert got["results"].dtype == np.float64 and got["ep_lengths"].dtype == np.int64
    assert np.array_equal(got["timesteps"], exp["timesteps"])
    assert np.array_equal(got["results"], exp["results"], equal_nan=True)
    assert np.array_equal(got["ep_lengths"], exp["ep_lengths"])
    assert cb.best_mean_reward == rcb.best_mean_reward or (math.isinf(cb.best_mean_reward) and
                                                           math.isinf(rcb.best_mean_reward))


def test_sparse_evaluations_npz(tmp_path):
    """eval_freq = 3 n_steps: one evaluation every third collection, the npz rewritten with every row so far."""
    cb, rcb, saved, logs = _drive(tmp_path, 12, 4, [1.0, 0.0, 4.0])
    assert len(logs) == 3
    got = np.load(tmp_path / "evaluations.npz")
    assert got["timesteps"].tolist() == rcb.npz()["timesteps"].tolist() == [12 * 6, 24 * 6, 36 * 6]
    assert got["results"].shape == (3, 6) and got["ep_lengths"].shape == (3, 6)


def test_no_files_without_paths(tmp_path):
    from rl_rocket_6dof_b200.evaluation import EvalCallback
    cb = EvalCallback(_batch(4), eval_freq=2)
    tr = _trainer(2)
    cb.run = lambda trainer: {"episode_return": np.ones(4), "episode_length": np.full(4, 3, np.int64),
                              "flags": np.zeros(4, np.uint8)}
    logs = cb.on_rollout_end(tr)
    assert logs["eval/mean_reward"] == 1.0 and logs["eval/best_mean_reward"] == 1.0
    assert cb.evaluations.timesteps == [0] and os.listdir(tmp_path) == []


# ---------------------------------------------------------------------------------------- construction errors

def test_construction_errors():
    from rl_rocket_6dof_b200.evaluation import EvalCallback
    with pytest.raises(ValueError, match="auto_reset"):
        EvalCallback(_batch(auto_reset=True), eval_freq=4)
    with pytest.raises(ValueError, match="time_limit"):
        EvalCallback(_batch(time_limit=False), eval_freq=4)
    with pytest.raises(ValueError, match="deterministic"):
        EvalCallback(_batch(), eval_freq=4, deterministic=False)
    with pytest.raises(ValueError, match="n_eval_episodes"):
        EvalCallback(_batch(8), eval_freq=4, n_eval_episodes=15)
    with pytest.raises(ValueError, match="eval_freq"):
        EvalCallback(_batch(), eval_freq=0)
    assert EvalCallback(_batch(8), eval_freq=4, n_eval_episodes=8).n_eval_episodes == 8
    assert EvalCallback(_batch(4, 4, 8), eval_freq=4).n_eval_episodes == 8      # the global count


def test_group_errors_are_a_function_of_the_rows():
    from rl_rocket_6dof_b200.evaluation import GROUP_FIELDS, group_errors
    def row(**kw):
        v = dict(num_envs=4, env_offset=0, num_envs_global=8, seed_hi=0, seed_lo=7, eval_freq=4, tensor_cores=-1,
                 local_error=0)
        v.update(kw)
        return [float(v[k]) for k in GROUP_FIELDS]
    assert group_errors(np.array([row(), row(env_offset=4)]), 2) == []
    errs = group_errors(np.array([row(), row(env_offset=0, eval_freq=8, local_error=4)]), 2)
    assert any("n_eval_episodes" in e for e in errs) and any("eval_freq" in e for e in errs)
    assert any("env_offset" in e for e in errs)
    assert group_errors(np.array([row(num_envs_global=6), row(env_offset=4, num_envs_global=6)]), 2)


# ---------------------------------------------------------------------------------------- data-parallel (gloo)

def _gloo_worker(rank, world, store_path, out_path):
    import torch.distributed as dist
    from rl_rocket_6dof_b200.evaluation import EvalCallback
    store = dist.FileStore(store_path, world)
    dist.init_process_group("gloo", store=store, rank=rank, world_size=world, timeout=datetime.timedelta(seconds=120))
    try:
        msgs = []
        good = _batch(4, 4 * rank, 8)
        cb = EvalCallback(good, eval_freq=4, group=dist.group.WORLD)
        msgs.append(f"ok {cb.world} {cb.rank} {cb.writer}")
        cases = [_batch(4, 0, 8),                                              # rank 1 claims rank 0's shard
                 _batch(4, 4 * rank, 8, auto_reset=rank == 1),                 # one rank's batch auto-resets
                 _batch(4, 4 * rank, 8, seed=7 + rank)]                        # different eval seeds
        for b in cases:
            try:
                EvalCallback(b, eval_freq=4, group=dist.group.WORLD)
                msgs.append("")
            except ValueError as e:
                msgs.append(str(e))
        try:
            EvalCallback(good, eval_freq=4 + rank, group=dist.group.WORLD)
            msgs.append("")
        except ValueError as e:
            msgs.append(str(e))
        dist.barrier()
        np.save(out_path, np.array(msgs))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_inconsistent_eval_shards_raise_the_same_error_on_every_rank(tmp_path):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    outs = [str(tmp_path / f"rank{r}.npy") for r in range(2)]
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, str(tmp_path / "store"), outs[r])) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=300)
    alive = [p for p in procs if p.is_alive()]
    for p in alive:
        p.terminate()
        p.join(timeout=30)
    assert not alive and [p.exitcode for p in procs] == [0, 0]
    r0, r1 = (np.load(o).tolist() for o in outs)
    assert r0[0] == "ok 2 0 True" and r1[0] == "ok 2 1 False"
    for a, b, word in zip(r0[1:], r1[1:], ["env_offset", "auto_reset", "seed", "eval_freq"]):
        assert a == b and word in a, (a, b)
