"""EvalCallback during PPOTrainer.learn on the GPU, for the shared trunk, the separate towers and both with gSDE.

1. Evaluation k is the Monte-Carlo driver: the returns and lengths of every evaluation equal, bit for bit,
   montecarlo.run_montecarlo on the parameters snapshotted at that evaluation, over the initial conditions drawn with
   episode id k (tests/philox_ref.py), with the same batch configuration (two-kernel loop, stream lanes) and, with
   VecNormalize, a frozen copy of the training statistics of that moment.
2. Evaluation leaves training untouched: learn with the callback gives the parameters, Adam state, VecNormalize
   statistics and train/ / rollout/ logs of learn without it, bit for bit.
3. best_model.npz is the snapshot of the highest eval/mean_reward; it loads with policy.load_npz and the Monte-Carlo
   CLI runs on it (with its VecNormalize statistics).
4. Two spawned gloo ranks on cuda:0 give the same eval/ logs and decisions, equal to one process evaluating the union;
   only the first rank writes files.  With two GPUs the same under NCCL.
5. `python -m rl_rocket_6dof_b200.train` runs end to end and the Monte-Carlo CLI runs on its best model."""
import datetime
import os
import sys
import time

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import philox_ref as pr  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEP = [dict(pi=[64, 64], vf=[64, 64])]
LAYOUTS = {"shared": {}, "sep": dict(net_arch=SEP), "sde": dict(use_sde=True), "sepsde": dict(use_sde=True, net_arch=SEP)}
N_TRAIN, N_EVAL, T, ITERS, EVAL_SEED, LANES = 512, 256, 8, 3, 77, 2


def _ic(ep, seed, genv, episode):
    return pr.normalize_ic_quaternion(pr.sample_ic(ep.ic_low, ep.ic_high, seed, genv, episode))


def _weights(flat):
    from rl_rocket_6dof_b200.ppo import ActorCriticParams
    return {k: v.cpu().numpy() for k, v in ActorCriticParams(flat).mlp().items()}


def _setup(kind, vecnorm, seed=5):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    env = Rocket6DOFBatch(N_TRAIN, device=DEV, seed=21)
    params = ActorCriticParams.sb3_init(seed=seed, device=DEV, **LAYOUTS[kind])
    vn = VecNormalize(env) if vecnorm else None
    cfg = PPOConfig(n_steps=T, n_epochs=2, use_sde=params.use_sde)
    return PPOTrainer(env, params, cfg, seed=9, vec_normalize=vn)


def _snapshotting(cb):
    """Wraps cb.on_rollout_end / cb.run: every evaluation's parameters, VecNormalize copy and gathered episodes."""
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    snaps = []
    run, on_end = cb.run, cb.on_rollout_end

    def wrapped_run(trainer):
        flat = trainer.params.flat.clone()
        vn = None
        if trainer.vec_normalize is not None:
            vn = VecNormalize(trainer.batch, training=False)
            vn.obs_rms.copy_(trainer.vec_normalize.obs_rms)
            before = (trainer.vec_normalize.obs_rms.clone(), trainer.vec_normalize.ret_rms.clone())
        ep = run(trainer)
        if vn is not None:          # the evaluation never updates the training statistics
            assert torch.equal(before[0], trainer.vec_normalize.obs_rms)
            assert torch.equal(before[1], trainer.vec_normalize.ret_rms)
        snaps.append(dict(flat=flat, vn=vn, ep=ep))
        return ep

    def wrapped_end(trainer):
        logs = on_end(trainer)
        if logs:
            snaps[-1]["logs"] = logs
        return logs

    cb.run, cb.on_rollout_end = wrapped_run, wrapped_end
    return snaps


def _flat_logs(logs, prefix):
    keys = sorted(k for k in logs[0] if k.startswith(prefix))
    return np.array([[float(log[k]) for k in keys] for log in logs])


@pytest.mark.parametrize("kind,vecnorm", [("shared", False), ("sep", False), ("sde", False), ("sepsde", False),
                                          ("shared", True), ("sepsde", True)])
def test_evaluations_are_the_montecarlo_driver_and_leave_training_untouched(tmp_path, kind, vecnorm):
    from rl_rocket_6dof_b200 import montecarlo, policy
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.evaluation import EvalCallback
    # ---- 2. training with and without the callback
    plain = _setup(kind, vecnorm)
    logs0 = plain.learn(ITERS * T * N_TRAIN)
    tr = _setup(kind, vecnorm)
    eb = Rocket6DOFBatch(N_EVAL, device=DEV, seed=EVAL_SEED, auto_reset=False, time_limit=True, split_step=True,
                         lanes=LANES)
    cb = EvalCallback(eb, eval_freq=T, n_eval_episodes=N_EVAL, log_path=str(tmp_path), best_model_save_path=str(tmp_path))
    snaps = _snapshotting(cb)
    logs1 = tr.learn(ITERS * T * N_TRAIN, eval_callback=cb)
    assert torch.equal(plain.params.flat, tr.params.flat)
    assert torch.equal(plain.m, tr.m) and torch.equal(plain.v, tr.v)
    for prefix in ("train/", "rollout/", "time/"):
        assert np.array_equal(_flat_logs(logs0, prefix), _flat_logs(logs1, prefix), equal_nan=True), prefix
    if vecnorm:
        assert torch.equal(plain.vec_normalize.obs_rms, tr.vec_normalize.obs_rms)
        assert torch.equal(plain.vec_normalize.ret_rms, tr.vec_normalize.ret_rms)
    assert len(snaps) == ITERS and all("eval/mean_reward" in log for log in logs1)
    assert not torch.equal(snaps[0]["flat"], snaps[-1]["flat"])
    # ---- 1. evaluation k against run_montecarlo over the initial conditions of episode k
    ep = eb.params
    ics = []
    for k, s in enumerate(snaps):
        ic = _ic(ep, EVAL_SEED, np.arange(N_EVAL), k)
        ics.append(ic)
        ref = montecarlo.run_montecarlo(N_EVAL, _weights(s["flat"]), device=DEV, seed=EVAL_SEED, ic_table=ic,
                                        tensor_cores=True, two_kernel=True, lanes=LANES, vec_normalize=s["vn"])
        assert np.array_equal(ref["episode_return"].view(np.int64), s["ep"]["episode_return"].view(np.int64)), k
        assert np.array_equal(ref["episode_length"], s["ep"]["episode_length"]), k
        assert np.array_equal(ref["flags"], s["ep"]["flags"]), k
        order = np.argsort(ref["episode_length"], kind="stable")
        r = np.array([round(x, 6) for x in ref["episode_return"].tolist()])[order]
        assert s["logs"]["eval/mean_reward"] == float(np.mean(r))
        assert s["logs"]["eval/landing_rate"] == float(np.mean(ref["landed"]))
    assert not np.array_equal(ics[0], ics[1])             # fresh initial conditions per evaluation
    # ---- 3. the best model
    means = [s["logs"]["eval/mean_reward"] for s in snaps]
    best = int(np.argmax(means))
    w = policy.load_npz(str(tmp_path / "best_model.npz"))
    for k, v in _weights(snaps[best]["flat"]).items():
        assert np.array_equal(w[k].reshape(-1), v.reshape(-1)), k
    ev = np.load(tmp_path / "evaluations.npz")
    assert ev["results"].shape == (ITERS, N_EVAL) and ev["timesteps"].tolist() == [(i + 1) * T * N_TRAIN
                                                                                  for i in range(ITERS)]
    args = ["--policy", str(tmp_path / "best_model.npz"), "--episodes", "64", "--csv", str(tmp_path / "mc.csv"),
            "--device", DEV, "--tensor-cores"]
    if vecnorm:
        args += ["--vecnormalize", str(tmp_path / "best_model_vecnormalize.npz")]
    assert montecarlo.main(args) == 0 and os.path.getsize(tmp_path / "mc.csv") > 0


# ---------------------------------------------------------------------------------------------- 4. data-parallel

N_DP, NE_DP = 256, 128


def _dp_worker(rank, world, backend, store_path, out_dir, devices):
    import torch.distributed as dist
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.evaluation import EvalCallback
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    from rl_rocket_6dof_b200.sharding import shard_batch_kwargs
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    dev = torch.device(devices[rank])
    torch.cuda.set_device(dev)
    kw = dict(device_id=dev) if backend == "nccl" else {}
    dist.init_process_group(backend, store=dist.FileStore(store_path, world), rank=rank, world_size=world,
                            timeout=datetime.timedelta(seconds=240), **kw)
    try:
        g = dist.group.WORLD
        env = Rocket6DOFBatch(N_DP, device=dev, seed=31, **shard_batch_kwargs(N_DP, rank, world))
        eb = Rocket6DOFBatch(NE_DP, device=dev, seed=EVAL_SEED, auto_reset=False, time_limit=True, split_step=True,
                             **shard_batch_kwargs(NE_DP, rank, world))
        vn = VecNormalize(env, group=g)
        tr = PPOTrainer(env, ActorCriticParams.sb3_init(seed=3, device=dev), PPOConfig(n_steps=T, n_epochs=2), seed=9,
                        group=g, vec_normalize=vn)
        d = os.path.join(out_dir, f"{backend}_files{rank}")
        cb = EvalCallback(eb, eval_freq=T, log_path=d, best_model_save_path=d, group=g)
        snaps = _snapshotting(cb)
        logs = tr.learn(ITERS * T * N_DP * world, eval_callback=cb)
        keys = sorted(k for k in logs[0] if k.startswith("eval/"))
        res = dict(logs=np.array([[log[k] for k in keys] for log in logs]), keys=np.array(keys),
                   best=np.array(cb.best_mean_reward))
        for k, s in enumerate(snaps):
            res[f"flat{k}"] = s["flat"].cpu().numpy()
            res[f"obs_rms{k}"] = s["vn"].obs_rms.cpu().numpy()
            for name, v in s["ep"].items():
                res[f"{name}{k}"] = v
        dist.barrier()
        np.savez(os.path.join(out_dir, f"{backend}_rank{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


def _spawn(backend, devices, tmp):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, backend, os.path.join(tmp, f"store_{backend}"), tmp, devices))
             for r in range(2)]
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
    assert not survivors and [p.exitcode for p in procs] == [0, 0]
    return [dict(np.load(os.path.join(tmp, f"{backend}_rank{r}.npz"))) for r in range(2)]


def _check_dp(runs, tmp, backend):
    from rl_rocket_6dof_b200 import montecarlo
    from rl_rocket_6dof_b200.evaluation import monitor_rewards, result_order, summarize
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.vec_normalize import VecNormalize
    r0, r1 = runs
    for k in r0:
        assert np.array_equal(np.asarray(r0[k]), np.asarray(r1[k])), k         # same logs and decisions everywhere
    assert os.path.exists(os.path.join(tmp, f"{backend}_files0", "best_model.npz"))
    assert os.path.exists(os.path.join(tmp, f"{backend}_files0", "best_model_vecnormalize.npz"))
    assert not os.path.exists(os.path.join(tmp, f"{backend}_files1"))
    keys = list(r0["keys"])
    ep = Rocket6DOFBatch(8, device=DEV).params
    for k in range(ITERS):
        # one process evaluating the union of the shards with the same parameters and statistics
        from rl_rocket_6dof_b200.ppo import ActorCriticParams
        flat = torch.from_numpy(r0[f"flat{k}"]).to(DEV)
        w = {n: v.cpu().numpy() for n, v in ActorCriticParams(flat).mlp().items()}
        vn = VecNormalize(Rocket6DOFBatch(8, device=DEV), training=False)
        vn.obs_rms.copy_(torch.from_numpy(r0[f"obs_rms{k}"]))
        ref = montecarlo.run_montecarlo(2 * NE_DP, w, device=DEV, seed=EVAL_SEED, ic_table=_ic(ep, EVAL_SEED,
                                        np.arange(2 * NE_DP), k), tensor_cores=True, two_kernel=True, vec_normalize=vn)
        assert np.array_equal(ref["episode_return"].view(np.int64), r0[f"episode_return{k}"].view(np.int64)), k
        assert np.array_equal(ref["episode_length"], r0[f"episode_length{k}"]), k
        order = result_order(ref["episode_length"])
        want = summarize(monitor_rewards(ref["episode_return"])[order], ref["episode_length"][order], ref["landed"])
        for name, v in want.items():
            assert r0["logs"][k, keys.index(name)] == v, (k, name)


@pytest.mark.timeout(1800)
def test_gloo_ranks_evaluate_as_one_process(tmp_path):
    runs = _spawn("gloo", ["cuda:0", "cuda:0"], str(tmp_path))
    _check_dp(runs, str(tmp_path), "gloo")


@pytest.mark.timeout(1800)
def test_nccl_ranks_evaluate_as_one_process(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    runs = _spawn("nccl", ["cuda:0", "cuda:1"], str(tmp_path))
    _check_dp(runs, str(tmp_path), "nccl")


# ---------------------------------------------------------------------------------------------------- 5. the CLI

@pytest.mark.timeout(1800)
@pytest.mark.parametrize("extra", [[], ["--net-arch", "separate", "--use-sde", "--vecnormalize", "--lanes", "2"]])
def test_train_cli_end_to_end(tmp_path, extra):
    from rl_rocket_6dof_b200 import montecarlo, train
    out = tmp_path / "run"
    n = 4096
    assert train.main(["--out", str(out), "--envs", str(n), "--total-timesteps", str(3 * 32 * n), "--eval-freq", "64",
                       "--n-eval-episodes", "256", "--device", DEV] + extra) == 0
    files = {"best_model.npz", "final_model.npz", "evaluations.npz", "progress.csv"}
    if "--vecnormalize" in extra:
        files |= {"best_model_vecnormalize.npz", "vecnormalize.npz"}
    assert files <= set(os.listdir(out))
    ev = np.load(out / "evaluations.npz")
    assert ev["timesteps"].tolist() == [2 * 32 * n] and ev["results"].shape == (1, 256)   # vec-env step 64 of 96
    rows = open(out / "progress.csv").read().splitlines()
    assert len(rows) == 4 and "eval/mean_reward" in rows[0]
    args = ["--policy", str(out / "best_model.npz"), "--episodes", "128", "--csv", str(tmp_path / "mc.csv"),
            "--device", DEV]
    if "--vecnormalize" in extra:
        args += ["--vecnormalize", str(out / "best_model_vecnormalize.npz")]
    assert montecarlo.main(args) == 0
