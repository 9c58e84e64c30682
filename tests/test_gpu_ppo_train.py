"""PPOTrainer.train / learn on the GPU against tests/ppo_train_ref.py, the float64 restatement of SB3 1.6's PPO.train:
every Adam step from the kernels' own pre-step state within the per-step bound, the minibatch split, the train/ logs,
the target_kl stop and the learning-rate schedule of learn."""
import dataclasses

import numpy as np
import pytest
import torch

import policy_ref as pr
import ppo_ref as rf
import ppo_train_ref as tr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N_ENVS, T = 2048, 16              # 32,768 samples: batch_size 10,000 gives three full minibatches and one of 2,768
BS = 10000


def _collect(family, seed):
    """A real collect_rollout (strided obs view) right after reset with the weights of `family`: no env reaches the
    1500-step TimeLimit, so the rollout needs none of the critic bootstrapping of truncations SB3 would add.  Returns
    (env, params, device rollout, host rollout of flat [T N, ...] arrays)."""
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams
    env = Rocket6DOFBatch(N_ENVS, device=DEV, seed=seed)
    params = ActorCriticParams.from_weights(pr.weights(family), DEV)
    env.reset()
    env.reset_stats()
    ro = env.collect_rollout(T, params.mlp())
    assert ro["obs"].stride(2) != 1                               # the in-place trajectory's strided view
    assert env.stats_dict()["truncated"] == 0
    host = {k: ro[k].contiguous().cpu().numpy().reshape(T * N_ENVS, -1) for k in ("obs", "actions")}
    host.update({k: ro[k].cpu().numpy().reshape(-1) for k in ("log_probs", "advantages", "returns", "values")})
    return env, params, ro, host


def _capture(mp):
    """Wraps ppo.loss_and_grad and ppo.adam_step (PPOTrainer.train resolves both through the module): records each
    call's inputs, and the parameters after each Adam step.  Returns the list of minibatches, in call order."""
    from rl_rocket_6dof_b200 import ppo
    mbs = []
    real_lg, real_adam = ppo.loss_and_grad, ppo.adam_step

    def loss_and_grad(params, rollout, idx, **kw):
        mbs.append(dict(idx=idx.clone(), params=params.flat.clone(),
                        kw={k: v for k, v in kw.items() if k not in ("grad_sum", "terms", "work")}))
        return real_lg(params, rollout, idx, **kw)

    def adam_step(params, grad_sum, m, v, **kw):
        rec = dict(params=params.clone(), m=m.clone(), v=v.clone(), grad=grad_sum.clone(), **kw)
        real_adam(params, grad_sum, m, v, **kw)
        rec["post"] = params.clone()
        mbs[-1]["adam"] = rec

    mp.setattr(ppo, "loss_and_grad", loss_and_grad)
    mp.setattr(ppo, "adam_step", adam_step)
    return mbs


def _host(mbs):
    cpu = lambda d: {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}
    return [dict(cpu(e), adam=cpu(e["adam"])) if "adam" in e else cpu(e) for e in mbs]


def _train(family, seed, **cfg_kw):
    """One PPOTrainer.train over a fresh rollout with every step captured; returns a dict of host arrays."""
    from rl_rocket_6dof_b200.ppo import PPOConfig, PPOTrainer
    env, params, ro, host = _collect(family, seed)
    cfg = PPOConfig(n_steps=T, **cfg_kw)
    trainer = PPOTrainer(env, params, cfg, seed=seed)
    with pytest.MonkeyPatch.context() as mp:
        mbs = _capture(mp)
        log = trainer.train(ro)
    return dict(cfg=cfg, host=host, mbs=_host(mbs), log=log, log_std=params.log_std.cpu().numpy(),
                adam_steps=trainer.adam_steps, final=params.flat.cpu().numpy())


# (family, seed, PPOConfig changes): (a) the defaults, (b) an entropy bonus on raw advantages, (c) the gradient clip
# off (1e6) and on (0.5)
CASES = {"defaults": ("sb3_init", 1, dict(batch_size=BS, n_epochs=2)),
         "ent_raw_adv": ("golden", 2, dict(batch_size=BS, n_epochs=2, ent_coef=0.01, normalize_advantage=False)),
         "clip_off": ("saturating", 3, dict(batch_size=BS, n_epochs=2, max_grad_norm=1e6)),
         "clip_on": ("saturating", 3, dict(batch_size=BS, n_epochs=2, max_grad_norm=0.5))}
_RUNS = {}


def _run(case):
    """The captured training of CASES[case] and the reference of each of its minibatches (cached: the reference costs
    about a second of CPU per minibatch)."""
    if case not in _RUNS:
        family, seed, kw = CASES[case]
        run = _train(family, seed, **kw)
        run["refs"] = [_reference(run, e) for e in run["mbs"]]
        _RUNS[case] = run
    return _RUNS[case]


def _reference(run, e, **kw):
    a = e.get("adam")
    if a is None:
        return tr.reference_step(e["params"], None, None, None, run["host"], e["idx"], None, run["cfg"])
    return tr.reference_step(a["params"], a["m"], a["v"], a["step"], run["host"], e["idx"], a["lr"],
                             kw.pop("cfg", run["cfg"]), **kw)


def _epochs(run, mbs):
    total = T * N_ENVS
    nmb = -(-total // run["cfg"].batch_size)
    return [mbs[i:i + nmb] for i in range(0, len(mbs), nmb)]


@pytest.mark.parametrize("case", list(CASES))
def test_train_steps_match_sb3(case):
    run = _run(case)
    cfg, mbs, total = run["cfg"], run["mbs"], T * N_ENVS
    epochs = _epochs(run, mbs)
    assert len(epochs) == cfg.n_epochs
    rem = total - (total // BS) * BS
    for ep in epochs:                       # each epoch: a permutation of the rollout in minibatches bs, ..., bs, rem
        assert [len(e["idx"]) for e in ep] == [BS] * (total // BS) + [rem]
        assert np.array_equal(np.sort(np.concatenate([e["idx"] for e in ep])), np.arange(total))
    worst, prev = 0.0, None
    for k, (e, ref) in enumerate(zip(mbs, run["refs"])):
        a = e["adam"]
        assert e["kw"] == dict(clip_range=cfg.clip_range, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef,
                               normalize_advantage=cfg.normalize_advantage)
        assert a["step"] == k + 1 and a["scale"] == 1.0 / len(e["idx"]), (k, a["step"], a["scale"])
        assert a["lr"] == cfg.learning_rate and a["max_grad_norm"] == cfg.max_grad_norm
        assert np.array_equal(a["params"], e["params"]) and (prev is None or np.array_equal(prev, e["params"]))
        prev = a["post"]
        r = np.abs(a["post"].astype(np.float64) - ref["p"]) / ref["bound"]
        print(f"{case} step {k + 1}: B {len(e['idx'])} pre-clip norm {ref['norm']:.4g} clip {ref['clip']:.4g} "
              f"max |kernel - ref| / bound {r.max():.3g}")
        assert np.all(r <= rf.C_BAR), (case, k, float(r.max()), int(r.argmax()))
        worst = max(worst, float(r.max()))
    assert np.array_equal(prev, run["final"])
    print(f"{case}: worst |kernel - ref| / bound over {len(mbs)} steps {worst:.3g}")
    clipped = [ref["clip"] < 1 for ref in run["refs"]]
    assert any(clipped) == (case in ("clip_on", "ent_raw_adv")), clipped        # which regime ran


def _check_logs(got, want, bounds, label):
    assert set(got) == set(want), set(got) ^ set(want)
    for key in ("train/n_updates", "train/learning_rate", "train/clip_range"):
        assert got[key] == want[key], (key, got[key], want[key])
    for key in ("train/explained_variance", "train/std"):
        assert abs(got[key] - want[key]) <= 1e-9 * abs(want[key]), (key, got[key], want[key])
    bad = {}
    for key, b in bounds.items():
        r = abs(got[key] - want[key]) / b
        print(f"{label} {key}: trainer {got[key]:.10g} reference {want[key]:.10g} |diff| / bound {r:.3g}")
        if not r <= rf.C_BAR:
            bad[key] = (got[key], want[key], r)
    assert not bad, bad


def test_train_logs_match_sb3():
    """Every train/ value against sb3_logs: approx_kl over the last epoch only, entropy_loss and loss from each
    minibatch's pre-step log_std (n_epochs = 2 so that both differ from an all-epoch / final-log_std statement)."""
    run = _run("defaults")
    cfg = run["cfg"]
    per_epoch = _epochs(run, run["refs"])
    want = tr.sb3_logs([[r["logs"] for r in ep] for ep in per_epoch], run["log_std"], run["host"]["values"],
                       run["host"]["returns"], cfg.n_epochs, cfg.learning_rate, cfg.clip_range)
    bounds = tr.sb3_log_bounds([[r["log_bounds"] for r in ep] for ep in per_epoch])
    _check_logs(run["log"], want, bounds, "defaults")


def test_target_kl_stops_where_sb3_stops():
    """target_kl set so that the reference stops in the middle of epoch 2 of 3: the trainer stops at the same minibatch,
    takes no Adam step for it, logs its terms, averages approx_kl over the partial last epoch, and still counts
    n_epochs updates."""
    family, seed, kw = "sb3_init", 4, dict(batch_size=BS, n_epochs=3, learning_rate=1e-3)
    run1 = _train(family, seed, **kw)
    nmb = -(-T * N_ENVS // BS)
    refs = [_reference(run1, e) for e in run1["mbs"][:2 * nmb]]
    kl = np.array([r["logs"]["approx_kl"] for r in refs])
    kb = rf.C_BAR * np.array([r["log_bounds"]["approx_kl"] for r in refs])
    # the deciding minibatch: inside epoch 2, not its first, with the largest lead over every earlier KL
    lead = {d: kl[d] - kl[:d].max() for d in range(nmb + 1, 2 * nmb)}
    d = max(lead, key=lead.get)
    thr = 0.5 * (kl[d] + kl[:d].max())
    print("reference approx_kl per minibatch", kl, "deciding", d, "1.5 target_kl", thr)
    assert lead[d] > 0 and np.all(np.abs(kl[:d + 1] - thr) > kb[:d + 1])    # no decision within the bound of its KL
    run2 = _train(family, seed, target_kl=thr / 1.5, **kw)
    mbs = run2["mbs"]
    assert len(mbs) == d + 1                                         # stopped at d, no epoch 3
    for e1, e2 in zip(run1["mbs"], mbs):
        assert np.array_equal(e1["idx"], e2["idx"]) and np.array_equal(e1["params"], e2["params"])
    assert all("adam" in e for e in mbs[:d]) and "adam" not in mbs[d] and run2["adam_steps"] == d
    assert np.array_equal(run2["final"], run1["mbs"][d]["params"])   # the breaking minibatch took no step
    per_epoch = [refs[:nmb], refs[nmb:d + 1]]
    want = tr.sb3_logs([[r["logs"] for r in ep] for ep in per_epoch], run2["log_std"], run2["host"]["values"],
                       run2["host"]["returns"], kw["n_epochs"], kw["learning_rate"], run2["cfg"].clip_range)
    bounds = tr.sb3_log_bounds([[r["log_bounds"] for r in ep] for ep in per_epoch])
    _check_logs(run2["log"], want, bounds, "target_kl")
    assert run2["log"]["train/n_updates"] == kw["n_epochs"]


def test_learn_schedule_matches_sb3():
    """learning_rate = lambda p: 3e-4 p over three iterations of learn: update i runs at lr(1 - i n_steps N / total),
    as SB3 updates the progress after collect_rollouts (the last update at lr(0))."""
    from rl_rocket_6dof_b200.batch import STAT_NAMES, Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    env = Rocket6DOFBatch(N_ENVS, device=DEV, seed=6)
    params = ActorCriticParams.sb3_init(6, DEV)
    sched = lambda p: 3e-4 * p
    trainer = PPOTrainer(env, params, PPOConfig(learning_rate=sched, n_steps=T, n_epochs=1), seed=6)
    total = 3 * T * N_ENVS
    with pytest.MonkeyPatch.context() as mp:
        mbs = _capture(mp)
        logs = trainer.learn(total)
    assert len(logs) == 3 and len(mbs) == 3 * 4
    for i, log in enumerate(logs, 1):
        lr = sched(tr.sb3_progress(i, T, N_ENVS, total))
        assert log["train/learning_rate"] == lr, (i, log["train/learning_rate"], lr)
        assert all(e["adam"]["lr"] == lr for e in mbs[4 * (i - 1):4 * i])
        assert log["time/total_timesteps"] == i * T * N_ENVS
        keys = STAT_NAMES + ["mean_return", "mean_length", "landing_rate"]
        assert {"rollout/" + k for k in keys} <= set(log) and log["rollout/truncated"] == 0
    assert logs[-1]["train/learning_rate"] == 0.0


def test_step_bound_has_teeth():
    """The per-step bound fails for a short minibatch scaled by 1 / batch_size, for minibatches applied in swapped
    order, and for the clip factor omitted."""
    off, on = _run("clip_off"), _run("clip_on")
    nmb = -(-T * N_ENVS // BS)
    exceeds = lambda e, ref: float(np.max(np.abs(e["adam"]["post"].astype(np.float64) - ref["p"]) / ref["bound"]))
    short = off["mbs"][nmb - 1]
    assert len(short["idx"]) < BS
    r_scale = exceeds(short, _reference(off, short, scale=1.0 / BS))
    e1, e2 = off["mbs"][1], off["mbs"][2]
    r_swap = exceeds(e1, _reference(off, dict(e1, idx=e2["idx"])))
    k = next(i for i, ref in enumerate(on["refs"]) if ref["clip"] < 1)
    r_clip = exceeds(on["mbs"][k], _reference(on, on["mbs"][k], cfg=dataclasses.replace(on["cfg"], max_grad_norm=1e30)))
    print(f"max |kernel - wrong reference| / bound: 1/bs scale {r_scale:.3g}, swapped order {r_swap:.3g}, "
          f"no clip {r_clip:.3g}")
    assert min(r_scale, r_swap, r_clip) > rf.C_BAR
