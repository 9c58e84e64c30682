"""SB3 1.6's default separate policy / value towers (net_arch [dict(pi=[64, 64], vf=[64, 64])]) on the B200: the policy
kernels in modes 0, 2 and 3 against the float64 network (each tower held to tests/policy_ref's bound for its mode), the
entry points that refuse the network, collection with truncation bootstrap, r6_ppo_grad against float64 autograd of
SB3's loss (tests/sep_ref.py), the trainer and the Monte-Carlo dispersion."""
import ctypes as C

import numpy as np
import pytest
import torch

import policy_ref as pr
import sep_ref
from rl_rocket_6dof_b200 import _lib
from rl_rocket_6dof_b200.ppo import LAYOUT_SEP, ActorCriticParams, PPOConfig, PPOTrainer, loss_and_grad
from test_gpu_bootstrap import _check as _check_bootstrap, _mk, _twin

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ARCH = [dict(pi=[64, 64], vf=[64, 64])]
U = 2.0 ** -24


def _dev(w):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(DEV) for k, v in w.items()}


def _families():
    return {"random": sep_ref.weights(11),
            "sb3_init": {k: v.cpu().numpy() for k, v in ActorCriticParams.sb3_init(3, DEV, net_arch=ARCH).mlp().items()}}


def _policy(wd, obs_cm, tc, stochastic, ranges, seed=7, step=3):
    """r6_policy_range over the env sub-ranges `ranges` of component-major obs [14, n] (one launch per range, like the
    stream lanes): (actions, raw, values, logp)."""
    L = _lib.load()
    n = obs_cm.shape[1]
    out = [torch.full((n, 3), np.nan, device=DEV), torch.full((n, 3), np.nan, device=DEV),
           torch.full((n,), np.nan, device=DEV), torch.full((n,), np.nan, device=DEV)]
    m = _lib.make_mlp(wd)
    for first, count in ranges:
        _lib.check(L.r6_policy_range(C.byref(m), obs_cm.data_ptr(), n, first, count, tc, int(stochastic), seed, 0, step,
                                     *[o.data_ptr() for o in out], torch.cuda.current_stream().cuda_stream), L)
    torch.cuda.synchronize()
    return [o.cpu().numpy().astype(np.float64) for o in out]


def _obs(n, seed):
    rng = np.random.default_rng(seed)
    x = np.concatenate([rng.uniform(-1, 1, (n // 2, 13)), rng.standard_normal((n - n // 2, 13)) * 2.0]).astype(np.float32)
    cm = torch.zeros(14, n, device=DEV)
    cm[:13] = torch.from_numpy(np.ascontiguousarray(x.T)).to(DEV)
    return x, cm


@pytest.mark.parametrize("n", [1, 127, 128, 129, 2 ** 20 + 37])
@pytest.mark.parametrize("tc", [0, 2, 3])
def test_policy_modes_within_bound(n, tc):
    """Deterministic and stochastic outputs of every mode against forward64, per tower within C_BAR times its mode's
    bound; the stochastic sample is the mean plus the same exp(log_std) eps as the shared-trunk kernel draws, and its
    log-prob that of the sample; two lane ranges with the seam inside a tile give the same bits as one."""
    fams = _families()
    x, cm = _obs(n, n + tc)
    # the bound is evaluated on every env up to 4096 and on a sample (tile edges and the tail included) beyond
    rows = np.arange(n) if n <= 4096 else np.unique(np.r_[np.arange(0, n, 97), np.arange(n - 300, n), 0, 127, 128, 129])
    for fam, w in fams.items():
        wd = _dev(w)
        act, _, val, logp = _policy(wd, cm, tc, False, [(0, n)])
        mean64, v64 = sep_ref.forward64(w, x[rows])
        pol, vt = sep_ref.towers(w)
        bp, bv = pr.bound(pol, x[rows], tc)[:, :3], pr.bound(vt, x[rows], tc)[:, 0]
        clipped = np.clip(mean64, -1, 1)
        rp = (np.abs(act[rows] - clipped) / bp).max()
        rv = (np.abs(val[rows] - v64) / bv).max()
        print(f"{fam} n={n} tc={tc}: worst |action - forward64| / bound {rp:.3g}, value {rv:.3g}")
        assert rp <= pr.C_BAR and rv <= pr.C_BAR
        # stochastic: raw - mean is the noise of the shared-trunk kernel for the same (seed, env, step)
        _, raw, val_s, logp_s = _policy(wd, cm, tc, True, [(0, n)])
        shared = pr.weights("sb3_init")
        shared["log_std"] = w["log_std"]
        _, raw_sh, _, logp_sh = _policy(_dev(shared), cm, tc, True, [(0, n)])
        noise_sep = raw[rows] - mean64
        sg = np.exp(np.asarray(w["log_std"], np.float64))
        mean_sh64, _ = pr.forward64(shared, x[rows])
        noise_sh = raw_sh[rows] - mean_sh64
        tol = 2 * pr.C_BAR * (bp + pr.bound(shared, x[rows], tc)[:, :3]) + 4 * U * (np.abs(raw[rows]) + np.abs(raw_sh[rows]))
        assert np.all(np.abs(noise_sep - noise_sh) <= tol)
        assert np.array_equal(val_s, val)                                       # the value does not depend on the draw
        assert np.array_equal(logp_s, logp_sh)                                   # logp of the sample is the noise's
        # lanes: a seam inside a tile, outputs bit-identical to one range
        seam = n // 2 + 5 if n > 10 else n
        for a_one, a_two in zip(_policy(wd, cm, tc, True, [(0, n)]), _policy(wd, cm, tc, True, [(0, seam), (seam, n - seam)])):
            assert np.array_equal(a_one, a_two, equal_nan=True)
        if tc == 3 and n > 2 ** 20:
            # the shared trunk's bar, under its conditions: SB3's initial weights, observations in the observation space
            # Box(-1, 1) (the first half of the rows).  Elsewhere both modes are within their bounds of forward64 above.
            a0, _, v0, _ = _policy(wd, cm, 0, False, [(0, n)])
            box = slice(0, n // 2)
            d = np.abs(act[box] - a0[box]).max()
            print(f"{fam}: max |mode 3 - mode 0| actions in the observation space {d:.3g}, everywhere "
                  f"{np.abs(act - a0).max():.3g}; values {np.abs(val - v0).max():.3g}")
            if fam == "sb3_init":
                assert d <= 3e-6


def test_refusals_leave_outputs_untouched():
    from rl_rocket_6dof_b200.batch import ACT_MLP, ACT_MLP_TC
    L = _lib.load()
    w = sep_ref.weights(12)
    wd = _dev(w)
    n = 256
    _, cm = _obs(n, 1)
    m = _lib.make_mlp(wd)
    outs = [torch.full((n, 3), 7.0, device=DEV), torch.full((n, 3), 7.0, device=DEV), torch.full((n,), 7.0, device=DEV),
            torch.full((n,), 7.0, device=DEV)]
    s = torch.cuda.current_stream().cuda_stream
    rc = L.r6_policy_range(C.byref(m), cm.data_ptr(), n, 0, n, 1, 1, 0, 0, 0, *[o.data_ptr() for o in outs], s)
    assert rc == -1 and b"mma.sync" in L.r6_last_error()
    xi = torch.zeros(192, n, device=DEV)
    ls = torch.zeros(64, 3, device=DEV)
    sde = _lib.R6Sde(ls.data_ptr(), xi.data_ptr())
    for tc in (0, 3):
        rc = L.r6_policy_sde_range(C.byref(m), C.byref(sde), cm.data_ptr(), n, 0, n, tc, 1, *[o.data_ptr() for o in outs], s)
        assert rc == -1 and b"gSDE" in L.r6_last_error()
    P = ActorCriticParams.from_weights(w, DEV)
    ro = {"obs": torch.zeros(2, n, 13, device=DEV), "actions": torch.zeros(2, n, 3, device=DEV),
          "log_probs": torch.zeros(2, n, device=DEV), "advantages": torch.zeros(2, n, device=DEV),
          "returns": torch.zeros(2, n, device=DEV)}
    grad = torch.full((_lib.PPO_NPARAMS_SDE,), 7.0, device=DEV)
    terms = torch.full((_lib.PPO_NTERMS_SDE,), 7.0, dtype=torch.float64, device=DEV)
    work = torch.empty(int(L.r6_ppo_sde_work_bytes(n)), dtype=torch.uint8, device=DEV)
    rol = _lib.R6PpoRollout(ro["obs"].data_ptr(), n * 13, 1, 13, ro["actions"].data_ptr(), ro["log_probs"].data_ptr(),
                            ro["advantages"].data_ptr(), ro["returns"].data_ptr(), 2, n)
    coef = _lib.R6PpoCoef(0.2, 0.5, 0.0, None)
    idx = torch.arange(n, device=DEV)
    rc = L.r6_ppo_grad_sde(C.byref(_lib.make_mlp(P.mlp())), C.byref(sde), C.byref(rol), idx.data_ptr(), n, C.byref(coef),
                           grad.data_ptr(), terms.data_ptr(), work.data_ptr(), s)
    assert rc == -1 and b"gSDE" in L.r6_last_error()
    env = _mk(n, auto_reset=False)
    env.reset()
    before = env.obs.clone()
    for mode in (ACT_MLP, ACT_MLP_TC):
        with pytest.raises(_lib.R6Error, match="separate"):
            env.rollout(4, mode, mlp=wd)
    with pytest.raises(ValueError):
        env.step_policy(1, wd, tensor_cores=1)
    torch.cuda.synchronize()
    for o in outs:
        assert bool((o == 7.0).all())
    assert bool((grad == 7.0).all()) and bool((terms == 7.0).all())
    assert torch.equal(env.obs, before)
    with pytest.raises(ValueError):
        PPOTrainer(_mk(64), P, PPOConfig(use_sde=True))
    with pytest.raises(ValueError):
        PPOTrainer(_mk(64), P, PPOConfig(tensor_cores=1))


@pytest.mark.parametrize("tc", [0, 3])
def test_collection_bootstraps_with_the_value_tower(tc):
    """collect_rollout(bootstrap_truncated=True): values are the value tower's V of the observations the actions were
    computed from (one r6_policy_range launch over the recorded observations, bit for bit), truncations are bootstrapped
    with the value tower's V of the terminal observation against the twin batch, and 1 and 2 lanes give the same bits."""
    w = sep_ref.weights(13, scale=0.2)
    wd = _dev(w)
    n, k = 4096, 12
    a, b, c = _mk(n, 5), _mk(n, 5), _mk(n, 5, lanes=2)
    a.reset(); b.reset(); c.reset()
    ro = a.collect_rollout(k, wd, tensor_cores=tc, bootstrap_truncated=True)
    tw = _twin(b, wd, k, tc)
    rew, trunc = _check_bootstrap(ro, tw)
    assert trunc.sum() > 0
    obs = ro["obs"].permute(0, 2, 1)          # [k, 13, n]
    for j in range(k):
        cm = torch.zeros(14, n, device=DEV)
        cm[:13] = obs[j]
        _, _, v, _ = _policy(wd, cm, tc, False, [(0, n)])
        assert np.array_equal(v, ro["values"][j].cpu().numpy().astype(np.float64))
    # the value tower, not the policy tower's latent: V of the terminal observations against float64 within the bound
    x = tw["tobs"][trunc.any(1)].transpose(0, 2, 1).reshape(-1, 13)
    v = tw["val"][trunc.any(1)].reshape(-1).astype(np.float64)
    _, v64 = sep_ref.forward64(w, x)
    r = np.abs(v - v64) / pr.bound(sep_ref.towers(w)[1], x, tc)[:, 0]
    print(f"tc={tc}: worst |V - forward64| / bound {r.max():.3g}")
    assert r.max() <= pr.C_BAR
    ro2 = c.collect_rollout(k, wd, tensor_cores=tc, bootstrap_truncated=True)
    for key in ("obs", "actions", "values", "log_probs", "rewards", "dones", "advantages", "returns"):
        assert torch.equal(ro[key], ro2[key]), key


def _grad_case(w, B, seed, T=4, bad=0):
    x, a, old, adv, ret = sep_ref.minibatch(w, B, seed)
    n = -(-B // T)
    pad = T * n - B
    f = lambda v, *s: torch.from_numpy(np.ascontiguousarray(np.concatenate([v, np.zeros((pad,) + v.shape[1:], v.dtype)]))).to(DEV).reshape(*s)
    ro = {"obs": f(x, T, n, 13), "actions": f(a, T, n, 3), "log_probs": f(old, T, n), "advantages": f(adv, T, n),
          "returns": f(ret, T, n)}
    idx = torch.from_numpy(np.random.default_rng(seed).permutation(B)).to(DEV)
    if bad:
        idx = torch.cat([idx, torch.tensor([-1, T * n + 5][:bad], device=DEV)])
    return (x, a, old, adv, ret), ro, idx


@pytest.mark.parametrize("B", [1, 127, 128, 129, 2 ** 20])
def test_grad_against_float64(B):
    """r6_ppo_grad on the separate towers against float64 autograd of SB3's loss, unnormalised advantages and an entropy
    bonus, within sep_ref.bound (the per-sample float32 chain of r6_ppo.cuh plus the busiest CTA's accumulation chain and
    the two roundings of the reduction)."""
    import ppo_ref
    w = sep_ref.weights(14)
    P = ActorCriticParams.from_weights(w, DEV)
    (x, a, old, adv, ret), ro, idx = _grad_case(w, B, B % 1000)
    g, t = loss_and_grad(P, ro, idx, clip_range=0.2, vf_coef=0.5, ent_coef=0.01, normalize_advantage=False)
    g = g.cpu().numpy().astype(np.float64)
    ref, terms, mag = sep_ref.grad_sum(w, x, a, old, adv, ret, clip=0.2, vf_coef=0.5, ent_coef=0.01)
    tol = sep_ref.bound(w, x, a, old, adv, ret, clip=0.2, vf_coef=0.5, ent_coef=0.01,
                        samples_per_cta=ppo_ref.samples_per_cta(B)) + 1e-300
    worst = (np.abs(g - ref) / tol).max()
    print(f"B={B}: worst |kernel - autograd| / bound {worst:.3g}")
    assert worst <= 1.0
    tt = t.cpu().numpy()
    assert np.allclose(tt[:4], terms, rtol=1e-4, atol=1e-3 * max(1, B / 1000)) and tt[4] == 0
    g2, t2 = loss_and_grad(P, ro, idx, clip_range=0.2, vf_coef=0.5, ent_coef=0.01, normalize_advantage=False)
    assert np.array_equal(g, g2.cpu().numpy().astype(np.float64)) and torch.equal(t, t2)      # bit-reproducible
    if B >= 128:   # two halves of the minibatch add up to the whole within float32 reordering
        h = B // 2
        ga, _ = loss_and_grad(P, ro, idx[:h].contiguous(), clip_range=0.2, vf_coef=0.5, ent_coef=0.01, normalize_advantage=False)
        gb, _ = loss_and_grad(P, ro, idx[h:].contiguous(), clip_range=0.2, vf_coef=0.5, ent_coef=0.01, normalize_advantage=False)
        s = ga.cpu().numpy().astype(np.float64) + gb.cpu().numpy().astype(np.float64)
        assert np.all(np.abs(s - g) <= 2 * ppo_ref.samples_per_cta(B) * U * mag + 2 * U * np.abs(g) + 1e-9)


def test_grad_counts_bad_indices():
    w = sep_ref.weights(15)
    P = ActorCriticParams.from_weights(w, DEV)
    (x, a, old, adv, ret), ro, idx = _grad_case(w, 200, 3, bad=2)
    g, t = loss_and_grad(P, ro, idx, normalize_advantage=False)
    _, ro0, idx0 = _grad_case(w, 200, 3)
    g0, t0 = loss_and_grad(P, ro0, idx0, normalize_advantage=False)
    assert float(t[4]) == 2.0 and torch.equal(g, g0)


def test_trainer_steps_and_learn_reproducible():
    """One train() on a collected rollout: every minibatch gradient the trainer computes (captured at the call) against
    float64 autograd at the parameters of that step, and a seeded learn() of three iterations twice: bit-identical
    parameters and the same finite logs."""
    import ppo_ref
    from rl_rocket_6dof_b200 import ppo as ppo_mod
    P = ActorCriticParams.sb3_init(seed=4, device=DEV, net_arch=ARCH)
    assert P.separate and P.flat.numel() == 10375
    env = _mk(2048, 40)
    env.reset()
    cfg = PPOConfig(n_steps=8, n_epochs=2, ent_coef=0.01)
    tr = PPOTrainer(env, P, cfg, seed=1)
    ro = env.collect_rollout(cfg.n_steps, P.mlp(), bootstrap_truncated=True)
    seen = []
    orig = ppo_mod.loss_and_grad

    def spy(params, rollout, idx, **kw):
        before = {k: v.detach().cpu().numpy().copy() for k, v in params.mlp().items()}
        out = orig(params, rollout, idx, **kw)
        seen.append((before, idx.cpu().numpy(), out[0].cpu().numpy().astype(np.float64), kw))
        return out
    ppo_mod.loss_and_grad = spy
    try:
        logs = tr.train(ro)
    finally:
        ppo_mod.loss_and_grad = orig
    assert len(seen) == cfg.n_epochs * 4
    T, n = ro["advantages"].shape
    X = ro["obs"].reshape(-1, 13).cpu().numpy()
    A = ro["actions"].reshape(-1, 3).cpu().numpy()
    LP, AD, RT = (ro[k].reshape(-1).cpu().numpy() for k in ("log_probs", "advantages", "returns"))
    for before, idx, g, kw in seen[:3] + seen[-1:]:
        a64 = AD[idx].astype(np.float64)
        mu, inv = a64.mean(), 1.0 / (a64.std(ddof=1) + 1e-8)
        adv_n = ((a64 - mu) * inv).astype(np.float32).astype(np.float64)
        ref, _, _ = sep_ref.grad_sum(before, X[idx], A[idx], LP[idx], adv_n, RT[idx], clip=0.2, vf_coef=0.5, ent_coef=0.01)
        # the advantages are normalised on the device with the same float64 formula; one float32 rounding of A' each
        tol = sep_ref.bound(before, X[idx], A[idx], LP[idx], adv_n, RT[idx], clip=0.2, vf_coef=0.5, ent_coef=0.01,
                            samples_per_cta=ppo_ref.samples_per_cta(len(idx))) + 1e-300
        worst = (np.abs(g - ref) / tol).max()
        print(f"trainer step: worst |grad - autograd| / bound {worst:.3g}")
        assert worst <= 1.0
    assert all(np.isfinite(v) for v in logs.values() if isinstance(v, float))

    def run():
        e = _mk(1024, 30, seed=9)
        p = ActorCriticParams.sb3_init(seed=2, device=DEV, net_arch=ARCH)
        lg = PPOTrainer(e, p, PPOConfig(n_steps=8, n_epochs=2), seed=3).learn(3 * 8 * 1024)
        return p.flat.clone(), lg
    p1, l1 = run()
    p2, l2 = run()
    assert torch.equal(p1, p2) and not torch.equal(p1, ActorCriticParams.sb3_init(seed=2, device=DEV, net_arch=ARCH).flat)
    assert l1 == l2 and all(np.isfinite(v) for lg in l1 for v in lg.values() if isinstance(v, float))


def test_params_round_trip(tmp_path):
    from rl_rocket_6dof_b200 import policy
    P = ActorCriticParams.sb3_init(seed=8, device=DEV, net_arch=ARCH)
    P.flat.add_(torch.randn(P.flat.shape, generator=torch.Generator(device=DEV).manual_seed(0), device=DEV) * 0.01)
    path = str(tmp_path / "p.npz")
    P.save_npz(path)
    Q = ActorCriticParams.from_weights(policy.load_npz(path), DEV)
    assert Q.separate and torch.equal(P.flat, Q.flat)


def test_montecarlo_matches_step_by_step():
    """run_montecarlo with a separate-tower policy (always the two-kernel path) against the same episodes driven by
    policy_forward mode 0 + step on a twin one-episode batch: identical terminal states."""
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.montecarlo import run_montecarlo
    w = {k: v.cpu().numpy() for k, v in ActorCriticParams.sb3_init(seed=6, device=DEV, net_arch=ARCH).mlp().items()}
    n = 4096
    res = run_montecarlo(n, w, seed=5, device=DEV)
    env = Rocket6DOFBatch(n, device=DEV, seed=5, auto_reset=False, clip_reward=True, time_limit=True, lanes=1,
                          split_step=True)
    wd = _dev(w)
    env.reset()
    for _ in range(int(env.params.max_episode_steps or 1500)):
        a, _, _, _ = env.policy_forward(wd, tensor_cores=0)
        env.step(a)
        if bool(env.done.all()):
            break
    assert np.array_equal(res["terminal_state"], env.terminal_state.t().cpu().numpy())
    assert np.array_equal(res["episode_length"], env.ep_info[1].cpu().numpy().astype(np.int64))
    with pytest.raises(ValueError):
        run_montecarlo(8, w, seed=5, device=DEV, two_kernel=False)
