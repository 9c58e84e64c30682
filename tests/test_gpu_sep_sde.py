"""gSDE on SB3 1.6's separate towers (PPO("MlpPolicy", env, use_sde=True) without policy_kwargs) on the B200: the policy
kernels of r6_policy_sde_sep_range in modes 0, 2 and 3 against float64, the refusals of the new entry points, collection
with sde_sample_freq and truncation bootstrap, r6_ppo_grad_sde_sep against float64 autograd of SB3's loss
(tests/sepsde_ref.py) with teeth, the trainer one Adam step at a time, and the Monte-Carlo dispersion."""
import ctypes as C

import numpy as np
import pytest
import torch

import policy_ref as pr
import ppo_ref
import sde_hostsim
import sep_ref
import sepsde_hostsim
import sepsde_ref
from rl_rocket_6dof_b200 import _lib
from rl_rocket_6dof_b200.ppo import NET_ARCH_SEP, ActorCriticParams, PPOConfig, PPOTrainer, loss_and_grad
from test_gpu_bootstrap import _check as _check_bootstrap, _mk, _twin

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
K = 1024                        # the per-sample gradient bar of sde_ref.reference_step: K u sum_s |per-sample gradient|


def _dev(w):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(DEV) for k, v in w.items()}


def _obs(n, seed):
    rng = np.random.default_rng(seed)
    x = np.concatenate([rng.uniform(-1, 1, (n // 2, 13)), rng.standard_normal((n - n // 2, 13)) * 2.0]).astype(np.float32)
    cm = torch.zeros(14, n, device=DEV)
    cm[:13] = torch.from_numpy(np.ascontiguousarray(x.T)).to(DEV)
    return x, cm


def _noise(n, seed=7, step=3):
    L = _lib.load()
    xi = torch.empty(192, n, device=DEV)
    _lib.check(L.r6_sde_noise(n, 0, n, seed, 0, step, xi.data_ptr(), torch.cuda.current_stream().cuda_stream), L)
    return xi


def _sde_policy(wd, xi, obs_cm, tc, stochastic, ranges):
    """r6_policy_sde_sep_range over the env sub-ranges `ranges` (one launch each): (actions, raw, values, logp)."""
    L = _lib.load()
    n = obs_cm.shape[1]
    out = [torch.full((n, 3), np.nan, device=DEV), torch.full((n, 3), np.nan, device=DEV),
           torch.full((n,), np.nan, device=DEV), torch.full((n,), np.nan, device=DEV)]
    m = _lib.make_mlp(wd)
    sde = _lib.R6Sde(wd["log_std"].data_ptr(), xi.data_ptr())
    for first, count in ranges:
        _lib.check(L.r6_policy_sde_sep_range(C.byref(m), C.byref(sde), obs_cm.data_ptr(), n, first, count, tc, int(stochastic),
                                             *[o.data_ptr() for o in out], torch.cuda.current_stream().cuda_stream), L)
    torch.cuda.synchronize()
    return [o.cpu().numpy().astype(np.float64) for o in out]


def _plain_policy(wd, obs_cm, tc):
    """r6_policy_range on the same towers, deterministic (make_mlp passes no [64, 3] log_std): (actions, values)."""
    L = _lib.load()
    n = obs_cm.shape[1]
    act, val = torch.empty(n, 3, device=DEV), torch.empty(n, device=DEV)
    m = _lib.make_mlp(wd)
    _lib.check(L.r6_policy_range(C.byref(m), obs_cm.data_ptr(), n, 0, n, tc, 0, 0, 0, 0, act.data_ptr(), None, val.data_ptr(),
                                 None, torch.cuda.current_stream().cuda_stream), L)
    torch.cuda.synchronize()
    return act.cpu().numpy().astype(np.float64), val.cpu().numpy().astype(np.float64)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 4096, 2 ** 20 + 37])
@pytest.mark.parametrize("tc", [0, 2, 3])
def test_policy_sde_sampling(n, tc):
    """raw = mean + hp (sigma xi), V and log_prob against float64, with test_gpu_sde.test_policy_sde_sampling's bars on
    the policy tower's bound (policy_ref.bound) and the value tower held to C_BAR times its bound as in
    test_gpu_separate; deterministic actions and values bit-identical to r6_policy_range; one, two and three sub-ranges
    bit-identical."""
    w = sepsde_ref.weights(21)
    w["w2"] = w["w2"] * 3.0                         # a mean that is not ~0
    wd = _dev(w)
    x, cm = _obs(n, n + tc)
    xi = _noise(n)
    rows = np.arange(n) if n <= 4096 else np.unique(np.r_[np.arange(0, n, 97), np.arange(n - 300, n), 0, 127, 128, 129])
    act, raw, val, logp = _sde_policy(wd, xi, cm, tc, True, [(0, n)])
    xr = xi.cpu().numpy().T[rows].astype(np.float64)
    raw64, logp64, mean64, v64, hp64 = sepsde_ref.sample(w, x[rows], xr)
    pol, vt = sep_ref.towers(w)
    E = np.exp(w["log_std"].astype(np.float64))[None] * xr.reshape(-1, 64, 3)
    hE = np.abs(hp64[:, :, None] * E).sum(1)
    act_acc = 2e-3 if tc == 2 else 4e-6
    bar = pr.bound(pol, x[rows], tc)[:, :3] + 64 * U * hE + act_acc * np.abs(E).sum(1) + 1e-6
    r_raw = (np.abs(raw[rows] - raw64) / bar).max()
    r_val = (np.abs(val[rows] - v64) / pr.bound(vt, x[rows], tc)[:, 0]).max()
    lbar = 1e-4 * (1 + np.abs(logp64)) + (2e-2 if tc == 2 else 1e-3)
    r_lp = (np.abs(logp[rows] - logp64) / lbar).max()
    print(f"n={n} tc={tc}: worst |raw - raw64| / bar {r_raw:.3f}, |V - V64| / bound {r_val:.3f} (bar {pr.C_BAR}), "
          f"|logp - logp64| / bar {r_lp:.3f}")
    assert r_raw <= 1.0 and r_val <= pr.C_BAR and r_lp <= 1.0
    assert np.array_equal(act, np.clip(raw, -1, 1))
    # deterministic outputs bit-identical to r6_policy_range on the same towers; the value does not depend on the draw
    dact, draw, dval, _ = _sde_policy(wd, xi, cm, tc, False, [(0, n)])
    pact, pval = _plain_policy(wd, cm, tc)
    assert np.array_equal(dact, pact) and np.array_equal(dval, pval) and np.array_equal(val, pval)
    # sub-ranges (seams inside tiles): the same bits as one launch
    for ranges in ([(0, n // 2 + 5), (n // 2 + 5, n - n // 2 - 5)] if n > 10 else [(0, n)],
                   [(0, n // 3 + 1), (n // 3 + 1, n // 3), (2 * (n // 3) + 1, n - 2 * (n // 3) - 1)] if n > 10 else [(0, n)]):
        for one, many in zip((act, raw, val, logp), _sde_policy(wd, xi, cm, tc, True, ranges)):
            assert np.array_equal(one, many, equal_nan=True)


def test_refusals_leave_outputs_untouched():
    """The new entry points refuse a shared trunk, mode 1, a misaligned vf_w1 and a bad clip_range_vf: R6_EINVAL, nothing
    written."""
    L = _lib.load()
    s = torch.cuda.current_stream().cuda_stream
    n = 256
    _, cm = _obs(n, 1)
    w = sepsde_ref.weights(22)
    wd = _dev(w)
    xi = torch.zeros(192, n, device=DEV)
    sde = _lib.R6Sde(wd["log_std"].data_ptr(), xi.data_ptr())
    outs = [torch.full((n, 3), 7.0, device=DEV), torch.full((n, 3), 7.0, device=DEV), torch.full((n,), 7.0, device=DEV),
            torch.full((n,), 7.0, device=DEV)]
    shared = ActorCriticParams.sb3_init(seed=0, device=DEV, use_sde=True)
    buf = torch.zeros(64 * 64 + 1, device=DEV)
    mis = dict(wd, vf_w1=buf[1:].view(64, 64))
    mis["vf_w1"].copy_(wd["vf_w1"])
    cases = [(_lib.make_mlp(shared.mlp()), 0, b"r6_policy_sde_range"), (_lib.make_mlp(wd), 1, b"mma.sync"),
             (_lib.make_mlp(mis), 3, b"aligned"), (_lib.make_mlp(mis), 2, b"aligned")]
    for m, tc, msg in cases:
        rc = L.r6_policy_sde_sep_range(C.byref(m), C.byref(sde), cm.data_ptr(), n, 0, n, tc, 1, *[o.data_ptr() for o in outs], s)
        assert rc == -1 and msg in L.r6_last_error(), (tc, L.r6_last_error())
    P = ActorCriticParams.from_weights(w, DEV)
    assert P.separate and P.use_sde
    ro = {k: torch.zeros(2, n, *s_, device=DEV) for k, s_ in (("obs", (13,)), ("actions", (3,)), ("log_probs", ()),
                                                               ("advantages", ()), ("returns", ()), ("values", ()))}
    rol = _lib.R6PpoRollout(ro["obs"].data_ptr(), n * 13, 1, 13, ro["actions"].data_ptr(), ro["log_probs"].data_ptr(),
                            ro["advantages"].data_ptr(), ro["returns"].data_ptr(), 2, n, ro["values"].data_ptr())
    grad = torch.full((_lib.PPO_NPARAMS_SEP_SDE,), 7.0, device=DEV)
    terms = torch.full((_lib.PPO_NTERMS_SDE,), 7.0, dtype=torch.float64, device=DEV)
    work = torch.empty(int(L.r6_ppo_sde_work_bytes(n)), dtype=torch.uint8, device=DEV)
    idx = torch.arange(n, device=DEV)
    psde = _lib.R6Sde(P.log_std.data_ptr(), None)
    for m, vfc, msg in ((_lib.make_mlp(shared.mlp()), 0.0, b"r6_ppo_grad_sde"), (_lib.make_mlp(P.mlp()), -0.1, b"clip_range_vf"),
                        (_lib.make_mlp(P.mlp()), float("nan"), b"clip_range_vf")):
        coef = _lib.R6PpoCoef(0.2, 0.5, 0.0, None, vfc)
        rc = L.r6_ppo_grad_sde_sep(C.byref(m), C.byref(psde), C.byref(rol), idx.data_ptr(), n, C.byref(coef), grad.data_ptr(),
                                   terms.data_ptr(), work.data_ptr(), s)
        assert rc == -1 and msg in L.r6_last_error(), L.r6_last_error()
    rol.old_values = None
    coef = _lib.R6PpoCoef(0.2, 0.5, 0.0, None, 0.2)
    rc = L.r6_ppo_grad_sde_sep(C.byref(_lib.make_mlp(P.mlp())), C.byref(psde), C.byref(rol), idx.data_ptr(), n, C.byref(coef),
                               grad.data_ptr(), terms.data_ptr(), work.data_ptr(), s)
    assert rc == -1 and b"old_values" in L.r6_last_error()
    torch.cuda.synchronize()
    for o in outs:
        assert bool((o == 7.0).all())
    assert bool((grad == 7.0).all()) and bool((terms == 7.0).all())
    with pytest.raises(ValueError):
        PPOTrainer(_mk(64), P, PPOConfig(use_sde=True, tensor_cores=1))


@pytest.mark.parametrize("freq", [-1, 4])
def test_sde_sample_freq(freq):
    """Two lanes: the noise each env used, recovered from raw - mean, is the draw keyed steps_done + j - j mod freq."""
    n, k = 2048, 16
    b = _mk(n, seed=5, lanes=2)
    b.reset()
    w = sepsde_ref.weights(23)
    ro = b.collect_rollout(k, _dev(w), tensor_cores=0, sde_sample_freq=freq)
    torch.cuda.synchronize()
    s0 = b.steps_done - k
    for j in range(k):
        x = ro["obs"][j].cpu().numpy()
        key = s0 + (j - j % freq if freq > 0 else 0)
        xi = sde_hostsim.sde_noise(5, np.arange(n, dtype=np.uint64), key).astype(np.float64)
        raw64 = sepsde_ref.sample(w, x, xi)[0]
        err = np.abs(ro["actions"][j].cpu().numpy() - raw64).max()
        assert err < 1e-3, (j, err)
        if freq > 0 and j % freq:
            xi_other = sde_hostsim.sde_noise(5, np.arange(n, dtype=np.uint64), key + 1).astype(np.float64)
            assert np.abs(ro["actions"][j].cpu().numpy() - sepsde_ref.sample(w, x, xi_other)[0]).max() > 1e-2


@pytest.mark.parametrize("tc", [0, 3])
def test_collection_bootstraps_with_the_value_tower(tc):
    """collect_rollout(bootstrap_truncated=True) with gSDE: rewards bootstrapped bit for bit against a twin batch stepped
    through policy_forward, values the value tower's (one r6_policy_range launch over the recorded observations), and one
    and two lanes give the same bits."""
    w = sepsde_ref.weights(24, scale=0.2)
    wd = _dev(w)
    n, k = 4096, 12
    a, b, c = _mk(n, 5), _mk(n, 5), _mk(n, 5, lanes=2)
    a.reset(); b.reset(); c.reset()
    ro = a.collect_rollout(k, wd, tensor_cores=tc, bootstrap_truncated=True)
    tw = _twin(b, wd, k, tc)
    _, trunc = _check_bootstrap(ro, tw)
    assert trunc.sum() > 0
    obs = ro["obs"].permute(0, 2, 1)
    for j in range(k):
        cm = torch.zeros(14, n, device=DEV)
        cm[:13] = obs[j]
        _, v = _plain_policy(wd, cm, tc)
        assert np.array_equal(v, ro["values"][j].cpu().numpy().astype(np.float64))
    x = tw["tobs"][trunc.any(1)].transpose(0, 2, 1).reshape(-1, 13)
    _, v64 = sep_ref.forward64(w, x)
    r = np.abs(tw["val"][trunc.any(1)].reshape(-1) - v64) / pr.bound(sep_ref.towers(w)[1], x, tc)[:, 0]
    print(f"tc={tc}: worst |V(terminal obs) - forward64| / bound {r.max():.3g}")
    assert r.max() <= pr.C_BAR
    ro2 = c.collect_rollout(k, wd, tensor_cores=tc, bootstrap_truncated=True)
    for key in ("obs", "actions", "values", "log_probs", "rewards", "dones", "advantages", "returns"):
        assert torch.equal(ro[key], ro2[key]), key


def _grad_case(w, B, seed, T=4, bad=0):
    x, a, old, adv, ret, vold = sepsde_ref.minibatch(w, B, seed)
    n = -(-B // T)
    pad = T * n - B
    f = lambda v, *s: torch.from_numpy(np.ascontiguousarray(np.concatenate([v, np.zeros((pad,) + v.shape[1:], v.dtype)]))).to(DEV).reshape(*s)
    ro = {"obs": f(x, T, n, 13), "actions": f(a, T, n, 3), "log_probs": f(old, T, n), "advantages": f(adv, T, n),
          "returns": f(ret, T, n), "values": f(vold, T, n)}
    idx = torch.from_numpy(np.random.default_rng(seed).permutation(B)).to(DEV)
    if bad:
        idx = torch.cat([idx, torch.tensor([-1, T * n + 5][:bad], device=DEV)])
    return (x, a, old, adv, ret, vold), ro, idx


@pytest.mark.parametrize("B", [1, 127, 128, 129, 2 ** 14, 2 ** 18 + 129])
def test_grad_against_float64(B):
    """r6_ppo_grad_sde_sep against float64 autograd of SB3's loss (unnormalised advantages, entropy bonus; clip_range_vf
    off and on) within K u sum_s |per-sample gradient| (K = 1024 as sde_ref.reference_step, magnitudes from the host
    build); bit-reproducible; two halves add up to the whole within the reorder bound of test_gpu_separate.  At 2^14
    the teeth: the value latent as h, the gradient let through std and one perturbed log_std entry each fail the bar."""
    w = sepsde_ref.weights(25)
    P = ActorCriticParams.from_weights(w, DEV)
    assert P.separate and P.use_sde
    data, ro, idx = _grad_case(w, B, B % 1000)
    x, a, old, adv, ret, vold = data
    for vfc in ((None, 0.15) if B < 2 ** 18 else (None,)):
        kw = dict(clip_range=0.2, vf_coef=0.5, ent_coef=0.01, normalize_advantage=False, clip_range_vf=vfc)
        g, t = loss_and_grad(P, ro, idx, **kw)
        g = g.cpu().numpy().astype(np.float64)
        ref, terms, ent = sepsde_ref.grad_sum(w, x, a, old, adv, ret, clip=0.2, vf_coef=0.5, ent_coef=0.01,
                                              clip_range_vf=vfc, old_values=vold)
        mag = sepsde_hostsim.magnitudes(sepsde_ref.flat(w), x, a, old, adv, ret, vold, vfc or 0.0, ent_coef=0.01)
        tol = K * U * mag + 1e-30
        worst = (np.abs(g - ref) / tol).max()
        print(f"B={B} vfc={vfc}: worst |kernel - autograd| / (K u sum|per-sample|) {worst:.3g}")
        assert worst <= 1.0
        tt = t.cpu().numpy()
        assert np.allclose(tt[:4], terms, rtol=1e-4, atol=1e-3 * max(1, B / 1000)) and tt[4] == 0
        assert abs(tt[5] - ent.sum()) <= 1e-5 * abs(ent.sum()) + 1e-3
        g2, t2 = loss_and_grad(P, ro, idx, **kw)
        assert np.array_equal(g, g2.cpu().numpy().astype(np.float64)) and torch.equal(t, t2)      # bit-reproducible
        if B >= 128:
            h = B // 2
            ga, _ = loss_and_grad(P, ro, idx[:h].contiguous(), **kw)
            gb, _ = loss_and_grad(P, ro, idx[h:].contiguous(), **kw)
            s = ga.cpu().numpy().astype(np.float64) + gb.cpu().numpy().astype(np.float64)
            assert np.all(np.abs(s - g) <= 2 * ppo_ref.samples_per_cta(B) * U * mag + 2 * U * np.abs(g) + 1e-9)
        if B == 2 ** 14:
            w2 = dict(w, log_std=w["log_std"].copy())
            w2["log_std"][7, 2] += 1e-2
            for name, ww, bad_kw in (("value latent as h", w, dict(latent="value")), ("not detached", w, dict(detach=False)),
                                     ("log_std[7][2] + 1e-2", w2, {})):
                bad, _, _ = sepsde_ref.grad_sum(ww, x, a, old, adv, ret, clip=0.2, vf_coef=0.5, ent_coef=0.01,
                                                clip_range_vf=vfc, old_values=vold, **bad_kw)
                f = (np.abs(g - bad) / tol).max()
                print(f"teeth ({name}, vfc={vfc}): {f:.3g} x bar")
                assert f > 1.0


def test_grad_counts_bad_indices():
    w = sepsde_ref.weights(26)
    P = ActorCriticParams.from_weights(w, DEV)
    _, ro, idx = _grad_case(w, 200, 3, bad=2)
    g, t = loss_and_grad(P, ro, idx, normalize_advantage=False)
    _, ro0, idx0 = _grad_case(w, 200, 3)
    g0, t0 = loss_and_grad(P, ro0, idx0, normalize_advantage=False)
    assert float(t[4]) == 2.0 and torch.equal(g, g0) and torch.equal(t[5], t0[5])


def _sep_sde_params(seed):
    p = ActorCriticParams.sb3_init(seed=seed, device=DEV, use_sde=True, net_arch=NET_ARCH_SEP)
    g = torch.Generator().manual_seed(seed + 1)
    p.log_std.copy_((torch.rand(64, 3, generator=g) * 1.5 - 1.0).to(DEV))     # not constant
    return p


def test_trainer_steps_match_sb3():
    """One PPOTrainer.train with use_sde=True on the separate towers (2048 envs x 16 steps, batch_size 10,000, one epoch,
    entropy bonus) against sepsde_ref.reference_step one Adam step at a time from the kernels' own pre-step state, and
    the train/ logs (entropy_loss from the kernel's entropy term, std); a log_std entry perturbed by 1e-3 in the
    reference breaks the check."""
    from rl_rocket_6dof_b200 import ppo
    n_envs, T, bs = 2048, 16, 10000
    b = _mk(n_envs, seed=4)
    b.reset()
    p = _sep_sde_params(4)
    cfg = PPOConfig(use_sde=True, n_steps=T, batch_size=bs, n_epochs=1, ent_coef=0.01)
    ro = b.collect_rollout(T, p.mlp(), tensor_cores=3)
    host = {k: ro[k].contiguous().cpu().numpy().reshape(T * n_envs, -1) for k in ("obs", "actions")}
    host.update({k: ro[k].cpu().numpy().reshape(-1) for k in ("log_probs", "advantages", "returns", "values")})
    trainer = PPOTrainer(b, p, cfg, seed=4)
    steps, perms = [], []
    real, real_lg = ppo.adam_step, ppo.loss_and_grad

    def adam_step(params, grad_sum, m, v, **kw):
        rec = dict(params=params.cpu().numpy(), m=m.cpu().numpy(), v=v.cpu().numpy(), **kw)
        real(params, grad_sum, m, v, **kw)
        rec["post"] = params.cpu().numpy()
        steps.append(rec)

    def loss_and_grad_spy(params, rollout, idx, **kw):
        perms.append(idx.cpu().numpy())
        return real_lg(params, rollout, idx, **kw)

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(ppo, "adam_step", adam_step)
        mp.setattr(ppo, "loss_and_grad", loss_and_grad_spy)
        log = trainer.train(ro)
    assert [len(q) for q in perms] == [bs, bs, bs, T * n_envs - 3 * bs] and len(steps) == 4
    worst, ents = 0.0, []
    for st, idx in zip(steps, perms):
        adv_n = sepsde_ref.tr.normalized_advantages(host["advantages"][idx], True)
        err = sepsde_hostsim.magnitudes(st["params"], host["obs"][idx], host["actions"][idx], host["log_probs"][idx], adv_n,
                                        host["returns"][idx], clip=cfg.clip_range, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef)
        ref = sepsde_ref.reference_step(st["params"], st["m"], st["v"], st["step"], host, idx, st["lr"], cfg, err_sum=err)
        r = np.abs(st["post"].astype(np.float64) - ref["p"]) / ref["bound"]
        worst = max(worst, r.max())
        ents.append(ref["entropy"])
        assert r.max() <= 1.0, (st["step"], r.max(), int(r.argmax()))
        if st["step"] == 1:
            bad = st["params"].copy()
            bad[sepsde_ref.LOG_STD + 3 * 7 + 2] += 1e-3
            ref2 = sepsde_ref.reference_step(bad, st["m"], st["v"], st["step"], host, idx, st["lr"], cfg, err_sum=err)
            r2 = (np.abs(st["post"].astype(np.float64) - ref2["p"]) / ref2["bound"]).max()
            print(f"teeth (log_std[7][2] + 1e-3): {r2:.1f} x bound")
            assert r2 > 1.0
    print(f"separate-tower gSDE trainer: worst |post-step - reference| / bound = {worst:.3f}")
    assert abs(log["train/entropy_loss"] + np.mean(ents)) <= 1e-5 * abs(np.mean(ents))
    assert log["train/std"] == pytest.approx(float(np.exp(p.log_std.double().cpu().numpy()).mean()), rel=1e-12)


def test_learn_reproducible():
    """A seeded learn of three iterations with sde_sample_freq=4 and clip_range_vf, twice: bit-identical parameters
    and the same finite logs."""
    def run():
        e = _mk(1024, 30, seed=9)
        p = ActorCriticParams.sb3_init(seed=2, device=DEV, use_sde=True, net_arch=[dict(pi=[64, 64], vf=[64, 64])])
        cfg = PPOConfig(use_sde=True, sde_sample_freq=4, clip_range_vf=0.2, n_steps=8, n_epochs=2, ent_coef=0.01)
        lg = PPOTrainer(e, p, cfg, seed=3).learn(3 * 8 * 1024)
        return p.flat.clone(), lg
    p1, l1 = run()
    p2, l2 = run()
    init = ActorCriticParams.sb3_init(seed=2, device=DEV, use_sde=True, net_arch=NET_ARCH_SEP).flat
    assert torch.equal(p1, p2) and not torch.equal(p1, init)
    assert len(l1) == 3 and l1 == l2
    assert all(np.isfinite(v) for lg in l1 for v in lg.values() if isinstance(v, float))
    assert all("train/clip_range_vf" in lg for lg in l1)


def test_montecarlo_matches_step_by_step():
    """run_montecarlo with a gSDE separate-tower policy (deterministic, two-kernel path) against the same episodes driven
    by policy_forward mode 0 (r6_policy_sde_sep_range, deterministic) + step on a twin one-episode batch: identical
    terminal states."""
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.montecarlo import run_montecarlo
    w = {k: v.cpu().numpy() for k, v in _sep_sde_params(6).mlp().items()}
    assert w["log_std"].shape == (64, 3)
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
