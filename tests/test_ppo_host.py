"""The per-sample PPO math of csrc/r6_ppo.cuh (host build, tests/ppo_hostsim) against a float64 autograd statement of
SB3 1.6's loss, the Adam / clip_grad_norm_ step against torch in float64, and argument checks of r6_ppo_grad /
r6_adam_step that need no GPU."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import ppo_hostsim
import policy_ref as pr
import ppo_ref as rf
import ppo_train_ref as tr


def autograd_sum(w, x, a, old, adv_n, ret, clip, vf_coef, ent_coef):
    """Sum over samples of the gradient of pg + vf_coef (R - v)^2 - ent_coef entropy: len(x) times the gradient of
    SB3's minibatch-mean loss (ppo_train_ref.sb3_loss), torch float64 autograd."""
    P = {k: torch.tensor(np.asarray(v, np.float32).astype(np.float64), requires_grad=True) for k, v in w.items()}
    loss, _ = tr.sb3_loss(P, x, a, old, adv_n, ret, clip, vf_coef, ent_coef)
    (len(x) * loss).backward()
    return np.concatenate([P[k].grad.numpy().reshape(-1) for k, _ in rf.LAYOUT])


CASES = [(f, o, ent) for f in pr.FAMILIES for o in ("golden", "uniform", "normal5") for ent in (0.0, 0.01)]


@pytest.mark.parametrize("family,obs,ent", CASES)
def test_host_sample_grad_matches_autograd(family, obs, ent):
    n = 96
    w = pr.weights(family)
    x = pr.obs_sets(n, seed=3)[obs]
    a, old, adv, ret = rf.minibatch(w, x, seed=7)
    st = rf.adv_stats(adv)
    adv_n = (adv.astype(np.float64) - st[0]) * st[1]
    g, terms = ppo_hostsim.ppo_sample_grad(rf.flat(w), x, a, old, adv, ret, adv_stats=st, ent_coef=ent)
    ref = autograd_sum(w, x, a, old, adv_n, ret, 0.2, 0.5, ent)
    q = rf.per_sample(w, x, a, old, adv_n, ret, ent_coef=ent)
    g64, t64 = rf.grad_sum(q)
    assert np.allclose(g64, ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())        # the reference is the autograd loss
    bnd, tb = rf.bound(q, ent_coef=ent, samples_per_cta=1)
    err = np.abs(g.astype(np.float64).sum(0) - ref)
    assert np.all(err <= rf.C_BAR * bnd), (family, obs, float((err / bnd).max()))
    # both clip branches and both advantage signs are present
    assert (q["wgt"] == 0).any() and (q["wgt"] != 0).any() and (adv_n > 0).any() and (adv_n < 0).any()
    assert np.array_equal(terms[:, 2], q["clipped"].astype(np.float32))
    assert np.all(np.abs(terms[:, :2].astype(np.float64).sum(0) - t64[:2]) <= rf.C_BAR * tb[:2])


def test_bound_has_teeth():
    """Omitting the advantage normalisation or a sample moves the host sum outside the bar."""
    w = pr.weights("sb3_init")
    x = pr.obs_sets(64, seed=1)["uniform"]
    a, old, adv, ret = rf.minibatch(w, x, seed=2)
    st = rf.adv_stats(adv)
    q = rf.per_sample(w, x, a, old, (adv.astype(np.float64) - st[0]) * st[1], ret)
    g64, _ = rf.grad_sum(q)
    bnd, _ = rf.bound(q, samples_per_cta=64)
    g_raw, _ = ppo_hostsim.ppo_sample_grad(rf.flat(w), x, a, old, adv, ret)
    assert np.any(np.abs(g_raw.astype(np.float64).sum(0) - g64) > rf.C_BAR * bnd)
    g, _ = ppo_hostsim.ppo_sample_grad(rf.flat(w), x, a, old, adv, ret, adv_stats=st)
    assert np.any(np.abs(g[1:].astype(np.float64).sum(0) - g64) > rf.C_BAR * bnd)


@pytest.mark.parametrize("max_norm", [0.5, 1e6, 0.0])
def test_adam_step_matches_torch(max_norm):
    """hs_adam_step (r6_adam_step's code) against torch.optim.Adam(eps=1e-5) + clip_grad_norm_ in float64, 3 steps."""
    rng = np.random.default_rng(0)
    P = 10311
    p32 = rng.standard_normal(P).astype(np.float32)
    m32, v32 = np.zeros(P, np.float32), np.zeros(P, np.float32)
    pt = torch.tensor(p32.astype(np.float64), requires_grad=True)
    opt = torch.optim.Adam([pt], lr=3e-4, eps=1e-5)
    B = 100
    for step in range(1, 4):
        gs = (rng.standard_normal(P) * 0.05 * B).astype(np.float32)
        coef = adam_coef(3e-4, max_norm, 1.0 / B)
        norm = ppo_hostsim.adam_step(p32, gs, m32, v32, coef, step)
        pt.grad = torch.tensor(gs.astype(np.float64) / B)
        tn = float(torch.linalg.vector_norm(pt.grad))
        if max_norm > 0:
            torch.nn.utils.clip_grad_norm_([pt], max_norm)
        opt.step()
        assert abs(norm - tn) <= 1e-6 * tn
        ref = pt.detach().numpy()
        # float32 arithmetic against float64: a few ulp of the update plus the parameter's own rounding
        assert np.all(np.abs(p32 - ref) <= 4 * 2.0 ** -24 * np.abs(ref) + 1e-3 * 3e-4 * step)
    if max_norm == 0.5:
        assert norm > max_norm          # the clip was active


@pytest.mark.parametrize("family,max_norm", [("saturating", 0.5), ("sb3_init", 1e6)])
def test_sb3_train_step_matches_grad_sum_and_bounds_the_host_step(family, max_norm):
    """ppo_train_ref's SB3 statement (autograd of the minibatch-mean loss, clip_grad_norm_, Adam) on one ppo_ref
    minibatch: its gradient is grad_sum / B to float64 round-off and its logged terms the term sums / B; the host build
    of r6_adam_step fed the host build's gradient sum lands within C_BAR x the per-step bound, and the bound fails for a
    step scaled by 1 / batch_size instead of 1 / len(idx) (clip off) and for the clip factor omitted (clip on)."""
    from rl_rocket_6dof_b200.ppo import NPARAMS, PPOConfig
    w = pr.weights(family)
    n, B, step, lr, ent = 400, 300, 3, 3e-4, 0.01
    x = pr.obs_sets(n, seed=4)["uniform"]
    a, old, adv, ret = rf.minibatch(w, x, seed=5)
    ro = dict(obs=x, actions=a, log_probs=old, advantages=adv, returns=ret)
    idx = np.random.default_rng(6).permutation(n)[:B]
    cfg = PPOConfig(ent_coef=ent, max_grad_norm=max_norm)
    rng = np.random.default_rng(7)
    p = rf.flat(w)
    m = (rng.standard_normal(NPARAMS) * 1e-2).astype(np.float32)
    v = (rng.standard_normal(NPARAMS) ** 2 * 1e-4).astype(np.float32)
    m[::7], v[::7] = 0, 0                                      # moments that start at zero, as after sb3_init
    ref = tr.reference_step(p, m, v, step, ro, idx, lr, cfg)
    st = rf.adv_stats(adv[idx])
    q = rf.per_sample(w, x[idx], a[idx], old[idx], (adv[idx].astype(np.float64) - st[0]) * st[1], ret[idx], ent_coef=ent)
    g64, t64 = rf.grad_sum(q)
    assert np.allclose(B * ref["grad"], g64, rtol=1e-10, atol=1e-10 * np.abs(g64).max())
    for k, j in (("pg", 0), ("value_loss", 1), ("clip_fraction", 2), ("approx_kl", 3)):
        assert math.isclose(B * ref["logs"][k], t64[j], rel_tol=1e-10, abs_tol=1e-12), k
    assert (ref["clip"] < 1) == (max_norm == 0.5)
    gs = ppo_hostsim.ppo_sample_grad(p, x[idx], a[idx], old[idx], adv[idx], ret[idx], adv_stats=st, ent_coef=ent)[0]
    gs = gs.astype(np.float64).sum(0).astype(np.float32)
    p32, m32, v32 = p.copy(), m.copy(), v.copy()
    norm = ppo_hostsim.adam_step(p32, gs, m32, v32, adam_coef(lr, max_norm, 1.0 / B), step)
    assert abs(norm - ref["norm"]) <= 1e-3 * ref["norm"]
    r = np.abs(p32 - ref["p"]) / ref["bound"]
    assert np.all(r <= rf.C_BAR), (float(r.max()), int(r.argmax()))
    wrong = (tr.reference_step(p, m, v, step, ro, idx, lr, cfg, scale=1.0 / (B + 100)) if max_norm > 1 else
             tr.reference_step(p, m, v, step, ro, idx, lr, PPOConfig(ent_coef=ent, max_grad_norm=1e30)))
    assert np.any(np.abs(p32 - wrong["p"]) > rf.C_BAR * wrong["bound"])


def adam_coef(lr, max_norm, scale):
    from rl_rocket_6dof_b200 import _lib
    return _lib.R6AdamCoef(lr, 0.9, 0.999, 1e-5, max_norm, scale)


def test_ppo_entries_reject_bad_arguments_without_a_gpu():
    """Null pointers, a missing critic head / log_std, negative sizes and step 0 return R6_EINVAL (-1) before any CUDA
    call."""
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    buf = (C.c_float * 16)()
    full = _lib.R6Mlp(*([C.addressof(buf)] * 9))
    no_head = _lib.R6Mlp(*([C.addressof(buf)] * 6))
    ro = _lib.R6PpoRollout(C.addressof(buf), 1, 1, 1, C.addressof(buf), C.addressof(buf), C.addressof(buf),
                           C.addressof(buf), 1, 1)
    coef = _lib.R6PpoCoef(0.2, 0.5, 0.0, None)
    p = C.addressof(buf)
    assert L.r6_ppo_grad(None, C.byref(ro), p, 1, C.byref(coef), p, p, p, None) == -1
    assert L.r6_ppo_grad(C.byref(no_head), C.byref(ro), p, 1, C.byref(coef), p, p, p, None) == -1
    assert b"critic" in L.r6_last_error()
    assert L.r6_ppo_grad(C.byref(full), None, p, 1, C.byref(coef), p, p, p, None) == -1
    assert L.r6_ppo_grad(C.byref(full), C.byref(ro), None, 1, C.byref(coef), p, p, p, None) == -1
    assert L.r6_ppo_grad(C.byref(full), C.byref(ro), p, 1, None, p, p, p, None) == -1
    assert L.r6_ppo_grad(C.byref(full), C.byref(ro), p, -1, C.byref(coef), p, p, p, None) == -1
    ac = _lib.R6AdamCoef(3e-4, 0.9, 0.999, 1e-5, 0.5, 1.0)
    assert L.r6_adam_step(None, p, p, p, 16, C.byref(ac), 1, None, None) == -1
    assert L.r6_adam_step(p, p, p, p, 16, None, 1, None, None) == -1
    assert L.r6_adam_step(p, p, p, p, 16, C.byref(ac), 0, None, None) == -1
    assert L.r6_ppo_work_bytes(0) == 0 and L.r6_ppo_work_bytes(1) > 4 * 10311


def test_sb3_init_and_layout_without_a_gpu():
    from rl_rocket_6dof_b200 import ppo
    assert sum(int(np.prod(s)) for _, s in ppo.LAYOUT) == ppo.NPARAMS == 10311
    off = 0
    for name, s in ppo.LAYOUT:
        if name == "w1":
            assert off == 1792 and off % 4 == 0
        off += int(np.prod(s))
    cfg = ppo.PPOConfig()
    assert (cfg.learning_rate, cfg.n_epochs, cfg.clip_range, cfg.ent_coef, cfg.vf_coef, cfg.max_grad_norm) == \
        (3e-4, 10, 0.2, 0.0, 0.5, 0.5)
    assert cfg.normalize_advantage and cfg.target_kl is None and (cfg.gamma, cfg.gae_lambda) == (0.99, 0.95)
    assert math.isclose(ppo._LOG_SQRT_2PI, 0.9189385332046727)
