"""SB3's value clipping (`clip_range_vf`) on the host: csrc/r6_ppo.cuh's ppo_value_clip after ppo_head / ppo_head_sde
(host build, tests/vfclip_hostsim) against float64 autograd of SB3's clipped loss (tests/vfclip_ref.py) inside the
band, outside it on both sides and exactly on its edges; the per-sample gradients of the shared trunk and the separate
towers; PPOConfig's validation; and the R6_EINVAL cases of r6_ppo_grad / r6_ppo_grad_sde, which need no GPU."""
import ctypes as C

import numpy as np
import pytest
import torch

import policy_ref as pr
import ppo_ref as rf
import sep_hostsim
import sep_ref
import vfclip_hostsim as hs
import vfclip_ref as vr

C_VF = 0.25


def _head_case(n, seed, sde):
    rng = np.random.default_rng(seed)
    out = rng.standard_normal((n, 4)).astype(np.float32)
    a = (out[:, :3] + rng.standard_normal((n, 3)) * 0.5).astype(np.float32)
    old = rng.normal(-2.0, 0.3, n).astype(np.float32)
    adv = rng.standard_normal(n).astype(np.float32)
    ret = (out[:, 3] + rng.standard_normal(n)).astype(np.float32)
    ls = rng.uniform(0.05, 0.5, (n, 3)).astype(np.float32) if sde else rng.uniform(-1.0, 0.2, 3).astype(np.float32)
    # d = V - V_old: inside the band, outside on both sides
    d = np.concatenate([rng.uniform(-0.8, 0.8, n // 2), rng.uniform(1.2, 3.0, n - n // 2) * rng.choice([-1, 1], n - n // 2)])
    vold = (out[:, 3].astype(np.float64) - d * C_VF).astype(np.float32)
    # exactly on the edges: V and V_old with d = +-c exact in float32
    out[:4, 3] = 1.0
    vold[:4] = [0.75, 1.25, 0.75, 1.25]
    return out, a, old, adv, ret, ls, vold


def _sb3_value_grad(V, vold, ret, c, vf_coef):
    """d (vf_coef (R - vp)^2) / d V and (R - vp)^2 by float64 autograd of SB3's clamp."""
    v = torch.tensor(np.asarray(V, np.float64), requires_grad=True)
    vo = torch.tensor(np.asarray(vold, np.float64))
    vp = vo + torch.clamp(v - vo, -c, c)
    vl = (torch.tensor(np.asarray(ret, np.float64)) - vp) ** 2
    (vf_coef * vl).sum().backward()
    return v.grad.numpy(), vl.detach().numpy()


@pytest.mark.parametrize("sde", [False, True])
def test_value_clip_head_matches_sb3(sde):
    n, vf = 512, 0.5
    out, a, old, adv, ret, ls, vold = _head_case(n, 3 + sde, sde)
    g, vl = hs.head(out, a, old, adv, ret, vold, ls, C_VF, sde=sde, vf_coef=vf)
    g64, vl64 = _sb3_value_grad(out[:, 3], vold, ret, C_VF, vf)
    d = out[:, 3].astype(np.float64) - vold
    inside = np.abs(d) <= C_VF
    assert inside[:4].all() and 0 < inside.sum() < n and (d > C_VF).any() and (d < -C_VF).any()
    # outside: exactly 0; inside and on the edges: 2 vf (vp - R) with vp = fl(V_old + fl(V - V_old)) (2 roundings) and
    # the head's subtraction and product
    assert np.all(g[~inside, 3] == 0.0)
    e = np.abs(g64[inside]) / (2 * vf)
    vp_err = 2 * rf.U * (np.abs(d) + np.abs(vold) + C_VF)
    assert np.all(np.abs(g[inside, 3] - g64[inside]) <= 2 * vf * (vp_err[inside] + 2 * rf.U * e) + 1e-30)
    vp = vold.astype(np.float64) + np.clip(d, -C_VF, C_VF)
    assert np.all(np.abs(vl - vl64) <= 2 * np.sqrt(vl64) * (vp_err + rf.U * np.abs(vp) + rf.U * np.sqrt(vl64))
                  + 2 * rf.U * vl64 + 1e-30)
    # the edges are inside (clamp's mask takes both bounds) and exact: vp = V_old +- c = 1 = V
    assert np.array_equal(g[:4, 3], np.float32(2 * vf) * (np.float32(1.0) - ret[:4]))
    # one ulp further out: zero gradient
    vold2 = vold.copy()
    vold2[:4] = np.nextafter(vold[:4], np.float32([-1, 2, -1, 2])).astype(np.float32)
    g2, _ = hs.head(out, a, old, adv, ret, vold2, ls, C_VF, sde=sde, vf_coef=vf)
    assert np.all(g2[:4, 3] == 0.0)
    # the policy outputs of the head are untouched
    assert np.array_equal(np.delete(g, 3, 1), np.delete(g2, 3, 1))


def _shared_case(n, seed):
    w = pr.weights("golden")
    x = pr.obs_sets(n, seed=seed)["golden"]
    a, old, adv, ret = rf.minibatch(w, x, seed=seed)
    v, ev = vr.value_err(w, x)
    vold = vr.old_values(v, 0.2, seed)
    return w, x, a, old, adv, ret, vold, v, ev


def test_shared_sample_grad_matches_autograd():
    n, c = 1024, 0.2
    w, x, a, old, adv, ret, vold, v, ev = _shared_case(n, 21)
    assert vr.margin(v, ev, vold, c) > 1.0
    st = rf.adv_stats(adv)
    adv_n = (adv.astype(np.float64) - st[0]) * st[1]
    g, t = hs.sample_grad(rf.flat(w), x, a, old, adv, ret, vold, c, adv_stats=st)
    ref, terms = vr.grad_sum(w, x, a, old, adv_n, ret, vold, c)
    q = vr.per_sample(w, x, a, old, adv_n, ret, vold, c)
    assert 0 < q["inside"].sum() < n
    bnd, tb = vr.bound(q, samples_per_cta=0)
    worst = (np.abs(g.astype(np.float64).sum(0) - ref) / (bnd + 1e-300)).max()
    print(f"shared trunk: worst |host - autograd| / bound = {worst:.3f}")
    assert worst <= 1.0
    assert np.all(np.abs(t.astype(np.float64).sum(0)[[0, 1, 3]] - terms[[0, 1, 3]]) <= tb[[0, 1, 3]])
    # the unclipped loss is far outside the clipped bound
    g0, _ = rf.grad_sum(rf.per_sample(w, x, a, old, adv_n, ret))
    assert (np.abs(g0 - ref) / (bnd + 1e-300)).max() > 100


def test_separate_sample_grad_matches_autograd():
    n, c = 1024, 0.2
    w = sep_ref.weights(5)
    x, a, old, adv, ret = sep_ref.minibatch(w, n, 5)
    v, ev = vr.value_err(w, x)
    vold = vr.old_values(v, c, 5)
    assert vr.margin(v, ev, vold, c) > 1.0
    st = rf.adv_stats(adv)
    adv_n = (adv.astype(np.float64) - st[0]) * st[1]
    g, t = hs.sample_grad(sep_ref.flat(w), x, a, old, adv, ret, vold, c, adv_stats=st)
    ref, terms = vr.grad_sum(w, x, a, old, adv_n, ret, vold, c)
    bnd = vr.sep_bound(w, x, a, old, adv_n, ret, vold, c, samples_per_cta=0)
    worst = (np.abs(g.astype(np.float64).sum(0) - ref) / (bnd + 1e-300)).max()
    print(f"separate towers: worst |host - autograd| / bound = {worst:.3f}")
    assert worst <= 1.0
    # a clipped sample gives its value tower nothing; the policy tower's entries are those of the unclipped head
    inside = np.abs(v - vold) <= c
    from rl_rocket_6dof_b200.ppo import LAYOUT_SEP
    off, o = {}, 0
    for k, s in LAYOUT_SEP:
        off[k] = slice(o, o + int(np.prod(s)))
        o += int(np.prod(s))
    for k in ("vf_w0", "vf_b0", "vf_w1", "vf_b1", "wv", "bv"):
        assert np.all(g[~inside][:, off[k]] == 0.0), k
    g0, _ = sep_hostsim.sample_grad(sep_ref.flat(w), x, a, old, adv, ret, adv_stats=st)
    for k in ("w0", "b0", "w1", "b1", "w2", "b2", "log_std"):
        assert np.array_equal(g[:, off[k]], g0[:, off[k]]), k
    assert np.allclose(t.astype(np.float64).sum(0)[[0, 2, 3]], terms[[0, 2, 3]], rtol=1e-4, atol=1e-3)


def test_ppoconfig_clip_options():
    from rl_rocket_6dof_b200.ppo import PPOConfig
    for bad in (0.0, -0.1, float("nan")):
        with pytest.raises(ValueError):
            PPOConfig(clip_range_vf=bad)
    assert PPOConfig().clip_range_vf is None
    sched = lambda p: 0.1 * p
    cfg = PPOConfig(clip_range=lambda p: 0.2 * p, clip_range_vf=sched)
    assert cfg.clip_range_vf is sched and cfg.clip_range(0.5) == 0.1
    assert PPOConfig(clip_range_vf=0.2).clip_range_vf == 0.2


def test_ppo_grad_rejects_bad_clip_range_vf_without_a_gpu():
    """clip_range_vf < 0 or not finite (B = 0 too), and > 0 without old_values, return R6_EINVAL before any CUDA call;
    the struct sizes match the ctypes mirrors, with the new fields last."""
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    assert L.r6_ppo_rollout_size() == C.sizeof(_lib.R6PpoRollout) and L.r6_ppo_coef_size() == C.sizeof(_lib.R6PpoCoef)
    assert _lib.R6PpoRollout.old_values.offset == C.sizeof(_lib.R6PpoRollout) - 8
    assert _lib.R6PpoCoef.clip_range_vf.offset == C.sizeof(_lib.R6PpoCoef) - 8
    buf = (C.c_float * 16)()
    p = C.addressof(buf)
    full = _lib.R6Mlp(*([p] * 9))
    ro = _lib.R6PpoRollout(p, 1, 1, 1, p, p, p, p, 1, 1)             # positional: old_values NULL
    assert ro.old_values is None
    sde = _lib.R6Sde(p, None)
    for vfc, with_old, B, what in ((-0.1, True, 1, b"clip_range_vf"), (float("nan"), True, 1, b"clip_range_vf"),
                                   (float("inf"), True, 1, b"clip_range_vf"), (0.2, False, 1, b"old_values"),
                                   (-1.0, True, 0, b"clip_range_vf")):
        coef = _lib.R6PpoCoef(0.2, 0.5, 0.0, None, vfc)
        ro.old_values = p if with_old else None
        assert L.r6_ppo_grad(C.byref(full), C.byref(ro), p, B, C.byref(coef), p, p, p, None) == -1, vfc
        assert what in L.r6_last_error()
        assert L.r6_ppo_grad_sde(C.byref(full), C.byref(sde), C.byref(ro), p, B, C.byref(coef), p, p, p, None) == -1
        assert what in L.r6_last_error()
    assert _lib.R6PpoCoef(0.2, 0.5, 0.0, None).clip_range_vf == 0.0        # positional: no clipping
