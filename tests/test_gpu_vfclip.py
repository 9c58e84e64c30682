"""SB3's value clipping (`clip_range_vf`) and clip-range schedules on the B200: r6_ppo_grad (shared trunk, separate
towers) and r6_ppo_grad_sde against float64 references with their first-order bounds extended by the value clip's
roundings (tests/vfclip_ref.py), an exact edge case, bit-identity with clipping off, PPOTrainer.train one Adam step at a
time against a float64 restatement of SB3's clipped PPO.train, and a scheduled learn."""
import ctypes as C

import numpy as np
import pytest
import torch

import policy_ref as pr
import ppo_ref as rf
import ppo_train_ref as tr
import sep_ref
import vfclip_ref as vr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CVF = 0.2
T, N = 32, 8400                      # 268,800 samples: room for B = 2^18 + 129 without replacement


def _weights(kind, seed):
    if kind == "sep":
        return sep_ref.weights(seed)
    w = dict(pr.weights("golden"))
    if kind == "sde":
        rng = np.random.default_rng(seed)
        w["log_std"] = rng.uniform(-1.0, 0.5, (64, 3)).astype(np.float32)
    return w


_ROLL = {}


def _rollout(kind, seed=7):
    """A real collect_rollout (strided obs view, mode 0) with the weights of `kind`, its `values` replaced by old values
    placed around the float64 critic so that half the samples lie inside the band and half outside on both sides, at
    least 0.2 c from its edges.  Cached per kind."""
    if kind not in _ROLL:
        from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
        from rl_rocket_6dof_b200.ppo import ActorCriticParams
        w = _weights(kind, seed)
        p = ActorCriticParams.from_weights(w, DEV)
        env = Rocket6DOFBatch(N, device=DEV, seed=seed)
        env.reset()
        ro = env.collect_rollout(T, p.mlp(), tensor_cores=0)
        assert ro["obs"].stride(2) != 1
        host = {k: ro[k].contiguous().cpu().numpy().reshape(T * N, -1) for k in ("obs", "actions")}
        host.update({k: ro[k].cpu().numpy().reshape(-1) for k in ("log_probs", "advantages", "returns")})
        v, ev = vr.value_err(w, host["obs"])
        host["values"] = vr.old_values(v, CVF, seed)
        host["v"], host["ev"] = v, ev
        ro["values"] = torch.from_numpy(host["values"].reshape(T, N)).to(DEV)
        _ROLL[kind] = (w, p, ro, host)
    return _ROLL[kind]


def _reference(kind, w, host, idx, normalize, spc, chunk=1 << 15):
    """(gradient sum, term sums [4], bound or None, term bound or None) of the clipped loss over idx, in chunks."""
    adv = host["advantages"][idx]
    st = rf.adv_stats(adv) if normalize else np.array([0.0, 1.0])
    g64, t64, bnd, tb = 0.0, 0.0, 0.0, 0.0
    for s in range(0, len(idx), chunk):
        j = idx[s:s + chunk]
        args = (w, host["obs"][j], host["actions"][j], host["log_probs"][j],
                (host["advantages"][j].astype(np.float64) - st[0]) * st[1], host["returns"][j], host["values"][j], CVF)
        if kind == "shared":
            q = vr.per_sample(*args)
            g_c, t_c = rf.grad_sum(q)
            b_c, tb_c = vr.bound(q, samples_per_cta=spc)
            tb = tb + tb_c
        else:
            g_c, t_c = vr.grad_sum(*args)
            b_c = vr.sep_bound(*args, samples_per_cta=spc) if kind == "sep" else 0.0
        g64, t64, bnd = g64 + g_c, t64 + t_c, bnd + b_c
    return g64, t64, (None if kind == "sde" else bnd), (tb if kind == "shared" else None)


@pytest.mark.parametrize("kind", ["shared", "sep", "sde"])
@pytest.mark.parametrize("B", [1, 127, 128, 129, 2 ** 18 + 129])
def test_clipped_grad_within_bound(kind, B):
    from rl_rocket_6dof_b200 import ppo
    w, p, ro, host = _rollout(kind)
    idx = np.random.default_rng(B).choice(T * N, B, replace=False)
    assert vr.margin(host["v"][idx], host["ev"][idx], host["values"][idx], CVF) > 1.0    # no decision can flip
    inside = np.abs(host["v"][idx] - host["values"][idx]) <= CVF
    assert B == 1 or 0 < inside.sum() < B
    g, terms = ppo.loss_and_grad(p, ro, torch.from_numpy(idx).to(DEV), clip_range_vf=CVF, normalize_advantage=B > 1)
    g, terms = g.cpu().numpy().astype(np.float64), terms.cpu().numpy()
    g64, t64, bnd, tb = _reference(kind, w, host, idx, B > 1, rf.samples_per_cta(B))
    assert terms[2] == t64[2] and terms[4] == 0
    if kind == "sde":
        # tests/test_gpu_sde.py's criterion for r6_ppo_grad_sde: 1e-4 of the gradient scale, 1e-3 of the log_std block
        err, scale = np.abs(g - g64), np.abs(g64).max() + 1e-6
        print(f"gSDE B {B}: worst |kernel - ref| / max|grad| {err.max() / scale:.2e}")
        assert err.max() <= 1e-4 * scale
        assert err[10308:].max() <= 1e-3 * np.abs(g64[10308:]).max()
        assert abs(terms[1] - t64[1]) <= 1e-5 * abs(t64[1]) + 1e-6
        return
    r = np.abs(g - g64) / bnd
    print(f"{kind} B {B}: max |kernel - ref| / bound {r.max():.3g}")
    assert np.all(r <= rf.C_BAR), (kind, B, float(r.max()), int(r.argmax()))
    if tb is not None:
        assert np.all(np.abs(terms[[0, 1, 3]] - t64[[0, 1, 3]]) <= rf.C_BAR * tb[[0, 1, 3]])


def _edge_params(kind):
    from rl_rocket_6dof_b200.ppo import ActorCriticParams
    w = dict(_weights(kind, 3))
    w["wv"] = np.zeros_like(w["wv"])
    w["bv"] = np.ones_like(w["bv"])                    # V = bv = 1 exactly
    return ActorCriticParams.from_weights(w, DEV)


@pytest.mark.parametrize("kind", ["shared", "sep", "sde"])
def test_band_edges_are_exact(kind):
    """wv = 0 makes V = bv = 1 exactly.  c = 0.25, V_old = 0.75 and 1.25: d = +-c, inside (clamp's mask takes both
    bounds), vp = V_old +- c = 1 exactly, and the one-sample dbv is 2 vf_coef (vp - R) bit for bit.  One ulp further
    out, dbv and dwv are exactly 0."""
    from rl_rocket_6dof_b200 import ppo
    p = _edge_params(kind)
    o = dict(shared=10243, sep=10307, sde=10243)[kind]           # wv, then bv
    R = np.float32(0.3125)
    for vold in (0.75, 1.25):
        for out in (False, True):
            vo = np.float32(vold)
            if out:
                vo = np.nextafter(vo, np.float32(-1.0 if vold < 1 else 2.0))
            ro = {k: torch.zeros(1, 1, s, device=DEV) for k, s in (("obs", 13), ("actions", 3))}
            ro.update({k: torch.zeros(1, 1, device=DEV) for k in ("log_probs", "advantages")})
            ro["returns"] = torch.full((1, 1), float(R), device=DEV)
            ro["values"] = torch.full((1, 1), float(vo), device=DEV)
            g, terms = ppo.loss_and_grad(p, ro, torch.zeros(1, dtype=torch.int64, device=DEV), clip_range_vf=0.25)
            g = g.cpu().numpy()
            if out:
                assert g[o + 64] == 0.0 and np.all(g[o:o + 64] == 0.0), (kind, vold)
            else:
                want = np.float32(np.float32(2.0) * np.float32(0.5)) * (np.float32(1.0) - R)
                assert g[o + 64] == want, (kind, vold, g[o + 64], want)
                assert float(terms[1]) == float((np.float32(1.0) - R) ** 2)


def _abi_call(p, ro, idx, clip_vf, old_values):
    """r6_ppo_grad / r6_ppo_grad_sde through the C ABI with R6PpoRollout.old_values and R6PpoCoef.clip_range_vf set as
    given (raw advantages)."""
    from rl_rocket_6dof_b200 import _lib
    L = _lib.load()
    obs = ro["obs"]
    r = _lib.R6PpoRollout(obs.data_ptr(), obs.stride(0), obs.stride(2), obs.stride(1), ro["actions"].data_ptr(),
                          ro["log_probs"].data_ptr(), ro["advantages"].data_ptr(), ro["returns"].data_ptr(), T, N,
                          None if old_values is None else old_values.data_ptr())
    coef = _lib.R6PpoCoef(0.2, 0.5, 0.01, None, clip_vf)
    B = idx.numel()
    nt = _lib.PPO_NTERMS_SDE if p.use_sde else _lib.PPO_NTERMS
    g = torch.full((p.flat.numel(),), float("nan"), device=DEV)
    t = torch.full((nt,), float("nan"), dtype=torch.float64, device=DEV)
    work = torch.empty(int(L.r6_ppo_sde_work_bytes(B) if p.use_sde else L.r6_ppo_work_bytes(B)), dtype=torch.uint8, device=DEV)
    m = _lib.make_mlp(p.mlp())
    s = torch.cuda.current_stream(DEV).cuda_stream
    if p.use_sde:
        sde = _lib.R6Sde(p.log_std.data_ptr(), None)
        rc = L.r6_ppo_grad_sde(C.byref(m), C.byref(sde), C.byref(r), idx.data_ptr(), B, C.byref(coef), g.data_ptr(),
                               t.data_ptr(), work.data_ptr(), s)
    else:
        rc = L.r6_ppo_grad(C.byref(m), C.byref(r), idx.data_ptr(), B, C.byref(coef), g.data_ptr(), t.data_ptr(),
                           work.data_ptr(), s)
    _lib.check(rc, L)
    return g, t


@pytest.mark.parametrize("kind", ["shared", "sep", "sde"])
def test_clipping_off_is_bit_identical(kind):
    """old_values set with clip_range_vf = 0, old_values absent, and loss_and_grad without clip_range_vf: the same bits."""
    from rl_rocket_6dof_b200 import ppo
    _, p, ro, _ = _rollout(kind)
    idx = torch.randperm(T * N, generator=torch.Generator(device=DEV).manual_seed(2), device=DEV)[:70001]
    g0, t0 = _abi_call(p, ro, idx, 0.0, None)
    g1, t1 = _abi_call(p, ro, idx, 0.0, ro["values"])
    g2, t2 = ppo.loss_and_grad(p, ro, idx, ent_coef=0.01, normalize_advantage=False)
    assert torch.equal(g0, g1) and torch.equal(t0, t1) and torch.equal(g0, g2) and torch.equal(t0, t2)
    g3, t3 = _abi_call(p, ro, idx, CVF, ro["values"])
    assert not torch.equal(g0, g3) and float(t3[1]) != float(t0[1])


def test_bounds_have_teeth():
    """On a minibatch with clipped samples, the clipping kernel fails the unclipped reference's bound and the unclipped
    kernel fails the clipped reference's."""
    from rl_rocket_6dof_b200 import ppo
    w, p, ro, host = _rollout("shared")
    B = 256
    idx = np.random.default_rng(5).choice(T * N, B, replace=False)
    it = torch.from_numpy(idx).to(DEV)
    g_clip = ppo.loss_and_grad(p, ro, it, clip_range_vf=CVF)[0].cpu().numpy().astype(np.float64)
    g_off = ppo.loss_and_grad(p, ro, it)[0].cpu().numpy().astype(np.float64)
    g64, _, bnd, _ = _reference("shared", w, host, idx, True, rf.samples_per_cta(B))
    st = rf.adv_stats(host["advantages"][idx])
    q0 = rf.per_sample(w, host["obs"][idx], host["actions"][idx], host["log_probs"][idx],
                       (host["advantages"][idx].astype(np.float64) - st[0]) * st[1], host["returns"][idx])
    g0, _ = rf.grad_sum(q0)
    b0, _ = rf.bound(q0, samples_per_cta=rf.samples_per_cta(B))
    assert np.all(np.abs(g_clip - g64) <= rf.C_BAR * bnd) and np.all(np.abs(g_off - g0) <= rf.C_BAR * b0)
    r1, r2 = (np.abs(g_clip - g0) / b0).max(), (np.abs(g_off - g64) / bnd).max()
    print(f"clipping kernel vs unclipped reference {r1:.3g} x bound; unclipped kernel vs clipped reference {r2:.3g} x bound")
    assert r1 > rf.C_BAR and r2 > rf.C_BAR


def _capture(mp):
    from rl_rocket_6dof_b200 import ppo
    mbs = []
    real_lg, real_adam = ppo.loss_and_grad, ppo.adam_step

    def loss_and_grad(params, rollout, idx, **kw):
        mbs.append(dict(idx=idx.cpu().numpy(), params=params.flat.cpu().numpy(),
                        kw={k: v for k, v in kw.items() if k not in ("grad_sum", "terms", "work")}))
        return real_lg(params, rollout, idx, **kw)

    def adam_step(params, grad_sum, m, v, **kw):
        rec = dict(params=params.cpu().numpy(), m=m.cpu().numpy(), v=v.cpu().numpy(), **kw)
        real_adam(params, grad_sum, m, v, **kw)
        rec["post"] = params.cpu().numpy()
        mbs[-1]["adam"] = rec

    mp.setattr(ppo, "loss_and_grad", loss_and_grad)
    mp.setattr(ppo, "adam_step", adam_step)
    return mbs


@pytest.mark.parametrize("kind,n_epochs", [("shared", 2), ("sep", 1)])
def test_trainer_steps_match_clipped_sb3(kind, n_epochs):
    """PPOTrainer.train(clip_range_vf = 0.2) on a 2048-env x 16-step rollout whose values straddle the band, in
    minibatches of 10,000 (three full, one of 2,768): every Adam step from the kernels' own pre-step state within
    ppo_train_ref.step_bound of the clipped gradient's bound, and (shared trunk) the train/ logs, value_loss clipped.
    learning_rate 1e-5 keeps the critic's drift over the run (about 0.04 per step at 3e-4) inside the 0.2 c gap the old
    values leave around the band's edges, so that no sample's in-band decision is within V's error bound of flipping."""
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    n_envs, steps, bs = 2048, 16, 10000
    w = _weights(kind, 11) if kind == "sep" else pr.weights("sb3_init")
    p = ActorCriticParams.from_weights(w, DEV)
    env = Rocket6DOFBatch(n_envs, device=DEV, seed=11)
    env.reset()
    env.reset_stats()
    ro = env.collect_rollout(steps, p.mlp())
    host = {k: ro[k].contiguous().cpu().numpy().reshape(steps * n_envs, -1) for k in ("obs", "actions")}
    host.update({k: ro[k].cpu().numpy().reshape(-1) for k in ("log_probs", "advantages", "returns")})
    v, _ = vr.value_err(w, host["obs"])
    host["values"] = vr.old_values(v, CVF, 11)
    ro["values"] = torch.from_numpy(host["values"].reshape(steps, n_envs)).to(DEV)
    cfg = PPOConfig(n_steps=steps, batch_size=bs, n_epochs=n_epochs, clip_range_vf=CVF, learning_rate=1e-5)
    trainer = PPOTrainer(env, p, cfg, seed=11)
    with pytest.MonkeyPatch.context() as mp:
        mbs = _capture(mp)
        log = trainer.train(ro)
    assert len(mbs) == 4 * n_epochs
    refs, worst = [], 0.0
    for k, e in enumerate(mbs):
        a = e["adam"]
        assert e["kw"] == dict(clip_range=0.2, vf_coef=0.5, ent_coef=0.0, normalize_advantage=True, clip_range_vf=CVF)
        vk, evk = vr.value_err(_unflat(kind, a["params"]), host["obs"][e["idx"]])
        assert vr.margin(vk, evk, host["values"][e["idx"]], CVF) > 1.0
        ref = vr.reference_step(a["params"], a["m"], a["v"], a["step"], host, e["idx"], a["lr"], cfg, CVF)
        r = np.abs(a["post"].astype(np.float64) - ref["p"]) / ref["bound"]
        print(f"{kind} step {k + 1}: max |kernel - ref| / bound {r.max():.3g}")
        assert np.all(r <= rf.C_BAR), (k, float(r.max()), int(r.argmax()))
        worst = max(worst, float(r.max()))
        refs.append(ref)
    assert log["train/clip_range_vf"] == CVF and log["train/clip_range"] == 0.2
    if kind == "shared":
        per_epoch = [refs[i:i + 4] for i in range(0, len(refs), 4)]
        want = tr.sb3_logs([[r["logs"] for r in ep] for ep in per_epoch], p.log_std.cpu().numpy(), host["values"],
                           host["returns"], n_epochs, cfg.learning_rate, 0.2)
        want["train/clip_range_vf"] = CVF
        bounds = tr.sb3_log_bounds([[r["log_bounds"] for r in ep] for ep in per_epoch])
        assert set(log) == set(want), set(log) ^ set(want)
        for key, b in bounds.items():
            assert abs(log[key] - want[key]) <= rf.C_BAR * b, (key, log[key], want[key], b)
        # the logged value loss is the clipped one: the unclipped mean differs by far more than its bound
        unclipped = np.mean([np.mean((host["returns"][e["idx"]] - vr.value_err(_unflat(kind, e["params"]),
                                                                               host["obs"][e["idx"]])[0]) ** 2)
                             for e in mbs])
        assert abs(unclipped - log["train/value_loss"]) > 100 * bounds["train/value_loss"]


def _unflat(kind, flat):
    from rl_rocket_6dof_b200.ppo import LAYOUT, LAYOUT_SEP
    out, o = {}, 0
    for k, s in (LAYOUT_SEP if kind == "sep" else LAYOUT):
        out[k] = np.asarray(flat[o:o + int(np.prod(s))], np.float32).reshape(s)
        o += int(np.prod(s))
    return out


def _learn(seed):
    from rl_rocket_6dof_b200.batch import Rocket6DOFBatch
    from rl_rocket_6dof_b200.ppo import ActorCriticParams, PPOConfig, PPOTrainer
    n_envs, steps = 2048, 16
    env = Rocket6DOFBatch(n_envs, device=DEV, seed=seed)
    params = ActorCriticParams.sb3_init(seed, DEV)
    cfg = PPOConfig(n_steps=steps, n_epochs=1, clip_range=lambda q: 0.2 * q, clip_range_vf=lambda q: 0.1 * q)
    trainer = PPOTrainer(env, params, cfg, seed=seed)
    logs = []
    with pytest.MonkeyPatch.context() as mp:
        mbs = _capture(mp)
        # four iterations' worth: updates 1..3 at progress 0.75, 0.5, 0.25; the fourth, at 0, would clip the value to
        # V_old +- 0, which the trainer refuses before launching anything
        with pytest.raises(ValueError, match="clip_range_vf"):
            trainer.learn(4 * steps * n_envs, callback=logs.append)
    return logs, mbs, params.flat.cpu().numpy(), steps, n_envs


def test_learn_clip_schedules():
    """clip_range = 0.2 p and clip_range_vf = 0.1 p: each update uses both at SB3's progress_remaining, logs them, the
    update at progress 0 raises before any launch, and two runs with one seed are bitwise equal."""
    logs, mbs, final, steps, n_envs = _learn(8)
    total = 4 * steps * n_envs
    assert len(logs) == 3 and len(mbs) == 3 * 4
    for i, log in enumerate(logs, 1):
        q = tr.sb3_progress(i, steps, n_envs, total)
        assert log["train/clip_range"] == 0.2 * q and log["train/clip_range_vf"] == 0.1 * q, (i, log)
        for e in mbs[4 * (i - 1):4 * i]:
            assert e["kw"]["clip_range"] == 0.2 * q and e["kw"]["clip_range_vf"] == 0.1 * q
    logs2, mbs2, final2, *_ = _learn(8)
    same = lambda a, b: a == b or (a != a and b != b)                    # NaN statistics of unfinished episodes
    assert np.array_equal(final, final2) and all(same(a[k], b[k]) for a, b in zip(logs, logs2) for k in a)
    assert all(np.array_equal(a["adam"]["post"], b["adam"]["post"]) for a, b in zip(mbs, mbs2))
