"""SB3 1.6's value clipping (`PPO(clip_range_vf=c)`) restated in float64 for the three networks of ppo.py [memory]:

    values_pred = old_values + clamp(values - old_values, -c, c);  value_loss = mse(returns, values_pred)

torch autograd of the clipped per-sample loss sum (shared trunk, separate towers, gSDE), and the first-order bounds of
tests/ppo_ref.py / tests/sep_ref.py extended by the roundings csrc/r6_ppo.cuh's ppo_value_clip adds: d = V - V_old, and
vp = V_old + clamp(d) (inside the band), and fl32(c) for a clipped sample's loss.  A clipped sample's value gradient is
exactly 0 in the kernel; its decision cannot flip when | |d| - c | exceeds the bound on V's error (value_err), which
the tests assert."""
import numpy as np
import torch

import policy_ref as pr
import ppo_ref as rf
import sde_ref
import sep_ref
from rl_rocket_6dof_b200.ppo import LAYOUT_SEP

U = rf.U


def _t(v):
    return torch.tensor(np.asarray(v, np.float32).astype(np.float64))


def value_err(w, x):
    """(V [n] float64, bound [n] on |fl32 V - V|): policy_ref's mode-0 forward bound of the value head (shared trunk or,
    with vf_w0, the value tower)."""
    W = {k: np.asarray(v, np.float32).astype(np.float64) for k, v in w.items()}
    x = np.asarray(x, np.float32).astype(np.float64).reshape(-1, 13)
    p = "vf_" if "vf_w0" in W else ""
    a0, e0 = pr._layer(0, x, np.zeros_like(x), W[p + "w0"], W[p + "b0"])
    h0, eh0 = np.tanh(a0), pr._through_tanh(a0, e0, 0)
    a1, e1 = pr._layer(0, h0, eh0, W[p + "w1"], W[p + "b1"])
    h1, eh1 = np.tanh(a1), pr._through_tanh(a1, e1, 0)
    wv = W["wv"].reshape(1, 64)
    return (h1 @ wv.T)[:, 0] + W["bv"].reshape(1)[0], pr._layer(0, h1, eh1, wv, W["bv"].reshape(1))[1][:, 0]


def old_values(v, c, seed, inside=0.5):
    """float32 V_old around the float64 values v: a fraction `inside` with |d| <= 0.8 c, the rest with 1.2 c <= |d| <= 3 c
    on both sides (d = V - V_old)."""
    rng = np.random.default_rng(seed)
    n = len(v)
    mag = np.where(rng.random(n) < inside, rng.uniform(0.0, 0.8 * c, n), rng.uniform(1.2 * c, 3.0 * c, n))
    return (np.asarray(v, np.float64) - mag * rng.choice([-1.0, 1.0], n)).astype(np.float32)


def margin(v, ev, vold, c):
    """min over the samples of | |V - V_old| - fl32(c) | / (the bound on fl32(V - V_old)'s error): > 1 means that no
    sample's in-band decision can differ between the kernel and the float64 reference."""
    d = np.asarray(v, np.float64) - np.asarray(vold, np.float32)
    cf = float(np.float32(c))
    return float(np.min(np.abs(np.abs(d) - cf) / (ev + 2 * U * (np.abs(d) + cf) + 1e-300)))


def clipped_loss(mean, values, dist, a, old, adv_n, ret, vold, clip, cvf, vf_coef, ent_coef):
    """Per-sample SB3 loss terms with value clipping (cvf None: SB3's unclipped loss); returns (loss sum, terms [4])."""
    log_prob, entropy = dist.log_prob(_t(a)).sum(1), dist.entropy().sum(1)
    A = torch.as_tensor(np.asarray(adv_n, np.float64))
    lr = log_prob - _t(old)
    ratio = torch.exp(lr)
    pg = -torch.min(A * ratio, A * torch.clamp(ratio, 1 - clip, 1 + clip))
    if cvf is None:
        vp = values
    else:
        vo = _t(vold)
        vp = vo + torch.clamp(values - vo, -cvf, cvf)
    vl = (_t(ret) - vp) ** 2
    with torch.no_grad():
        terms = np.array([float(pg.sum()), float(vl.sum()), float((torch.abs(ratio - 1) > clip).double().sum()),
                          float(((ratio - 1) - lr).sum())])
    return pg.sum() - ent_coef * entropy.sum() + vf_coef * vl.sum(), terms


def grad_sum(w, x, a, old, adv_n, ret, vold, cvf, clip=0.2, vf_coef=0.5, ent_coef=0.0, chunk=65536):
    """Float64 autograd of the clipped loss SUM (what r6_ppo_grad / r6_ppo_grad_sde return) for the network of w: the
    shared trunk (LAYOUT), the separate towers (vf_w0 present) or gSDE (log_std [64, 3]).  Returns (gradient, terms [4])."""
    sep = "vf_w0" in w
    sde = np.asarray(w["log_std"]).size == 192
    layout = LAYOUT_SEP if sep else (sde_ref.LAYOUT_SDE if sde else rf.LAYOUT)
    n = len(np.asarray(ret))
    g, terms = 0.0, 0.0
    for i in range(0, n, chunk):
        sl = slice(i, min(i + chunk, n))
        P = {k: torch.tensor(np.asarray(w[k], np.float32).astype(np.float64).reshape(s), requires_grad=True)
             for k, s in layout}
        xs = _t(np.asarray(x)[sl])
        if sep:
            hp = torch.tanh(torch.tanh(xs @ P["w0"].T + P["b0"]) @ P["w1"].T + P["b1"])
            hv = torch.tanh(torch.tanh(xs @ P["vf_w0"].T + P["vf_b0"]) @ P["vf_w1"].T + P["vf_b1"])
            mean, values = hp @ P["w2"].T + P["b2"], hv @ P["wv"] + P["bv"][0]
        else:
            h = torch.tanh(torch.tanh(xs @ P["w0"].T + P["b0"]) @ P["w1"].T + P["b1"])
            mean, values = h @ P["w2"].T + P["b2"], h @ P["wv"] + P["bv"][0]
        dist = (sde_ref.distribution(P, mean, h) if sde else
                torch.distributions.Normal(mean, torch.exp(P["log_std"]).expand_as(mean)))
        loss, tm = clipped_loss(mean, values, dist, np.asarray(a)[sl], np.asarray(old)[sl], np.asarray(adv_n)[sl],
                                np.asarray(ret)[sl], np.asarray(vold)[sl], clip, cvf, vf_coef, ent_coef)
        loss.backward()
        g = g + torch.cat([P[k].grad.reshape(-1) for k, _ in layout]).numpy()
        terms = terms + tm
    return g, terms


def _clip_parts(v, vold, ret, cvf):
    """(inside mask, d, vp, e = vp - R) in float64."""
    d = np.asarray(v, np.float64) - np.asarray(vold, np.float32)
    inside = np.abs(d) <= cvf
    vp = np.asarray(vold, np.float32) + np.clip(d, -cvf, cvf)
    return inside, d, vp, vp - np.asarray(ret, np.float32)


def per_sample(w, x, a, old, adv_n, ret, vold, cvf, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """ppo_ref.per_sample with the clipped value loss: gv = 2 vf_coef (vp - R) inside the band, 0 outside, and the
    deltas and vloss that follow (shared trunk)."""
    q = rf.per_sample(w, x, a, old, adv_n, ret, clip=clip, vf_coef=vf_coef, ent_coef=ent_coef)
    W = q["W"]
    inside, d, vp, e = _clip_parts(q["v"], vold, ret, cvf)
    gv = np.where(inside, 2 * vf_coef * e, 0.0)
    s = q["gm"] @ W["w2"] + gv[:, None] * W["wv"].reshape(1, 64)
    d1 = s * (1 - q["h1"] ** 2)
    t = d1 @ W["w1"]
    q.update(gv=gv, s=s, d1=d1, t=t, d0=t * (1 - q["h0"] ** 2), vloss=e * e, inside=inside, dv=d, vp=vp, e=e, cvf=cvf)
    return q


def _vloss_extra(q):
    """The term-bound extra of the clipped vloss over ppo_ref.bound's: d and vp inside the band, fl32(c) and vp outside."""
    return float(np.sum(2 * np.abs(q["e"]) * U * (np.where(q["inside"], np.abs(q["dv"]), q["cvf"]) + np.abs(q["vp"]))))


def bound(q, vf_coef=0.5, ent_coef=0.0, samples_per_cta=128):
    """ppo_ref.bound of the clipped per_sample q plus the two roundings of d and vp on every in-band sample's value
    gradient, carried through the trunk like ppo_ref.bound's egv (an outside sample's value gradient is exactly 0 in the
    kernel, which ppo_ref.bound covers with room to spare)."""
    bnd, tb = rf.bound(q, vf_coef=vf_coef, ent_coef=ent_coef, samples_per_cta=samples_per_cta)
    W = q["W"]
    eg = np.where(q["inside"], 2 * abs(vf_coef) * U * (np.abs(q["dv"]) + np.abs(q["vp"])), 0.0)
    ed1 = eg[:, None] * np.abs(W["wv"]).reshape(1, 64) * (1 - q["h1"] ** 2)
    ed0 = (ed1 @ np.abs(W["w1"])) * (1 - q["h0"] ** 2)
    z3 = np.zeros(3)
    bnd = bnd + rf._pack(ed0.T @ np.abs(q["x"]), ed0.sum(0), ed1.T @ np.abs(q["h0"]), ed1.sum(0), np.zeros((3, 64)), z3,
                         eg @ np.abs(q["h1"]), eg.sum(), z3)
    tb = tb.copy()
    tb[1] += _vloss_extra(q)
    return bnd, tb


def sep_bound(w, x, a, old, adv_n, ret, vold, cvf, clip=0.2, vf_coef=0.5, ent_coef=0.0, samples_per_cta=128):
    """sep_ref.bound of the unclipped loss (every value-tower term of it grows with |V - R| and its error, and the
    clipped sample's exact 0 has none, so it covers the clipped loss's) plus the roundings of d and vp on the in-band
    samples, through the value tower."""
    bnd = sep_ref.bound(w, x, a, old, adv_n, ret, clip=clip, vf_coef=vf_coef, ent_coef=ent_coef,
                        samples_per_cta=samples_per_cta)
    W = {k: np.asarray(v, np.float32).astype(np.float64) for k, v in w.items()}
    xs = np.asarray(x, np.float32).astype(np.float64)
    h0v = np.tanh(xs @ W["vf_w0"].T + W["vf_b0"])
    h1v = np.tanh(h0v @ W["vf_w1"].T + W["vf_b1"])
    v = h1v @ W["wv"].reshape(64) + W["bv"].reshape(1)[0]
    inside, d, vp, _ = _clip_parts(v, vold, ret, cvf)
    eg = np.where(inside, 2 * abs(vf_coef) * U * (np.abs(d) + np.abs(vp)), 0.0)
    ed1 = eg[:, None] * np.abs(W["wv"]).reshape(1, 64) * (1 - h1v ** 2)
    ed0 = (ed1 @ np.abs(W["vf_w1"])) * (1 - h0v ** 2)
    extra = {k: np.zeros(int(np.prod(s))) for k, s in LAYOUT_SEP}
    extra.update(vf_w0=ed0.T @ np.abs(xs), vf_b0=ed0.sum(0), vf_w1=ed1.T @ np.abs(h0v), vf_b1=ed1.sum(0),
                 wv=eg @ np.abs(h1v), bv=np.array([eg.sum()]))
    return bnd + np.concatenate([np.asarray(extra[k]).reshape(-1) for k, _ in LAYOUT_SEP])


def reference_step(params, m, v, step, rollout, idx, lr, cfg, cvf):
    """ppo_train_ref.reference_step with SB3's clipped value loss at clip_range_vf = cvf and clip_range = cfg's float:
    one minibatch from the float32 pre-step state (shared trunk or separate towers, by the size of params), the mean
    loss's gradient, clip_grad_norm_, Adam(eps=1e-5) step `step` in float64, and ppo_train_ref.step_bound of this
    module's gradient bound.  rollout: host arrays obs [n, 13], actions [n, 3], log_probs / advantages / returns /
    values [n].  Returns dict(p, bound, logs (shared trunk: with log_bounds))."""
    import ppo_train_ref as tr
    sep = len(params) == sep_ref.flat(sep_ref.weights(0)).size
    layout = LAYOUT_SEP if sep else rf.LAYOUT
    w, o = {}, 0
    for k, s in layout:
        w[k] = np.asarray(params[o:o + int(np.prod(s))], np.float32).reshape(s)
        o += int(np.prod(s))
    B = len(idx)
    x, a = rollout["obs"][idx], rollout["actions"][idx]
    old, ret, vold = rollout["log_probs"][idx], rollout["returns"][idx], rollout["values"][idx]
    adv_n = tr.normalized_advantages(rollout["advantages"][idx], cfg.normalize_advantage)
    clip = float(cfg.clip_range)
    g_sum, terms = grad_sum(w, x, a, old, adv_n, ret, vold, cvf, clip=clip, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef)
    spc = rf.samples_per_cta(B)
    out = {}
    if sep:
        bnd = sep_bound(w, x, a, old, adv_n, ret, vold, cvf, clip=clip, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef,
                        samples_per_cta=spc)
    else:
        q = per_sample(w, x, a, old, adv_n, ret, vold, cvf, clip=clip, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef)
        bnd, tb = bound(q, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef, samples_per_cta=spc)
        ent = float(np.sum(np.asarray(w["log_std"], np.float64)) + 3 * rf.LOG_SQRT_2PI + 1.5)
        logs = dict(pg=terms[0] / B, value_loss=terms[1] / B, clip_fraction=terms[2] / B, approx_kl=terms[3] / B,
                    entropy_loss=-ent)
        logs["loss"] = logs["pg"] + cfg.ent_coef * logs["entropy_loss"] + cfg.vf_coef * logs["value_loss"]
        lb = dict(pg=tb[0] / B, value_loss=tb[1] / B, clip_fraction=1e-15, approx_kl=tb[3] / B, entropy_loss=1e-13)
        lb["loss"] = lb["pg"] + cfg.vf_coef * lb["value_loss"] + abs(cfg.ent_coef) * lb["entropy_loss"]
        out.update(logs=logs, log_bounds=lb)
    s = 1.0 / B
    g = g_sum * s
    plist, o = [], 0
    for k, sh in layout:
        nk = int(np.prod(sh))
        t = torch.tensor(np.asarray(params[o:o + nk], np.float32).astype(np.float64), requires_grad=True)
        t.grad = torch.tensor(g[o:o + nk].copy())
        plist.append(t)
        o += nk
    norm = float(torch.nn.utils.clip_grad_norm_(plist, cfg.max_grad_norm))
    opt = torch.optim.Adam(plist, lr=lr, betas=tr.BETAS, eps=tr.EPS, foreach=False)
    o = 0
    for t in plist:
        nk = t.numel()
        opt.state[t] = {"step": torch.tensor(float(step - 1)),
                        "exp_avg": torch.tensor(np.asarray(m[o:o + nk], np.float32).astype(np.float64)),
                        "exp_avg_sq": torch.tensor(np.asarray(v[o:o + nk], np.float32).astype(np.float64))}
        o += nk
    opt.step()
    cat = lambda f: torch.cat([f(t).reshape(-1) for t in plist]).detach().numpy().copy()
    gc, pp = cat(lambda t: t.grad), cat(lambda t: t)
    mp, vp = cat(lambda t: opt.state[t]["exp_avg"]), cat(lambda t: opt.state[t]["exp_avg_sq"])
    out.update(p=pp, norm=norm, bound=tr.step_bound(g, s * bnd, norm, cfg.max_grad_norm, gc, np.asarray(m, np.float64),
                                                    mp, vp, pp, lr, step))
    return out
