"""SB3 1.6's `PPO.train` / `PPO.learn` restated in torch float64 on the CPU for the network of ppo.py (no gSDE, no
clip_range_vf, a constant clip_range), one Adam step at a time from the kernels' own float32 pre-step state, and a
first-order per-entry bound on the float32 step `r6_ppo_grad` + `r6_adam_step` take.  SB3 is not in the image: the
statements follow its source from memory [memory], as csrc/r6_ppo.cuh does.

The gradient of the loss below is pinned to `ppo_ref.grad_sum` (tests/test_ppo_host.py); its error bound is
`ppo_ref.bound`, so there is one float64 statement of the gradient and one of its error."""
import numpy as np
import torch
import torch.nn.functional as F

import ppo_ref as rf

U = rf.U
BETAS, EPS = (0.9, 0.999), 1e-5        # torch.optim.Adam's betas, SB3's eps
LOG_KEYS = ("pg", "value_loss", "clip_fraction", "approx_kl", "entropy_loss", "loss")


def unflat(p):
    """{name: float32 array} of a flat [NPARAMS] vector (LAYOUT order)."""
    out, o = {}, 0
    for k, s in rf.LAYOUT:
        n = int(np.prod(s))
        out[k] = np.asarray(p[o:o + n], np.float32).reshape(s)
        o += n
    return out


def normalized_advantages(adv, normalize):
    """A' in float64 as loss_and_grad forms it: SB3's per-minibatch (A - mean) / (std + 1e-8) with torch's unbiased std;
    raw A without normalisation or for a single sample (its std is undefined)."""
    a = np.asarray(adv, np.float32).astype(np.float64)
    if not normalize or len(a) < 2:
        return a
    st = rf.adv_stats(a)
    return (a - st[0]) * st[1]


def sb3_loss(P, x, a, old, adv_n, ret, clip, vf_coef, ent_coef):
    """The minibatch loss of SB3 1.6 PPO.train as it writes it, on float64 parameter tensors P (LAYOUT names); returns
    (loss, {LOG_KEYS: 0-d tensors})."""
    t = lambda v: torch.tensor(np.asarray(v, np.float32).astype(np.float64))
    h = torch.tanh(torch.tanh(t(x) @ P["w0"].T + P["b0"]) @ P["w1"].T + P["b1"])
    mean, values = h @ P["w2"].T + P["b2"], h @ P["wv"].reshape(64) + P["bv"][0]
    dist = torch.distributions.Normal(mean, torch.exp(P["log_std"]))
    log_prob, entropy = dist.log_prob(t(a)).sum(1), dist.entropy().sum(1)
    A = torch.as_tensor(np.asarray(adv_n, np.float64))
    ratio = torch.exp(log_prob - t(old))
    policy_loss = -torch.min(A * ratio, A * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    clip_fraction = torch.mean((torch.abs(ratio - 1) > clip).double())
    value_loss = F.mse_loss(t(ret), values)
    entropy_loss = -torch.mean(entropy)
    loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
    with torch.no_grad():
        log_ratio = log_prob - t(old)
        approx_kl = torch.mean((torch.exp(log_ratio) - 1) - log_ratio)
    return loss, dict(pg=policy_loss, value_loss=value_loss, clip_fraction=clip_fraction, approx_kl=approx_kl,
                      entropy_loss=entropy_loss, loss=loss)


def reference_step(params, m, v, step, rollout, idx, lr, cfg, scale=None):
    """One minibatch of SB3 1.6 PPO.train from the float32 pre-step state params / m / v [NPARAMS] (loaded into
    torch.optim.Adam as float64): loss, loss.backward(), clip_grad_norm_(max_grad_norm), Adam(eps=1e-5) step number
    `step`.  rollout: host arrays obs [n, 13], actions [n, 3], log_probs / advantages / returns [n]; idx: the minibatch.
    m = v = None stops after the loss (the minibatch target_kl breaks at takes no step).  scale replaces the mean's
    1 / len(idx) on the summed gradient (the teeth tests use it to state a wrong step).

    Returns dict(logs={LOG_KEYS}, log_bounds={LOG_KEYS}: bounds on the kernel's float64 means of float32 per-sample
    terms, and when stepping p (post-step params float64), bound [NPARAMS] on |r6_adam_step - p|, grad (the scaled
    pre-clip gradient), norm (its norm), clip (clip_grad_norm_'s factor))."""
    B = len(idx)
    w = unflat(params)
    x, a = rollout["obs"][idx], rollout["actions"][idx]
    old, ret = rollout["log_probs"][idx], rollout["returns"][idx]
    adv_n = normalized_advantages(rollout["advantages"][idx], cfg.normalize_advantage)
    P = {k: torch.tensor(w[k].astype(np.float64), requires_grad=True) for k, _ in rf.LAYOUT}
    loss, logs = sb3_loss(P, x, a, old, adv_n, ret, cfg.clip_range, cfg.vf_coef, cfg.ent_coef)
    q = rf.per_sample(w, x, a, old, adv_n, ret, clip=cfg.clip_range, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef)
    bnd, tb = rf.bound(q, vf_coef=cfg.vf_coef, ent_coef=cfg.ent_coef, samples_per_cta=rf.samples_per_cta(B))
    # the logged terms are float64 sums of float32 per-sample terms over B (ppo_ref.bound's term bounds); the clipped
    # count is exact, and the entropy is the float32 log_std summed in float64 (round-off of float64 only)
    lb = dict(pg=tb[0] / B, value_loss=tb[1] / B, clip_fraction=1e-15, approx_kl=tb[3] / B, entropy_loss=1e-13)
    lb["loss"] = lb["pg"] + cfg.vf_coef * lb["value_loss"] + abs(cfg.ent_coef) * lb["entropy_loss"]
    out = dict(logs={k: float(v.detach()) for k, v in logs.items()}, log_bounds=lb)
    if m is None:
        return out
    loss.backward()
    plist = [P[k] for k, _ in rf.LAYOUT]
    s = 1.0 / B if scale is None else float(scale)
    if scale is not None:
        for t in plist:
            t.grad *= s * B
    g = torch.cat([t.grad.reshape(-1) for t in plist]).numpy().copy()           # pre-clip, scaled
    norm = float(torch.nn.utils.clip_grad_norm_(plist, cfg.max_grad_norm))
    opt = torch.optim.Adam(plist, lr=lr, betas=BETAS, eps=EPS, foreach=False)
    mm, vv = unflat(m), unflat(v)
    for (k, _), t in zip(rf.LAYOUT, plist):
        opt.state[t] = {"step": torch.tensor(float(step - 1)),
                        "exp_avg": torch.tensor(mm[k].astype(np.float64)),
                        "exp_avg_sq": torch.tensor(vv[k].astype(np.float64))}
    opt.step()
    cat = lambda f: torch.cat([f(t).reshape(-1) for t in plist]).detach().numpy().copy()
    gc = cat(lambda t: t.grad)
    pp = cat(lambda t: t)
    mp = cat(lambda t: opt.state[t]["exp_avg"])
    vp = cat(lambda t: opt.state[t]["exp_avg_sq"])
    c = min(1.0, cfg.max_grad_norm / (norm + 1e-6))
    out.update(p=pp, grad=g, norm=norm, clip=c,
               bound=step_bound(g, s * bnd, norm, cfg.max_grad_norm, gc, np.asarray(m, np.float64), mp, vp, pp, lr, step))
    return out


def step_bound(g, e_sum, norm, max_norm, gc, m, mp, vp, pp, lr, step):
    """Per-entry first-order bound on |r6_adam_step - reference| for one step from the same float32 pre-step state,
    counted from adam_kernel / adam_element (csrc/r6_kernels.cu, csrc/r6_ppo.cuh).  g: the reference's scaled
    pre-clip gradient, e_sum: scale * ppo_ref.bound (the kernel's gradient sum, scaled), gc = c g, m the pre-step first
    moment, mp / vp / pp the reference's post-step moments and parameters."""
    b1, b2 = BETAS
    ag = np.abs(g)
    # g = fl(fl(1 / B) * grad_sum): the kernel's sum error scaled, fl(1 / B) and the product one rounding each
    e_g = e_sum + 2 * U * ag
    # c = fl32(max / (||g|| + 1e-6)) (float64 norm of the float32 g): relative error <= ||e_g||_2 / ||g|| + the
    # rounding to float32; c = 1 exactly (fminf) when the norm stays below max_norm by more than that
    rel = float(np.linalg.norm(e_g)) / max(norm, 1e-300)
    cdot = max_norm / (norm + 1e-6) if max_norm > 0 else np.inf
    c = min(1.0, cdot)
    e_c = 0.0 if cdot * (1 - rel) >= 1 else c * (rel + U)
    # g_c = fl(g * c): one rounding
    e_gc = c * e_g + ag * e_c + U * np.abs(gc)
    # m' = fma(fl(1 - b1), fl(g - m), m): the subtraction, fl(1 - b1) and the fma one rounding each
    e_m = (1 - b1) * e_gc + 2 * U * (1 - b1) * np.abs(gc - m) + U * np.abs(mp)
    # v' = fma(fl(1 - b2), fl(g g), fl(v fl(b2))): g g, fl(1 - b2), fl(b2), v fl(b2) and the fma, each <= u of a part
    # of v' = (1 - b2) g^2 + b2 v  ->  3 u v'
    e_v = 2 * (1 - b2) * np.abs(gc) * e_gc + 3 * U * vp
    bc1, sb2 = 1 - b1 ** step, np.sqrt(1 - b2 ** step)
    sv = np.sqrt(vp)
    D = sv / sb2 + EPS
    # sqrt is 1/2-Hoelder at 0: |sqrt(v' + e) - sqrt(v')| <= min(e / (2 sqrt v'), sqrt e), so a parameter whose gradient
    # vanishes (v' ~ 0) keeps a finite bound; eps bounds D below
    with np.errstate(divide="ignore", invalid="ignore"):
        e_sqrt = np.minimum(np.where(sv > 0, e_v / (2 * sv), np.inf), np.sqrt(e_v))
    # denom = fl(fl(f32_sqrt(v') / fl(sqrt(bc2))) + fl(eps)): sqrt, fl(sqrt(bc2)), the division (3u of sqrt(v') / sqrt
    # (bc2)), fl(eps) and the add
    e_D = e_sqrt / sb2 + 3 * U * sv / sb2 + U * EPS + U * D
    st = lr / bc1
    # p' = fma(-fl(lr / bc1), fl(m' / denom), p): fl(lr / bc1) and the division, then the fma's rounding of p'
    return st * (e_m / D + np.abs(mp) * e_D / D ** 2) + 2 * U * st * np.abs(mp) / D + U * np.abs(pp)


def _reduce(per_epoch, key):
    mbs = [d for e in per_epoch for d in e]
    if key == "approx_kl":
        return float(np.mean([d[key] for d in per_epoch[-1]]))       # approx_kl_divs is reset at every epoch
    if key == "loss":
        return float(mbs[-1][key])                                   # loss.item() after the loop: the last minibatch
    return float(np.mean([d[key] for d in mbs]))


_LOG_NAMES = dict(pg="policy_gradient_loss", value_loss="value_loss", clip_fraction="clip_fraction",
                  approx_kl="approx_kl", entropy_loss="entropy_loss", loss="loss")


def sb3_logs(per_epoch, final_log_std, values, returns, n_updates, learning_rate, clip_range):
    """SB3 1.6 PPO.train's train/ dict [memory].  per_epoch: for each epoch that ran, the `logs` of its minibatches
    in order (target_kl's breaking minibatch included, as SB3 appends before it breaks); final_log_std: log_std after
    the last step; values / returns: the rollout buffer's (explained_variance with np.var)."""
    y, yp = np.asarray(returns, np.float64).reshape(-1), np.asarray(values, np.float64).reshape(-1)
    var_y = np.var(y)
    d = {"train/" + n: _reduce(per_epoch, k) for k, n in _LOG_NAMES.items()}
    d.update({"train/explained_variance": float("nan") if var_y == 0 else float(1 - np.var(y - yp) / var_y),
              "train/std": float(np.exp(np.asarray(final_log_std, np.float32).astype(np.float64)).mean()),
              "train/n_updates": n_updates, "train/learning_rate": learning_rate, "train/clip_range": clip_range})
    return d


def sb3_log_bounds(per_epoch_bounds):
    """Bounds on the kernel-side train/ values of sb3_logs: each log is a mean (or the last) of per-minibatch terms,
    so its bound is the same reduction of their `log_bounds`."""
    return {"train/" + n: _reduce(per_epoch_bounds, k) for k, n in _LOG_NAMES.items()}


def sb3_progress(iteration, n_steps, n_envs, total):
    """_current_progress_remaining of update `iteration` (1, 2, ...) of SB3's learn from 0 timesteps: learn calls
    _update_current_progress_remaining(num_timesteps, total) after collect_rollouts, so it counts the new rollout."""
    return 1.0 - float(iteration * n_steps * n_envs) / float(total)
