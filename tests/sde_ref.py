"""SB3 1.6's StateDependentNoiseDistribution (full_std=True, use_expln=False, learn_features=False, epsilon=1e-6) and the
PPO.train loss on it, restated in torch float64 on the CPU for the network of ppo.py with use_sde=True [memory]:

    sigma = exp(log_std) [64, 3];  E_i = sigma * xi_i;  h = the 64-unit trunk output, detached for the noise
    actions = mean + h E_i;  distribution = Normal(mean, sqrt(h^2 @ sigma^2 + 1e-6))
    log_prob, entropy: sums over the 3 actions

and a NumPy restatement of the Philox noise draw of r6_core.cuh (sde_noise_block)."""
import numpy as np
import torch

import philox_ref
import ppo_train_ref as tr

LAYOUT_SDE = (("w0", (128, 13)), ("b0", (128,)), ("w1", (64, 128)), ("b1", (64,)), ("w2", (3, 64)), ("b2", (3,)),
              ("wv", (64,)), ("bv", (1,)), ("log_std", (64, 3)))
NPARAMS_SDE = 10500
STREAM_SDE = 0x47534445            # 'GSDE' ^ (step hi << 8) ^ block


def unflat(p):
    out, o = {}, 0
    for k, s in LAYOUT_SDE:
        n = int(np.prod(s))
        out[k] = np.asarray(p[o:o + n], np.float32).reshape(s)
        o += n
    return out


def noise(seed, genv, step):
    """xi [n, 192] in float64 for global env ids genv [n] and one draw step: Philox block b gives components 4b .. 4b + 3,
    Box-Muller on the kernel's float32 uniforms (philox_ref.policy_uniforms) with both the cos and sin of each pair."""
    genv = np.atleast_1d(np.asarray(genv, np.uint64))
    step = np.uint64(step)
    out = np.zeros((len(genv), 192))
    for b in range(48):
        w = np.uint32(STREAM_SDE) ^ np.uint32((int(step) >> 32) << 8 & 0xFFFFFFFF) ^ np.uint32(b)
        ctr = np.stack([(genv & np.uint64(0xFFFFFFFF)).astype(np.uint32), (genv >> np.uint64(32)).astype(np.uint32),
                        np.full(len(genv), int(step) & 0xFFFFFFFF, np.uint32), np.full(len(genv), w, np.uint32)], -1)
        r = philox_ref.philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
        u1, u2, u3, u4 = (u.astype(np.float64) for u in philox_ref.policy_uniforms(r))
        ra, rb = np.sqrt(-2.0 * np.log(u1)), np.sqrt(-2.0 * np.log(u3))
        out[:, 4 * b:4 * b + 4] = np.stack([ra * np.cos(2 * np.pi * u2), ra * np.sin(2 * np.pi * u2),
                                            rb * np.cos(2 * np.pi * u4), rb * np.sin(2 * np.pi * u4)], -1)
    return out


def noise_bar(xi):
    """|xi_kernel - noise| bound of philox_ref.policy_noise_bar: 3 ulp relative plus 2^-48 of the radius (<= 6)."""
    return 3 * 2.0 ** -23 * np.abs(xi) + 2.0 ** -48 * 6.0


def _t(v):
    return torch.tensor(np.asarray(v, np.float32).astype(np.float64))


def forward(P, x):
    """(mean [n, 3], value [n], h [n, 64]) in float64."""
    h = torch.tanh(torch.tanh(_t(x) @ P["w0"].T + P["b0"]) @ P["w1"].T + P["b1"])
    return h @ P["w2"].T + P["b2"], h @ P["wv"].reshape(64) + P["bv"][0], h


def distribution(P, mean, h):
    variance = (h.detach() ** 2) @ (torch.exp(P["log_std"]) ** 2)
    return torch.distributions.Normal(mean, torch.sqrt(variance + 1e-6))


def sb3_loss_sum(P, x, a, old, adv_n, ret, clip, vf_coef, ent_coef):
    """SUM over the samples of SB3's per-sample PPO loss with gSDE (pg + vf_coef (R - V)^2 - ent_coef entropy) on float64
    parameter tensors P, and the per-sample entropy."""
    mean, values, h = forward(P, x)
    dist = distribution(P, mean, h)
    log_prob, entropy = dist.log_prob(_t(a)).sum(1), dist.entropy().sum(1)
    A = torch.as_tensor(np.asarray(adv_n, np.float64))
    ratio = torch.exp(log_prob - _t(old))
    pg = -torch.min(A * ratio, A * torch.clamp(ratio, 1 - clip, 1 + clip))
    loss = pg + vf_coef * (_t(ret) - values) ** 2 - ent_coef * entropy
    return loss.sum(), entropy


def grad_sum(w, x, a, old, adv_n, ret, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """(flat float64 gradient [NPARAMS_SDE] of the summed loss, per-sample entropy) by autograd."""
    P = {k: torch.tensor(np.asarray(w[k], np.float64), requires_grad=True) for k, _ in LAYOUT_SDE}
    loss, ent = sb3_loss_sum(P, x, a, old, adv_n, ret, clip, vf_coef, ent_coef)
    loss.backward()
    return torch.cat([P[k].grad.reshape(-1) for k, _ in LAYOUT_SDE]).numpy(), ent.detach().numpy()


def sample(w, x, xi):
    """SB3's gSDE sample for observations x [n, 13] and noise xi [n, 192] in float64: (raw actions, log_prob, mean, h)."""
    P = {k: torch.tensor(np.asarray(w[k], np.float64)) for k, _ in LAYOUT_SDE}
    mean, _, h = forward(P, x)
    E = torch.exp(P["log_std"])[None] * torch.tensor(np.asarray(xi, np.float64)).reshape(-1, 64, 3)
    raw = mean + torch.bmm(h[:, None], E)[:, 0]
    logp = distribution(P, mean, h).log_prob(raw).sum(1)
    return raw.numpy(), logp.numpy(), mean.numpy(), h.numpy()


def reference_step(params, m, v, step, rollout, idx, lr, cfg, K=1024, err_sum=None):
    """One minibatch of SB3 1.6 PPO(use_sde=True).train from the float32 pre-step state params / m / v [NPARAMS_SDE]:
    the mean loss, backward, clip_grad_norm_, torch.optim.Adam(eps=1e-5) step number `step` in float64 (as
    ppo_train_ref.reference_step for the diagonal Gaussian).  err_sum [NPARAMS_SDE]: the sum over the minibatch of the
    per-sample gradient magnitudes; the kernel's gradient sum is held to K u err_sum (K = 1024: each per-sample entry is a
    float32 product of factors that each carry at most a few hundred roundings -- the 128- and 64-term dot products of the
    forward and backward pass, std's 64-term sum, exp / log of the ratio -- and the sum adds one per sample), and the
    step to ppo_train_ref.step_bound of that.  Returns dict(p, bound, entropy = mean per-sample entropy)."""
    B = len(idx)
    w = unflat(params)
    x, a = rollout["obs"][idx], rollout["actions"][idx]
    old, ret = rollout["log_probs"][idx], rollout["returns"][idx]
    adv_n = tr.normalized_advantages(rollout["advantages"][idx], cfg.normalize_advantage)
    P = {k: torch.tensor(w[k].astype(np.float64), requires_grad=True) for k, _ in LAYOUT_SDE}
    loss, ent = sb3_loss_sum(P, x, a, old, adv_n, ret, cfg.clip_range, cfg.vf_coef, cfg.ent_coef)
    (loss / B).backward()
    plist = [P[k] for k, _ in LAYOUT_SDE]
    g = torch.cat([t.grad.reshape(-1) for t in plist]).numpy().copy()
    norm = float(torch.nn.utils.clip_grad_norm_(plist, cfg.max_grad_norm))
    opt = torch.optim.Adam(plist, lr=lr, betas=tr.BETAS, eps=tr.EPS, foreach=False)
    mm, vv = unflat(m), unflat(v)
    for (k, _), t in zip(LAYOUT_SDE, plist):
        opt.state[t] = {"step": torch.tensor(float(step - 1)), "exp_avg": torch.tensor(mm[k].astype(np.float64)),
                        "exp_avg_sq": torch.tensor(vv[k].astype(np.float64))}
    opt.step()
    cat = lambda f: torch.cat([f(t).reshape(-1) for t in plist]).detach().numpy().copy()
    gc, pp = cat(lambda t: t.grad), cat(lambda t: t)
    mp, vp = cat(lambda t: opt.state[t]["exp_avg"]), cat(lambda t: opt.state[t]["exp_avg_sq"])
    e_sum = K * tr.U * np.asarray(err_sum, np.float64) / B
    bound = tr.step_bound(g, e_sum, norm, cfg.max_grad_norm, gc, np.asarray(m, np.float64), mp, vp, pp, lr, step)
    return dict(p=pp, bound=bound, entropy=float(ent.detach().mean()))
