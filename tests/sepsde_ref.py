"""SB3 1.6's PPO("MlpPolicy", env, use_sde=True) without policy_kwargs -- the separate tanh towers of tests/sep_ref.py
with the StateDependentNoiseDistribution of tests/sde_ref.py -- restated in torch float64 on the CPU [memory]:

    hp, hv = the policy and value towers' 64-unit latents;  mean = action_net(hp), V = value_net(hv)
    latent_sde = hp, detached (learn_features=False);  distribution = Normal(mean, sqrt(hp^2 @ exp(log_std)^2 + 1e-6))
    actions = mean + hp (exp(log_std) * xi)

with autograd for the gradient in the flat R6_PPO_NPARAMS_SEP_SDE layout, the sample of the policy kernels, and one
minibatch of PPO.train (as sde_ref.reference_step).  `latent` and `detach` select the two wrong statements the tests
must tell apart from SB3's: the value latent as h, and the gradient let through std into the policy tower."""
import numpy as np
import torch

import sde_ref
import sep_ref
import ppo_train_ref as tr
from rl_rocket_6dof_b200.ppo import LAYOUT_SEP_SDE, NPARAMS_SEP_SDE

LOG_STD = sum(int(np.prod(s)) for _, s in LAYOUT_SEP_SDE[:-1])     # offset of log_std: 10372


def flat(w):
    return np.concatenate([np.asarray(w[k], np.float32).reshape(-1) for k, _ in LAYOUT_SEP_SDE])


def unflat(p):
    out, o = {}, 0
    for k, s in LAYOUT_SEP_SDE:
        n = int(np.prod(s))
        out[k] = np.asarray(p[o:o + n], np.float32).reshape(s)
        o += n
    return out


def weights(seed, scale=0.3):
    """sep_ref.weights with a [64, 3] log_std that is not constant."""
    w = sep_ref.weights(seed, scale)
    w["log_std"] = np.random.default_rng(seed + 1000).uniform(-1.0, 0.5, (64, 3)).astype(np.float32)
    return w


def _t(v):
    return torch.tensor(np.asarray(v, np.float32).astype(np.float64))


def forward(P, x):
    """(mean [n, 3], value [n], hp [n, 64], hv [n, 64]) in float64: sep_ref.forward64's network on tensors."""
    x = _t(x).reshape(-1, 13)
    hp = torch.tanh(torch.tanh(x @ P["w0"].T + P["b0"]) @ P["w1"].T + P["b1"])
    hv = torch.tanh(torch.tanh(x @ P["vf_w0"].T + P["vf_b0"]) @ P["vf_w1"].T + P["vf_b1"])
    return hp @ P["w2"].T + P["b2"], hv @ P["wv"].reshape(64) + P["bv"].reshape(1)[0], hp, hv


def distribution(P, mean, hp, hv, latent="policy", detach=True):
    """sde_ref.distribution on the policy latent (SB3); latent="value" or detach=False are the wrong statements."""
    h = hp if latent == "policy" else hv
    if detach:
        return sde_ref.distribution(P, mean, h)
    return torch.distributions.Normal(mean, torch.sqrt((h ** 2) @ (torch.exp(P["log_std"]) ** 2) + 1e-6))


def sb3_loss_sum(P, x, a, old, adv_n, ret, clip, vf_coef, ent_coef, clip_range_vf=None, old_values=None,
                 latent="policy", detach=True):
    """SUM over the samples of SB3's per-sample PPO loss on float64 parameter tensors P, the term sums [4] (pg, value
    loss, clipped count, approx-kl) and the per-sample entropy.  clip_range_vf: SB3's value clipping around old_values."""
    mean, values, hp, hv = forward(P, x)
    dist = distribution(P, mean, hp, hv, latent, detach)
    log_prob, entropy = dist.log_prob(_t(a)).sum(1), dist.entropy().sum(1)
    A = torch.as_tensor(np.asarray(adv_n, np.float64))
    lr = log_prob - _t(old)
    ratio = torch.exp(lr)
    pg = -torch.min(A * ratio, A * torch.clamp(ratio, 1 - clip, 1 + clip))
    if clip_range_vf is not None:
        vo = _t(old_values)
        values = vo + torch.clamp(values - vo, -clip_range_vf, clip_range_vf)
    vl = (_t(ret) - values) ** 2
    with torch.no_grad():
        terms = np.array([float(pg.sum()), float(vl.sum()), float((torch.abs(ratio - 1) > clip).double().sum()),
                          float(((ratio - 1) - lr).sum())])
    return (pg + vf_coef * vl - ent_coef * entropy).sum(), terms, entropy


def grad_sum(w, x, a, old, adv_n, ret, clip=0.2, vf_coef=0.5, ent_coef=0.0, clip_range_vf=None, old_values=None,
             latent="policy", detach=True, chunk=65536):
    """(flat float64 gradient [R6_PPO_NPARAMS_SEP_SDE] of the summed loss, term sums [4], per-sample entropy) by autograd,
    in chunks of samples (the loss is a sum)."""
    n = len(np.asarray(ret))
    g, terms, ents = 0.0, 0.0, []
    sl = lambda v, s: None if v is None else np.asarray(v)[s]
    for i in range(0, n, chunk):
        s = slice(i, min(i + chunk, n))
        P = {k: torch.tensor(np.asarray(w[k], np.float32).astype(np.float64).reshape(sh), requires_grad=True)
             for k, sh in LAYOUT_SEP_SDE}
        loss, t, ent = sb3_loss_sum(P, sl(x, s), sl(a, s), sl(old, s), sl(adv_n, s), sl(ret, s), clip, vf_coef, ent_coef,
                                    clip_range_vf, sl(old_values, s), latent, detach)
        loss.backward()
        g = g + torch.cat([P[k].grad.reshape(-1) for k, _ in LAYOUT_SEP_SDE]).numpy()
        terms = terms + t
        ents.append(ent.detach().numpy())
    return g, terms, np.concatenate(ents)


def sample(w, x, xi):
    """The gSDE sample of the separate towers for observations x [n, 13] and noise xi [n, 192] in float64:
    (raw actions, log_prob, mean, value, hp)."""
    P = {k: torch.tensor(np.asarray(w[k], np.float32).astype(np.float64).reshape(s)) for k, s in LAYOUT_SEP_SDE}
    mean, value, hp, hv = forward(P, x)
    E = torch.exp(P["log_std"])[None] * torch.tensor(np.asarray(xi, np.float64)).reshape(-1, 64, 3)
    raw = mean + torch.bmm(hp[:, None], E)[:, 0]
    logp = distribution(P, mean, hp, hv).log_prob(raw).sum(1)
    return raw.numpy(), logp.numpy(), mean.numpy(), value.numpy(), hp.numpy()


def minibatch(w, n, seed, ratio_noise=0.4):
    """Observations, gSDE actions of the policy itself (ratios near 1), perturbed old log-probs (ratios on both sides of
    the clip range), advantages, returns, and old values on both sides of any value-clip band."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((n, 13)) * 0.8).astype(np.float32)
    raw, logp, _, v, _ = sample(w, x, rng.standard_normal((n, 192)))
    old = (logp + rng.normal(0.0, ratio_noise, n)).astype(np.float32)
    adv = (rng.standard_normal(n) * 3.0 + 0.5).astype(np.float32)
    ret = (v + rng.standard_normal(n)).astype(np.float32)
    vold = (v + rng.normal(0.0, 0.3, n)).astype(np.float32)
    return x, raw.astype(np.float32), old, adv, ret, vold


def reference_step(params, m, v, step, rollout, idx, lr, cfg, K=1024, err_sum=None):
    """One minibatch of SB3 1.6 PPO(use_sde=True).train on the separate towers from the float32 pre-step state
    params / m / v [R6_PPO_NPARAMS_SEP_SDE], as sde_ref.reference_step: mean loss, backward, clip_grad_norm_,
    torch.optim.Adam(eps=1e-5) step `step` in float64; the kernel's gradient sum held to K u err_sum (err_sum: the sum
    over the minibatch of the per-sample gradient magnitudes) and the step to ppo_train_ref.step_bound of that.
    Returns dict(p, bound, entropy = mean per-sample entropy)."""
    B = len(idx)
    w = unflat(params)
    x, a = rollout["obs"][idx], rollout["actions"][idx]
    old, ret = rollout["log_probs"][idx], rollout["returns"][idx]
    adv_n = tr.normalized_advantages(rollout["advantages"][idx], cfg.normalize_advantage)
    vfc = cfg.clip_range_vf
    P = {k: torch.tensor(w[k].astype(np.float64), requires_grad=True) for k, _ in LAYOUT_SEP_SDE}
    loss, _, ent = sb3_loss_sum(P, x, a, old, adv_n, ret, cfg.clip_range, cfg.vf_coef, cfg.ent_coef, vfc,
                                None if vfc is None else rollout["values"][idx])
    (loss / B).backward()
    plist = [P[k] for k, _ in LAYOUT_SEP_SDE]
    g = torch.cat([t.grad.reshape(-1) for t in plist]).numpy().copy()
    norm = float(torch.nn.utils.clip_grad_norm_(plist, cfg.max_grad_norm))
    opt = torch.optim.Adam(plist, lr=lr, betas=tr.BETAS, eps=tr.EPS, foreach=False)
    mm, vv = unflat(m), unflat(v)
    for (k, _), t in zip(LAYOUT_SEP_SDE, plist):
        opt.state[t] = {"step": torch.tensor(float(step - 1)), "exp_avg": torch.tensor(mm[k].astype(np.float64)),
                        "exp_avg_sq": torch.tensor(vv[k].astype(np.float64))}
    opt.step()
    cat = lambda f: torch.cat([f(t).reshape(-1) for t in plist]).detach().numpy().copy()
    gc, pp = cat(lambda t: t.grad), cat(lambda t: t)
    mp, vp = cat(lambda t: opt.state[t]["exp_avg"]), cat(lambda t: opt.state[t]["exp_avg_sq"])
    e_sum = K * tr.U * np.asarray(err_sum, np.float64) / B
    bound = tr.step_bound(g, e_sum, norm, cfg.max_grad_norm, gc, np.asarray(m, np.float64), mp, vp, pp, lr, step)
    return dict(p=pp, bound=bound, entropy=float(ent.detach().mean()))


assert NPARAMS_SEP_SDE == LOG_STD + 192 == 10564
