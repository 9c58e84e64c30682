"""Float64 statement of SB3 1.6's default MlpPolicy without policy_kwargs — separate tanh towers
net_arch [dict(pi=[64, 64], vf=[64, 64])], action_net on the policy latent, value_net on the value latent — and of
PPO.train's loss on it (the shared-trunk statement is tests/ppo_train_ref.sb3_loss), with torch autograd for the
gradient in the flat R6_PPO_NPARAMS_SEP layout.  Also the weight and minibatch generators of the separate-tower tests."""
import numpy as np
import torch

from rl_rocket_6dof_b200.ppo import LAYOUT_SEP

POLICY_KEYS = ("w0", "b0", "w1", "b1", "w2", "b2")


def flat(w):
    return np.concatenate([np.asarray(w[k], np.float32).reshape(-1) for k, _ in LAYOUT_SEP])


def weights(seed, scale=0.3):
    """Random separate-tower weights (not orthogonal: every entry differs) with critic and log_std."""
    rng = np.random.default_rng(seed)
    w = {k: (rng.standard_normal(s) * (scale if "w" in k and k != "log_std" else 0.05)).astype(np.float32)
         for k, s in LAYOUT_SEP}
    w["log_std"] = rng.uniform(-1.0, 0.3, 3).astype(np.float32)
    return w


def forward64(w, x):
    """(mean [n, 3], value [n]) in float64 from the float32 weights and observations."""
    W = {k: np.asarray(v, np.float32).astype(np.float64) for k, v in w.items()}
    x = np.asarray(x, np.float32).astype(np.float64).reshape(-1, 13)
    hp = np.tanh(np.tanh(x @ W["w0"].T + W["b0"]) @ W["w1"].T + W["b1"])
    hv = np.tanh(np.tanh(x @ W["vf_w0"].T + W["vf_b0"]) @ W["vf_w1"].T + W["vf_b1"])
    return hp @ W["w2"].T + W["b2"], hv @ W["wv"].reshape(64) + W["bv"].reshape(1)[0]


def towers(w):
    """The two towers as shared-trunk-shaped dicts (policy with action_net; value with value_net as its only output row),
    for the per-tower forward error bound of tests/policy_ref.bound."""
    pol = {k: w[k] for k in POLICY_KEYS}
    val = {"w0": w["vf_w0"], "b0": w["vf_b0"], "w1": w["vf_w1"], "b1": w["vf_b1"],
           "w2": np.asarray(w["wv"]).reshape(1, 64), "b2": np.asarray(w["bv"]).reshape(1)}
    return pol, val


def grad_sum(w, x, a, old, adv_n, ret, clip=0.2, vf_coef=0.5, ent_coef=0.0, chunk=65536):
    """SB3 1.6 PPO.train's loss on this network (policy_loss - ent_coef entropy + vf_coef mse, on the normalised
    advantages adv_n) written as the SUM over the samples — n times SB3's mean, the sum r6_ppo_grad returns — through
    torch float64 autograd.  Returns (gradient [R6_PPO_NPARAMS_SEP], term sums [4] = pg, (R - V)^2, clipped, approx-kl,
    mag [R6_PPO_NPARAMS_SEP] = sum over the samples of |per-sample gradient| of each entry).  The per-sample gradients are
    the deltas autograd leaves on the pre-activations (the loss is a sum, so they are per sample), times the layer
    inputs: mag of a weight is |delta|^T |input|."""
    t = lambda v: torch.tensor(np.asarray(v, np.float32).astype(np.float64))
    n = len(np.asarray(ret))
    g, terms, mag = 0.0, 0.0, 0.0
    for i in range(0, n, chunk):
        sl = slice(i, min(i + chunk, n))
        P = {k: torch.tensor(np.asarray(w[k], np.float32).astype(np.float64).reshape(s), requires_grad=True)
             for k, s in LAYOUT_SEP}
        xs = t(np.asarray(x)[sl])
        m = len(xs)
        pre = {}

        def keep(name, v):
            v.retain_grad()
            pre[name] = v
            return v
        h0p = torch.tanh(keep("a0p", xs @ P["w0"].T + P["b0"]))
        hp = torch.tanh(keep("a1p", h0p @ P["w1"].T + P["b1"]))
        h0v = torch.tanh(keep("a0v", xs @ P["vf_w0"].T + P["vf_b0"]))
        hv = torch.tanh(keep("a1v", h0v @ P["vf_w1"].T + P["vf_b1"]))
        mean = keep("mean", hp @ P["w2"].T + P["b2"])
        values = keep("v", hv @ P["wv"].reshape(64) + P["bv"][0])
        ls = keep("ls", P["log_std"].unsqueeze(0).expand(m, 3))
        dist = torch.distributions.Normal(mean, torch.exp(ls))
        log_prob, entropy = dist.log_prob(t(np.asarray(a)[sl])).sum(1), dist.entropy().sum(1)
        A = torch.as_tensor(np.asarray(adv_n, np.float64)[sl])
        lr = log_prob - t(np.asarray(old)[sl])
        ratio = torch.exp(lr)
        pg = -torch.min(A * ratio, A * torch.clamp(ratio, 1 - clip, 1 + clip))
        vl = (t(np.asarray(ret)[sl]) - values) ** 2
        (pg.sum() - ent_coef * entropy.sum() + vf_coef * vl.sum()).backward()
        with torch.no_grad():
            terms = terms + np.array([float(pg.sum()), float(vl.sum()), float((torch.abs(ratio - 1) > clip).double().sum()),
                                      float(((ratio - 1) - lr).sum())])
            g = g + np.concatenate([P[k].grad.numpy().reshape(-1) for k, _ in LAYOUT_SEP])
            d = {k: v.grad.abs() for k, v in pre.items()}
            ax, ah0p, ah0v, ahp, ahv = xs.abs(), h0p.abs(), h0v.abs(), hp.abs(), hv.abs()
            parts = {"w0": d["a0p"].T @ ax, "b0": d["a0p"].sum(0), "vf_w0": d["a0v"].T @ ax, "vf_b0": d["a0v"].sum(0),
                     "w1": d["a1p"].T @ ah0p, "b1": d["a1p"].sum(0), "vf_w1": d["a1v"].T @ ah0v, "vf_b1": d["a1v"].sum(0),
                     "w2": d["mean"].T @ ahp, "b2": d["mean"].sum(0), "wv": d["v"] @ ahv, "bv": d["v"].sum().reshape(1),
                     "log_std": d["ls"].sum(0)}
            mag = mag + np.concatenate([parts[k].numpy().reshape(-1) for k, _ in LAYOUT_SEP])
    return g, terms, mag


def minibatch(w, n, seed, ratio_noise=0.4):
    """Observations, Gaussian actions of the policy itself (ratios near 1), perturbed old log-probs (ratios on both sides
    of the clip range), advantages and returns."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((n, 13)) * 0.8).astype(np.float32)
    mean, v = forward64(w, x)
    sg = np.exp(np.asarray(w["log_std"], np.float64))
    eps = rng.standard_normal((n, 3))
    a = (mean + sg * eps).astype(np.float32)
    logp = np.sum(-0.5 * eps ** 2 - np.log(sg) - 0.5 * np.log(2 * np.pi), 1)
    old = (logp + rng.normal(0.0, ratio_noise, n)).astype(np.float32)
    adv = (rng.standard_normal(n) * 3.0 + 0.5).astype(np.float32)
    ret = (v + rng.standard_normal(n)).astype(np.float32)
    return x, a, old, adv, ret


def bound(w, x, a, old, adv_n, ret, clip=0.2, vf_coef=0.5, ent_coef=0.0, samples_per_cta=128, chunk=32768):
    """Per-entry bound [R6_PPO_NPARAMS_SEP] on |r6_ppo_grad - exact gradient sum| for the separate towers: tests/ppo_ref.bound
    (the shared-trunk derivation, csrc/r6_ppo.cuh's float32 chain one rounding at a time) restated for ppo_forward_sep /
    ppo_delta1_sep / ppo_delta0 per tower.  The forward errors of the mean and of V are policy_ref's mode-0 bounds of each
    tower; they enter through z = (a - mean) / sigma and V - R, so a sample whose V - R or z^2 - 1 nearly cancels gets the
    absolute error those carry, not a relative one.  Summed over chunks of samples (the bound is a sum over samples)."""
    import policy_ref as pr
    import ppo_ref
    U = 2.0 ** -24
    W = {k: np.asarray(v, np.float32).astype(np.float64) for k, v in w.items()}
    aW = {k: np.abs(v) for k, v in W.items()}
    wv = W["wv"].reshape(1, 64)
    n = len(np.asarray(ret))
    total = 0.0
    for i in range(0, n, chunk):
        sl = slice(i, min(i + chunk, n))
        xs = np.asarray(x, np.float32)[sl].astype(np.float64)
        As = np.asarray(a, np.float32)[sl].astype(np.float64)
        adv = np.asarray(adv_n, np.float64)[sl]
        # forward with the mode-0 bounds of each tower
        a0p, e0p = pr._layer(0, xs, np.zeros_like(xs), W["w0"], W["b0"])
        h0p, eh0p = np.tanh(a0p), pr._through_tanh(a0p, e0p, 0)
        a1p, e1p = pr._layer(0, h0p, eh0p, W["w1"], W["b1"])
        h1p, eh1p = np.tanh(a1p), pr._through_tanh(a1p, e1p, 0)
        mean, em = h1p @ W["w2"].T + W["b2"], pr._layer(0, h1p, eh1p, W["w2"], W["b2"])[1]
        a0v, e0v = pr._layer(0, xs, np.zeros_like(xs), W["vf_w0"], W["vf_b0"])
        h0v, eh0v = np.tanh(a0v), pr._through_tanh(a0v, e0v, 0)
        a1v, e1v = pr._layer(0, h0v, eh0v, W["vf_w1"], W["vf_b1"])
        h1v, eh1v = np.tanh(a1v), pr._through_tanh(a1v, e1v, 0)
        v, ev = (h1v @ wv.T)[:, 0] + W["bv"][0], pr._layer(0, h1v, eh1v, wv, W["bv"].reshape(1))[1][:, 0]
        # the head (ppo_head), as ppo_ref.per_sample / ppo_ref.bound
        ls = W["log_std"]
        isg = np.exp(-ls)
        z = (As - mean) * isg
        logp = np.sum(-0.5 * z * z - ls - ppo_ref.LOG_SQRT_2PI, axis=1)
        lr = logp - np.asarray(old, np.float32)[sl]
        ratio = np.exp(lr)
        s1, s2 = adv * ratio, adv * np.clip(ratio, 1 - clip, 1 + clip)
        wgt = np.where(s1 <= s2, -s1, 0.0)
        gm = wgt[:, None] * z * isg
        gls = wgt[:, None] * (z * z - 1) - ent_coef
        gv = 2 * vf_coef * (v - np.asarray(ret, np.float32)[sl])
        az = np.abs(z)
        ez = isg * em + 4 * U * az
        elogp = np.sum(az * ez + 6 * U * (0.5 * z * z + np.abs(ls) + 1.0), axis=1)
        eratio = ratio * (elogp + U * np.abs(lr) + 2 * U)
        ewgt = np.where(wgt == 0, 0.0, np.abs(adv) * eratio + ratio * U * np.abs(adv) + U * np.abs(wgt))
        aw = np.abs(wgt)[:, None]
        egm = ewgt[:, None] * az * isg + aw * ez * isg + 3 * U * np.abs(gm)
        egls = ewgt[:, None] * np.abs(z * z - 1) + aw * 2 * az * ez + 3 * U * (aw * (z * z + 1) + abs(ent_coef))
        egv = 2 * vf_coef * ev + 2 * U * np.abs(gv)
        # ppo_delta1_sep: policy s = 3-term chain over action_net, value s = wv_k g_v (one product); * fma(-h, h, 1)
        sp, sv = gm @ W["w2"], gv[:, None] * wv
        esp = egm @ aW["w2"] + 3 * U * (np.abs(gm) @ aW["w2"])
        esv = egv[:, None] * np.abs(wv) + U * np.abs(sv)
        d1p, d1v = sp * (1 - h1p * h1p), sv * (1 - h1v * h1v)
        ed1p = esp * (1 - h1p * h1p) + np.abs(sp) * (2 * np.abs(h1p) * eh1p + 2 * U)
        ed1v = esv * (1 - h1v * h1v) + np.abs(sv) * (2 * np.abs(h1v) * eh1v + 2 * U)
        # ppo_delta0 per tower: 64-term fma chain * fma(-h0, h0, 1)
        tp, tv = d1p @ W["w1"], d1v @ W["vf_w1"]
        etp = ed1p @ aW["w1"] + 64 * U * (np.abs(d1p) @ aW["w1"])
        etv = ed1v @ aW["vf_w1"] + 64 * U * (np.abs(d1v) @ aW["vf_w1"])
        d0p, d0v = tp * (1 - h0p * h0p), tv * (1 - h0v * h0v)
        ed0p = etp * (1 - h0p * h0p) + np.abs(tp) * (2 * np.abs(h0p) * eh0p + 2 * U)
        ed0v = etv * (1 - h0v * h0v) + np.abs(tv) * (2 * np.abs(h0v) * eh0v + 2 * U)
        ax = np.abs(xs)
        prop = {"w0": ed0p.T @ ax, "b0": ed0p.sum(0), "vf_w0": ed0v.T @ ax, "vf_b0": ed0v.sum(0),
                "w1": ed1p.T @ np.abs(h0p) + np.abs(d1p).T @ eh0p, "b1": ed1p.sum(0),
                "vf_w1": ed1v.T @ np.abs(h0v) + np.abs(d1v).T @ eh0v, "vf_b1": ed1v.sum(0),
                "w2": egm.T @ np.abs(h1p) + np.abs(gm).T @ eh1p, "b2": egm.sum(0),
                "wv": egv @ np.abs(h1v) + np.abs(gv) @ eh1v, "bv": np.array([egv.sum()]), "log_std": egls.sum(0)}
        S = {"w0": np.abs(d0p).T @ ax, "b0": np.abs(d0p).sum(0), "vf_w0": np.abs(d0v).T @ ax, "vf_b0": np.abs(d0v).sum(0),
             "w1": np.abs(d1p).T @ np.abs(h0p), "b1": np.abs(d1p).sum(0), "vf_w1": np.abs(d1v).T @ np.abs(h0v),
             "vf_b1": np.abs(d1v).sum(0), "w2": np.abs(gm).T @ np.abs(h1p), "b2": np.abs(gm).sum(0),
             "wv": np.abs(gv) @ np.abs(h1v), "bv": np.array([np.abs(gv).sum()]), "log_std": np.abs(gls).sum(0)}
        flat_ = lambda d: np.concatenate([np.asarray(d[k]).reshape(-1) for k, _ in LAYOUT_SEP])
        total = total + flat_(prop) + U * (samples_per_cta + 2) * flat_(S)
    return total
