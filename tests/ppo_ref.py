"""Float64 statement of the PPO minibatch loss gradient (SB3 1.6 PPO.train, see csrc/r6_ppo.cuh) and a per-entry error
bound for the float32 kernel r6_ppo_grad, derived from its arithmetic in the style of policy_ref.py.  Also the
synthetic minibatches the tests feed it."""
import numpy as np

import policy_ref as pr

U = 2.0 ** -24                  # float32 unit roundoff
NPARAMS = 10311
LAYOUT = (("w0", (128, 13)), ("b0", (128,)), ("w1", (64, 128)), ("b1", (64,)), ("w2", (3, 64)), ("b2", (3,)),
          ("wv", (64,)), ("bv", (1,)), ("log_std", (3,)))
LOG_SQRT_2PI = 0.5 * np.log(2.0 * np.pi)
# |kernel - reference| <= C_BAR * bound: the bound takes every rounding at its maximum with one sign, and is first order
C_BAR = 2.0


def flat(w):
    return np.concatenate([np.asarray(w[k], np.float32).reshape(-1) for k, _ in LAYOUT])


def _f64(w):
    return {k: np.asarray(v, np.float32).astype(np.float64) for k, v in w.items()}


def _forward(W, x):
    h0 = np.tanh(x @ W["w0"].T + W["b0"])
    h1 = np.tanh(h0 @ W["w1"].T + W["b1"])
    return h0, h1, h1 @ W["w2"].T + W["b2"], h1 @ W["wv"].reshape(64) + W["bv"].reshape(1)[0]


def per_sample(w, x, a, old, adv_n, ret, clip=0.2, vf_coef=0.5, ent_coef=0.0):
    """Float64 per-sample quantities of the loss and its gradient (x [n,13], a [n,3], old / adv_n / ret [n]); adv_n is
    the normalised advantage A'."""
    W = _f64(w)
    x = np.asarray(x, np.float32).astype(np.float64)
    a = np.asarray(a, np.float32).astype(np.float64)
    h0, h1, mean, v = _forward(W, x)
    ls = W["log_std"]
    isg = np.exp(-ls)
    z = (a - mean) * isg
    logp = np.sum(-0.5 * z * z - ls - LOG_SQRT_2PI, axis=1)
    lr = logp - np.asarray(old, np.float32)
    ratio = np.exp(lr)
    rc = np.clip(ratio, 1 - clip, 1 + clip)
    s1, s2 = adv_n * ratio, adv_n * rc
    wgt = np.where(s1 <= s2, -s1, 0.0)
    gm = wgt[:, None] * z * isg
    gls = wgt[:, None] * (z * z - 1) - ent_coef
    gv = 2 * vf_coef * (v - np.asarray(ret, np.float32))
    s = gm @ W["w2"] + gv[:, None] * W["wv"].reshape(1, 64)
    d1 = s * (1 - h1 * h1)
    t = d1 @ W["w1"]
    d0 = t * (1 - h0 * h0)
    return dict(W=W, x=x, h0=h0, h1=h1, mean=mean, v=v, z=z, isg=isg, logp=logp, lr=lr, ratio=ratio, wgt=wgt, gm=gm,
                gls=gls, gv=gv, s=s, d1=d1, t=t, d0=d0, pg=-np.minimum(s1, s2), vloss=(np.asarray(ret, np.float32) - v) ** 2,
                clipped=(np.abs(ratio - 1) > clip).astype(np.float64), kl=(ratio - 1) - lr, adv=adv_n)


def _pack(dW0, db0, dW1, db1, dW2, db2, dwv, dbv, dls):
    return np.concatenate([dW0.reshape(-1), db0, dW1.reshape(-1), db1, dW2.reshape(-1), db2, dwv, [dbv], dls])


def grad_sum(q):
    """(gradient sum [P], term sums [4] = pg, vloss, clipped, kl) in float64."""
    g = _pack(q["d0"].T @ q["x"], q["d0"].sum(0), q["d1"].T @ q["h0"], q["d1"].sum(0), q["gm"].T @ q["h1"], q["gm"].sum(0),
              q["gv"] @ q["h1"], q["gv"].sum(), q["gls"].sum(0))
    return g, np.array([q["pg"].sum(), q["vloss"].sum(), q["clipped"].sum(), q["kl"].sum()])


def bound(q, vf_coef=0.5, ent_coef=0.0, samples_per_cta=128, forward_err=None):
    """Per-entry bound [P] on |r6_ppo_grad - grad_sum| and [4] on the term sums.  Each per-sample quantity carries a
    first-order running error bound through the float32 chain of csrc/r6_ppo.cuh; the CTA accumulation adds one
    rounding per sample to the running sum (<= u * samples_per_cta * sum |contribution|, a bound on the partial sums) and
    the two-stage reduction rounds the CTA partial and the float64 total once each (2u)."""
    W, x, h0, h1 = q["W"], q["x"], q["h0"], q["h1"]
    aW = {k: np.abs(v) for k, v in W.items()}
    # forward: the mode-0 bound of policy_ref (ppo_forward is mlp_forward's arithmetic, same order)
    a0, e0 = pr._layer(0, x, np.zeros_like(x), W["w0"], W["b0"])
    eh0 = pr._through_tanh(a0, e0, 0)
    a1, e1 = pr._layer(0, h0, eh0, W["w1"], W["b1"])
    eh1 = pr._through_tanh(a1, e1, 0)
    W2 = np.concatenate([W["w2"], W["wv"].reshape(1, 64)], 0)
    _, eo = pr._layer(0, h1, eh1, W2, np.concatenate([W["b2"], W["bv"].reshape(1)]))
    em, ev = eo[:, :3], eo[:, 3]
    z, isg, ratio, wgt, adv = q["z"], q["isg"], q["ratio"], q["wgt"], q["adv"]
    az = np.abs(z)
    # z = (a - mean) * expf(-ls): expf 2 ulp, the subtraction and the product 1 rounding each -> 4u relative
    ez = isg * em + 4 * U * az
    # logp: per dimension z*z, *0.5, - ls, - const, + running sum: 6 roundings on magnitudes <= 0.5 z^2 + |ls| + 1
    elogp = np.sum(az * ez + 6 * U * (0.5 * z * z + np.abs(W["log_std"]) + 1.0), axis=1)
    # ratio = expf(logp - old): the subtraction 1 rounding of |lr|, expf 2 ulp
    eratio = ratio * (elogp + U * np.abs(q["lr"]) + 2 * U)
    eadv = U * np.abs(adv)                                       # A' rounded once from float64
    ewgt = np.abs(adv) * eratio + ratio * eadv + U * np.abs(wgt)
    ewgt = np.where(wgt == 0, 0.0, ewgt)                        # clipped branch: exactly 0 (the decision cannot flip)
    aw = np.abs(wgt)[:, None]
    egm = ewgt[:, None] * az * isg + aw * ez * isg + 3 * U * np.abs(q["gm"])
    egls = ewgt[:, None] * np.abs(z * z - 1) + aw * 2 * az * ez + 3 * U * (aw * (z * z + 1) + abs(ent_coef))
    egv = 2 * vf_coef * ev + 2 * U * np.abs(q["gv"])          # 2 vf (v - R): the subtraction and the product
    ag = np.concatenate([np.abs(q["gm"]), np.abs(q["gv"])[:, None]], 1)
    eg = np.concatenate([egm, egv[:, None]], 1)
    # delta1 = (4-term fma chain) * fma(-h1, h1, 1): 4 + 1 + 1 roundings
    es = eg @ np.abs(W2) + 4 * U * (ag @ np.abs(W2))
    th1 = 1 - h1 * h1
    ed1 = es * th1 + np.abs(q["s"]) * (2 * np.abs(h1) * eh1 + 2 * U)
    # delta0 = (64-term fma chain) * fma(-h0, h0, 1)
    ad1 = np.abs(q["d1"])
    et = ed1 @ aW["w1"] + 64 * U * (ad1 @ aW["w1"])
    ed0 = et * (1 - h0 * h0) + np.abs(q["t"]) * (2 * np.abs(h0) * eh0 + 2 * U)
    ad0, ax, ah0, ah1 = np.abs(q["d0"]), np.abs(x), np.abs(h0), np.abs(h1)
    agm = np.abs(q["gm"])
    prop = _pack(ed0.T @ ax, ed0.sum(0), ed1.T @ ah0 + ad1.T @ eh0, ed1.sum(0), egm.T @ ah1 + agm.T @ eh1, egm.sum(0),
                 egv @ ah1 + np.abs(q["gv"]) @ eh1, egv.sum(), egls.sum(0))
    S = _pack(ad0.T @ ax, ad0.sum(0), ad1.T @ ah0, ad1.sum(0), agm.T @ ah1, agm.sum(0), np.abs(q["gv"]) @ ah1,
              np.abs(q["gv"]).sum(), np.abs(q["gls"]).sum(0))
    bnd = prop + U * (samples_per_cta + 2) * S
    # terms: float32 per sample, float64 sums.  pg = -min(A' r, A' rc): 1 rounding + the ratio / A' errors
    epg = np.abs(adv) * eratio + ratio * eadv + U * np.abs(q["pg"]) * 2
    evl = 2 * np.sqrt(q["vloss"]) * ev + 3 * U * q["vloss"]
    ekl = eratio + elogp + 4 * U * (np.abs(ratio - 1) + np.abs(q["lr"]) + 1)
    tb = np.array([epg.sum(), evl.sum(), 0.0, ekl.sum()]) + 1e-12
    return bnd, tb


def samples_per_cta(B, ctas=148, threads=128):
    """Samples of the busiest CTA of r6_ppo_grad (the length of its accumulation chains)."""
    tiles = -(-B // threads)
    return -(-tiles // min(tiles, ctas)) * threads


def minibatch(w, x, seed, clip=0.2):
    """Synthetic rollout data for observations x [n,13]: float32 raw actions a = mean + sigma z, old log-probs that put
    every float64 ratio in one of three bands (below 1 - clip, inside, above 1 + clip) at least 1e-3 away from 1 +- clip,
    advantages of both signs and returns around the value."""
    rng = np.random.default_rng(seed)
    n = len(x)
    W = _f64(w)
    _, _, mean, v = _forward(W, np.asarray(x, np.float32).astype(np.float64))
    sg = np.exp(W["log_std"])
    a = (mean + sg * rng.standard_normal((n, 3))).astype(np.float32)
    z = (a.astype(np.float64) - mean) / sg
    logp = np.sum(-0.5 * z * z - W["log_std"] - LOG_SQRT_2PI, axis=1)
    band = rng.integers(0, 3, n)
    r = np.where(band == 0, rng.uniform(0.5, 1 - clip - 0.01, n),
                 np.where(band == 1, rng.uniform(1 - clip + 0.01, 1 + clip - 0.01, n), rng.uniform(1 + clip + 0.01, 1.6, n)))
    old = (logp - np.log(r)).astype(np.float32)
    for _ in range(8):                                      # float32 rounding of old moved the ratio: keep the margin
        ratio = np.exp(logp - old.astype(np.float64))
        near = (np.abs(ratio - (1 - clip)) < 1e-3) | (np.abs(ratio - (1 + clip)) < 1e-3)
        if not near.any():
            break
        old[near] = (old[near] - 0.01).astype(np.float32)
    adv = (rng.standard_normal(n) * 2 + 0.3).astype(np.float32)
    ret = (v + rng.standard_normal(n)).astype(np.float32)
    return a, old, adv, ret


def adv_stats(adv):
    """(mean, 1 / (std + 1e-8)) in float64 with torch's unbiased std, as loss_and_grad forms them."""
    a = np.asarray(adv, np.float32).astype(np.float64)
    return np.array([a.mean(), 1.0 / (a.std(ddof=1) + 1e-8)])
