"""Float64 statement of the policy network the kernels evaluate (SB3 ActorCriticPolicy, net_arch [128, 64], tanh, shared
trunk with the value head on the last latent) and a forward error bound for each of the four kernel implementations
(r6_policy* tensor_cores = 0..3).  The bound is derived from the arithmetic each mode performs, not fitted to
measurements: a kernel that misses it by more than a small constant computes something else than the network.

Also the weight families and observation sets the policy tests run on."""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policy_cl.npz")

U_RN = 2.0 ** -24        # float32 unit roundoff, round to nearest
U_TZ = 2.0 ** -23        # float32 unit roundoff of an adder that may truncate (tensor-core accumulation)
FAMILIES = ("golden", "sb3_init", "saturating", "tf32_edges")
MODES = (0, 1, 2, 3)


def forward64(w, x):
    """(unclipped mean [n,3], value [n]) in float64 from the float32 weights and observations; value 0 without a critic."""
    x = np.asarray(x, np.float32).astype(np.float64).reshape(-1, 13)
    W = {k: np.asarray(v, np.float32).astype(np.float64) for k, v in w.items() if v is not None}
    h0 = np.tanh(x @ W["w0"].T + W["b0"])
    h1 = np.tanh(h0 @ W["w1"].T + W["b1"])
    mean = h1 @ W["w2"].T + W["b2"]
    value = h1 @ W["wv"].reshape(64) + W["bv"].reshape(1)[0] if "wv" in W else np.zeros(len(x))
    return mean, value


# ---- the bound ---------------------------------------------------------------------------------------------------------
# A pre-activation a = W h + b with K inputs is computed with absolute error at most (first order)
#     prod(mode) |W||h|  +  acc(mode)  +  |W| e_h            (e_h = error bound of the layer's input h)
# where prod is the relative error of one product as the mode forms it and acc the error of accumulating the products
# and the bias, a running bound evaluated on the exact partial sums in the order the mode adds them.
def _prod(mode):
    if mode == 0:
        return 0.0          # FMA: the product enters the sum unrounded
    if mode == 1:
        # mma.sync 3xTF32 (r6_mlp_tc.cuh): a = hi + lo, hi = round_tf32(a) (|a - hi| <= 2^-11 |a|), lo = a - hi exact in
        # float32 but read by the TF32 MMA with its 13 low bits ignored (truncation: < 2^-10 |lo| <= 2^-21 |a|).
        # Dropped lo*lo 2^-22 + the truncated lo of either operand 2 * 2^-21 = 2.5 * 2^-21 of |W h| per product.
        return 2.5 * 2.0 ** -21
    if mode == 2:
        # single-pass TF32 (tcgen05 fast mode): both operands rounded to the nearest TF32 (2^-11 each), and their product
        return 2.0 * 2.0 ** -11 + 2.0 ** -22
    if mode == 3:
        # tcgen05 3xTF32: hi = round_tf32(a), lo = round_tf32(a - hi) (error <= 2^-11 |a - hi| <= 2^-22 |a|): dropped
        # lo*lo 2^-22 + the rounded lo of either operand 2 * 2^-22 = 1.5 * 2^-21
        return 1.5 * 2.0 ** -21
    raise ValueError(mode)


def _acc(mode, h, W, b, chunk=512):
    """Accumulation error of h @ W.T + b as the mode sums it (h [n,K], W [m,K], b [m], all float64)."""
    n, K = h.shape
    out = np.empty((n, W.shape[0]))
    for i in range(0, n, chunk):
        hc = h[i:i + chunk]
        if mode == 0:
            # mlp_forward: s = w_1 h_1, then s = fma(w_j, h_j, s) for j = 2..K, then s + b: K + 1 roundings to nearest,
            # each at most 2^-24 of the exact partial sum it rounds (Higham, running error bound)
            s = np.cumsum(hc[:, None, :] * W[None, :, :], axis=2)
            out[i:i + chunk] = U_RN * (np.abs(s).sum(2) + np.abs(s[:, :, -1] + b))
            continue
        # One MMA adds a K-block of 8 products to the accumulator c.  Allowing alignment to the largest addend with
        # truncation (no guard bits) and a truncated result: each of the 8 addends that are not the largest loses < 1 ulp
        # of the largest, the result one more ulp -> at most 9 * 2^-23 * M per MMA, M the largest magnitude in play.
        # Modes 1 and 3 issue three MMAs per K-block (hi*hi, lo*hi, hi*lo in some order) whose accumulator values lie
        # between c_b and c_(b+1) = c_b + block within the lo products (<= 2^-9 of sum |p|), so for all three
        # M_b = max(|c_b|, |c_(b+1)|) + max |p| + 2^-9 sum_block |p|.
        # mma.sync (mode 1) starts the accumulator at the bias; tcgen05 (modes 2, 3) starts at 0 and adds the bias in the
        # epilogue: fma(acc, c, RN(c b)) with c = RN(2 log2 e) in the hidden layers (three roundings to nearest), one
        # float32 add in the output layer -> 3 * 2^-24 (|acc| + |b|) + 2^-24 |a|, bounded by 4 * 2^-24 (sum |p| + |b|).
        passes = 1 if mode == 2 else 3
        c = np.broadcast_to(b if mode == 1 else np.zeros_like(b), (len(hc), len(b))).copy()
        e = np.zeros_like(c)
        for k in range(0, K, 8):
            p = np.abs(hc[:, None, k:k + 8] * W[None, :, k:k + 8])
            c1 = c + hc[:, k:k + 8] @ W[:, k:k + 8].T
            e += 9.0 * U_TZ * passes * (np.maximum(np.abs(c), np.abs(c1)) + p.max(2) + 2.0 ** -9 * p.sum(2))
            c = c1
        if mode != 1:
            e += 4.0 * U_RN * (np.abs(hc) @ np.abs(W).T + np.abs(b))
        out[i:i + chunk] = e
    return out


def _tanh_err(mode, h):
    """Error a tanh evaluation adds to an exact pre-activation, as a bound on |tanh_kernel(a) - tanh(a)|."""
    if mode == 0:
        # tanhf: at most 2 ulp (CUDA math library table; glibc's tanhf likewise) -> 2 * 2^-23 |h|, plus the smallest
        # normal as absolute floor (subnormal results)
        return 2.0 * 2.0 ** -23 * np.abs(h) + 2.0 ** -126
    if mode in (1, 3):
        # 1 - 2 rcp(ex2(2 x log2 e) + 1):  ex2.approx relative 2^-22 -> 2 r(1 - r) 2^-22 <= 2^-23 absolute; e + 1 rounded
        # and rcp.approx (1 ulp) -> 2 r (2^-24 + 2^-23) <= 3 * 2^-23; final fma 2^-24; the argument 2 x log2 e carries
        # 2 * 2^-24 relative (constant and product), which tanh damps to x sech^2(x) 2^-23 <= 0.45 * 2^-23.
        # Total < 5 * 2^-23 (a flushed subnormal argument gives tanh = 0: off by less than 2^-126).
        return np.full_like(h, 5.0 * 2.0 ** -23)
    if mode == 2:
        # tanh.approx.f32: maximum absolute error 2^-10.987 over the whole range (PTX ISA)
        return np.full_like(h, 2.0 ** -10.987)
    raise ValueError(mode)


def _through_tanh(a, e_pre, mode):
    """Bound on |tanh_kernel(a + d) - tanh(a)| for |d| <= e_pre: the mean-value theorem with the largest sech^2 on
    [a - e_pre, a + e_pre], plus the evaluation error of tanh itself; never more than the range 2 + that error."""
    lo = np.minimum(np.maximum(np.abs(a) - e_pre, 0.0), 300.0)
    prop = np.minimum(e_pre / np.cosh(lo) ** 2, 2.0)
    return prop + _tanh_err(mode, np.tanh(a))


def _layer(mode, h, eh, W, b):
    """(exact pre-activation, its error bound) of h @ W.T + b."""
    a = h @ W.T + b
    e = _prod(mode) * (np.abs(h) @ np.abs(W).T) + _acc(mode, h, W, b) + eh @ np.abs(W).T
    # subnormal partial products / sums that a flushing unit may drop: 2^-126 per addend
    return a, e + 2.0 ** -126 * 3 * (h.shape[1] + 8)


def bound(w, x, mode):
    """Bound [n,4] on |kernel - forward64| for the unclipped mean (columns 0..2) and the value (column 3) of
    r6_policy* with tensor_cores = mode.  Value column 0 without a critic (the kernels write exact zeros)."""
    x = np.asarray(x, np.float32).astype(np.float64).reshape(-1, 13)
    W = {k: np.asarray(v, np.float32).astype(np.float64) for k, v in w.items() if v is not None}
    # the observations are exact float32 inputs: layer 0 carries no error in
    a0, e0 = _layer(mode, x, np.zeros_like(x), W["w0"], W["b0"])
    h0, eh0 = np.tanh(a0), _through_tanh(a0, e0, mode)
    a1, e1 = _layer(mode, h0, eh0, W["w1"], W["b1"])
    h1, eh1 = np.tanh(a1), _through_tanh(a1, e1, mode)
    W2, b2 = W["w2"], W["b2"]
    if "wv" in W:
        W2 = np.concatenate([W2, W["wv"].reshape(1, 64)], 0)
        b2 = np.concatenate([b2, W["bv"].reshape(1)])
    _, e2 = _layer(mode, h1, eh1, W2, b2)
    out = np.zeros((len(x), 4))
    out[:, :W2.shape[0]] = e2
    return out


# ---- weight families ---------------------------------------------------------------------------------------------------
def _orthogonal(rng, rows, cols, gain):
    """torch.nn.init.orthogonal_ (what SB3's ortho_init calls): QR of a Gaussian matrix, sign-fixed by diag(R)."""
    a = rng.standard_normal((rows, cols))
    t = rows < cols
    if t:
        a = a.T
    q, r = np.linalg.qr(a)
    q = q * np.sign(np.diag(r))
    if t:
        q = q.T
    return (gain * q).astype(np.float32)


def _sb3_init(rng):
    """SB3 ActorCriticPolicy at construction (ortho_init=True): sqrt(2) on the shared trunk, 0.01 on action_net,
    1 on value_net, zero biases, log_std 0 — the network PPO collects its first rollout with."""
    g = np.sqrt(2.0)
    return {"w0": _orthogonal(rng, 128, 13, g), "b0": np.zeros(128, np.float32),
            "w1": _orthogonal(rng, 64, 128, g), "b1": np.zeros(64, np.float32),
            "w2": _orthogonal(rng, 3, 64, 0.01), "b2": np.zeros(3, np.float32),
            "wv": _orthogonal(rng, 1, 64, 1.0).reshape(64), "bv": np.zeros(1, np.float32),
            "log_std": np.zeros(3, np.float32)}


def _tf32_edge(rng, a):
    """Replace entries of a float32 array by TF32 edge cases: low 13 mantissa bits exactly 0x1000 (a tie of
    round_tf32), low 13 bits zero (exactly TF32, lo = 0), +-0.0, and magnitudes below 2^-100; a fifth stay as drawn."""
    a = np.array(a, np.float32)
    b = a.view(np.uint32)
    kind = rng.integers(0, 5, a.shape)
    b[kind == 0] = (b[kind == 0] & np.uint32(0xFFFFE000)) | np.uint32(0x1000)
    b[kind == 1] &= np.uint32(0xFFFFE000)
    z = kind == 2
    a[z] = np.where(rng.random(z.sum()) < 0.5, np.float32(0.0), np.float32(-0.0))
    t = kind == 3
    a[t] = (rng.choice([-1.0, 1.0], t.sum()) * rng.uniform(1.0, 2.0, t.sum()) * 2.0 ** rng.integers(-126, -100, t.sum())).astype(np.float32)
    return a


def weights(family, seed=0):
    """float32 actor-critic weights (w0..b2, wv, bv, log_std) of one family."""
    rng = np.random.default_rng(seed + 1000 * FAMILIES.index(family))
    if family == "golden":
        g = np.load(GOLD)
        w = {k: np.ascontiguousarray(g["mlp_" + k], np.float32) for k in ("w0", "b0", "w1", "b1", "w2", "b2")}
        r5 = np.random.default_rng(5)                # the critic head of tests/test_gpu_policy.py::_actor_critic_weights
        w["wv"] = (r5.standard_normal(64) * 0.3).astype(np.float32)
        w["bv"] = np.array([0.7], np.float32)
        w["log_std"] = np.array([-0.5, -1.0, 0.2], np.float32)
        return w
    w = _sb3_init(rng)
    if family == "sb3_init":
        return w
    if family == "saturating":
        # |pre-activations| mostly > 10 with both signs: the overflow / underflow branches of the exp2 form of tanh
        # (w0 is 128 x 13 with orthonormal columns: its rows have norm ~0.45 against 1.4 for w1, hence 4 x more)
        w["w0"] = (w["w0"] * 64).astype(np.float32)
        w["w1"] = (w["w1"] * 16).astype(np.float32)
        w["b0"] = rng.uniform(-4, 4, 128).astype(np.float32)
        w["b1"] = rng.uniform(-4, 4, 64).astype(np.float32)
        w["w2"] = (w["w2"] * 50).astype(np.float32)            # outputs of order 1, so the clip is exercised
        w["log_std"] = np.array([0.3, -0.7, 1.0], np.float32)
        return w
    if family == "tf32_edges":
        for k in ("w0", "w1", "wv"):
            w[k] = _tf32_edge(rng, w[k])
        w["w2"] = _tf32_edge(rng, w["w2"] * 60)
        for k, n in (("b0", 128), ("b1", 64), ("b2", 3)):
            w[k] = _tf32_edge(rng, rng.uniform(-0.5, 0.5, n).astype(np.float32))
        w["bv"] = np.array([0.25], np.float32)
        w["log_std"] = np.array([-5.0, 0.0, 2.0], np.float32)
        return w
    raise ValueError(family)


def obs_sets(n, seed=0):
    """{name: float32 [n,13]}: the golden closed-loop observations (cycled to n rows), U(-1, 1) and N(0, 5^2).  (The
    GPU tests add the observations of a closed-loop rollout of the device.)"""
    rng = np.random.default_rng(seed)
    g = np.load(GOLD)["obs"][:, :13].astype(np.float32)
    return {"golden": g[np.arange(n) % len(g)],
            "uniform": rng.uniform(-1, 1, (n, 13)).astype(np.float32),
            "normal5": (5.0 * rng.standard_normal((n, 13))).astype(np.float32)}


# One constant for every mode and family: a kernel passes when |kernel - forward64| <= C_BAR * bound(w, x, mode).  The
# bound is a worst case (every rounding error at its maximum, all with the same sign), so a correct kernel sits well
# below it; C_BAR = 2 leaves room only for a first-order term the analysis neglects.
C_BAR = 2.0


def round_tf32(a):
    """round_tf32 of r6_mlp_tcgen05.cuh (nearest TF32, ties away from zero) on float32 values, returned as float64."""
    b = np.asarray(a, np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32).astype(np.float64)
