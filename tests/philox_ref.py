"""Independent NumPy statement of the device RNG contract (include/r6dof.h, r6_reset / r6_rollout):
Philox4x32-10, key = seed, counter = (global env id lo, hi, a, b).  Used to check the CUDA reset
sampler and the synthetic action stream bit-for-bit."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
STREAM_RESET = 0x52534554
STREAM_ACTION = 0x41435431


def philox4x32_10(ctr, key):
    """ctr: uint32 [..., 4], key: (k0, k1) -> uint32 [..., 4]"""
    c = np.array(ctr, dtype=np.uint32, copy=True)
    k0, k1 = np.uint32(key[0]), np.uint32(key[1])
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = M0 * c[..., 0].astype(np.uint64)
            p1 = M1 * c[..., 2].astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), p0.astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), p1.astype(np.uint32)
            n = np.empty_like(c)
            n[..., 0] = hi1 ^ c[..., 1] ^ k0
            n[..., 1] = lo1
            n[..., 2] = hi0 ^ c[..., 3] ^ k1
            n[..., 3] = lo0
            c = n
            k0 = np.uint32(k0 + W0)
            k1 = np.uint32(k1 + W1)
    return c


def u53(a, b):
    return ((a >> np.uint32(5)).astype(np.float64) * 67108864.0 + (b >> np.uint32(6)).astype(np.float64)) / 9007199254740992.0


def sample_ic(ic_low, ic_high, seed, genv, episode):
    """Box.sample for global env ids `genv` (int64 array) and episode counters -> float32 [n,14]
    BEFORE the quaternion normalisation."""
    genv = np.asarray(genv, np.uint64)
    episode = np.broadcast_to(np.asarray(episode, np.uint32), genv.shape)
    lo, hi = np.asarray(ic_low, np.float32).astype(np.float64), np.asarray(ic_high, np.float32).astype(np.float64)
    out = np.zeros(genv.shape + (14,), np.float32)
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    for b in range(7):
        ctr = np.stack([(genv & np.uint64(0xFFFFFFFF)).astype(np.uint32), (genv >> np.uint64(32)).astype(np.uint32),
                        episode, np.full(genv.shape, STREAM_RESET + b, np.uint32)], -1)
        r = philox4x32_10(ctr, key)
        ua, ub = u53(r[..., 0], r[..., 1]), u53(r[..., 2], r[..., 3])
        i = 2 * b
        out[..., i] = (lo[i] + (hi[i] - lo[i]) * ua).astype(np.float32)
        out[..., i + 1] = (lo[i + 1] + (hi[i + 1] - lo[i + 1]) * ub).astype(np.float32)
    return out


def normalize_ic_quaternion(ic):
    """rocket_env.py:190 in float32 (sdot rule: f32 products, f64 accumulation, f32 rounding)."""
    ic = np.array(ic, np.float32, copy=True)
    q = ic[..., 6:10]
    acc = (q * q).astype(np.float64).sum(-1)
    n = np.sqrt(acc.astype(np.float32))
    ic[..., 6:10] = q / n[..., None]
    return ic


def actions(seed, genv, step):
    """uniform(-1,1) float32 actions of r6_rollout's R6_ACT_PHILOX for (global env, global step)."""
    genv = np.asarray(genv, np.uint64)
    step = np.broadcast_to(np.asarray(step, np.uint64), genv.shape)
    ctr = np.stack([(genv & np.uint64(0xFFFFFFFF)).astype(np.uint32), (genv >> np.uint64(32)).astype(np.uint32),
                    (step & np.uint64(0xFFFFFFFF)).astype(np.uint32),
                    np.uint32(STREAM_ACTION) ^ (step >> np.uint64(32)).astype(np.uint32)], -1)
    r = philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    return (-1.0 + 2.0 * ((r[..., :3].astype(np.float64) + 0.5) / 4294967296.0)).astype(np.float32)


STREAM_POLICY = 0x50414354          # 'PACT': Gaussian exploration noise of the policy kernels (r6_core.cuh gaussian_head)


def policy_block(seed, genv, step):
    """The Philox block of gaussian_head for (global env, global step): uint32 [..., 4]."""
    genv = np.asarray(genv, np.uint64)
    step = np.broadcast_to(np.asarray(step, np.uint64), genv.shape)
    ctr = np.stack([(genv & np.uint64(0xFFFFFFFF)).astype(np.uint32), (genv >> np.uint64(32)).astype(np.uint32),
                    (step & np.uint64(0xFFFFFFFF)).astype(np.uint32),
                    np.uint32(STREAM_POLICY) ^ (step >> np.uint64(32)).astype(np.uint32)], -1)
    return philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))


def policy_uniforms(r):
    """The four float32 uniforms gaussian_head forms from a block, with its float32 roundings:
    u1, u3 = ((r >> 8) + 0.5f) * 2^-24 in (0, 1] (k + 0.5 rounds to even for k >= 2^23, so the top value is 1.0),
    u2, u4 = float(r) * 2^-32 in [0, 1] (the uint32 -> float conversion rounds to nearest, so 1.0 occurs)."""
    r = np.asarray(r, np.uint32)
    half = np.float32(0.5)
    u1 = ((r[..., 0] >> np.uint32(8)).astype(np.float32) + half) * np.float32(1.0 / 16777216.0)
    u3 = ((r[..., 2] >> np.uint32(8)).astype(np.float32) + half) * np.float32(1.0 / 16777216.0)
    u2 = r[..., 1].astype(np.float32) * np.float32(1.0 / 4294967296.0)
    u4 = r[..., 3].astype(np.float32) * np.float32(1.0 / 4294967296.0)
    return u1, u2, u3, u4


def policy_noise(seed, genv, step):
    """Standard-normal eps [..., 3] of the stochastic policy head for (seed, global env, global step): Box-Muller on the
    kernel's float32 uniforms in float64,
        z0 = sqrt(-2 ln u1) cos(2 pi u2),  z1 = sqrt(-2 ln u1) sin(2 pi u2),  z2 = sqrt(-2 ln u3) cos(2 pi u4)."""
    u1, u2, u3, u4 = (u.astype(np.float64) for u in policy_uniforms(policy_block(seed, genv, step)))
    ra = np.sqrt(-2.0 * np.log(u1))
    rb = np.sqrt(-2.0 * np.log(u3))
    return np.stack([ra * np.cos(2 * np.pi * u2), ra * np.sin(2 * np.pi * u2), rb * np.cos(2 * np.pi * u4)], -1)


def policy_noise_bar(z, seed, genv, step):
    """Bound on |z_kernel - policy_noise| (both builds of gaussian_head).  logf 1 ulp -> 2^-24 relative in the root,
    sqrtf 0.5 ulp, sincospif / cospif 1 ulp (the host build: double precision rounded, 0.5 ulp), the product 0.5 ulp:
    |dz| <= 3 * 2^-23 |z|, plus the float64 reference's own error where sin / cos(2 pi u) vanish (2 pi u rounded in
    double: < 2^-48 of the radius)."""
    u1, _, u3, _ = (u.astype(np.float64) for u in policy_uniforms(policy_block(seed, genv, step)))
    r = np.stack([np.sqrt(-2.0 * np.log(u1))] * 2 + [np.sqrt(-2.0 * np.log(u3))], -1)
    return 3 * 2.0 ** -23 * np.abs(z) + 2.0 ** -48 * r


LOG_SQRT_2PI = 0.5 * np.log(2.0 * np.pi)


def log_prob_at_mean(log_std):
    """gaussian_head's float32 log-prob of a deterministic action (z = 0), summed in its order:
    sum_i (-log_std_i - ln(2 pi) / 2) with the constant 0.9189385f."""
    c = np.float32(0.9189385332046727)
    acc = np.float32(0.0)
    for i in range(3):
        li = np.float32(0.0) if log_std is None else np.float32(log_std[i])
        acc = np.float32(acc + np.float32(np.float32(-li) - c))
    return acc


def gaussian_log_prob(z, log_std):
    """SB3 DiagGaussianDistribution.log_prob of mean + std * z in float64: sum_i (-z_i^2 / 2 - log_std_i - ln(2 pi) / 2)."""
    z = np.asarray(z, np.float64)
    ls = np.zeros(3) if log_std is None else np.asarray(log_std, np.float32).astype(np.float64)
    return (-0.5 * z * z - ls - LOG_SQRT_2PI).sum(-1)
