// r6_ppo.cuh — per-sample math of the PPO update (stable-baselines3 1.6.0 `PPO.train`, main_6DOF.py:136): one
// sample's forward pass, its contribution to the clipped-surrogate + value + entropy loss, and the backward pass
// through the shared-trunk actor-critic (13 -> 128 -> 64 tanh, action_net 64 -> 3, value_net 64 -> 1, state-independent
// log_std).  Compiled for the device (r6_ppo_grad) and, for tests/ppo_hostsim only, for the host.
//
// The loss, from memory of SB3 1.6.0 PPO.train [memory]:
//     logp   = sum_j -(a_j - mean_j)^2 / (2 sigma_j^2) - log sigma_j - log sqrt(2 pi),  sigma = exp(log_std),
//              on the stored UNclipped action
//     ratio  = exp(logp - old_logp),   A' = (A - mu_B) * inv_std_B when the advantages are normalised
//     pg     = -min(A' ratio, A' clip(ratio, 1 - eps, 1 + eps))
//     vloss  = (R - v)^2
//     loss   = pg + vf_coef vloss - ent_coef entropy,   entropy = sum_j (log sigma_j + 1/2 + log sqrt(2 pi))
// Gradient (torch.min / clamp semantics): d pg / d logp = -A' ratio when the unclipped branch is the minimum (always so
// for ratio inside [1 - eps, 1 + eps]), else 0; d logp / d mean_j = (a_j - mean_j) / sigma_j^2,
// d logp / d log_std_j = (a_j - mean_j)^2 / sigma_j^2 - 1; the entropy adds -ent_coef to every d / d log_std_j.
#pragma once

#include "r6_core.cuh"

namespace r6 {

// flat parameter layout of include/r6dof.h (SB3 [out][in] order)
constexpr int kPpoOffW0 = 0, kPpoOffB0 = 1664, kPpoOffW1 = 1792, kPpoOffB1 = 9984, kPpoOffW2 = 10048,
              kPpoOffB2 = 10240, kPpoOffWv = 10243, kPpoOffBv = 10307, kPpoOffLogStd = 10308, kPpoParams = 10311;
static_assert(kPpoParams == R6_PPO_NPARAMS, "flat layout");
static_assert(kPpoOffB0 == kMlpH0 * kMlpIn && kPpoOffW1 == kPpoOffB0 + kMlpH0 && kPpoOffB1 == kPpoOffW1 + kMlpH1 * kMlpH0 &&
              kPpoOffW2 == kPpoOffB1 + kMlpH1 && kPpoOffB2 == kPpoOffW2 + 3 * kMlpH1 && kPpoOffWv == kPpoOffB2 + 3 &&
              kPpoOffBv == kPpoOffWv + kMlpH1 && kPpoOffLogStd == kPpoOffBv + 1 && kPpoOffW1 % 4 == 0, "flat layout");

// per-sample gradient w.r.t. the network outputs: g[0..2] = d/d mean, g[3] = d/d value, g[4..6] = d/d log_std
struct PpoHead {
    float g[7];
    float pg, vloss, clipped, kl;
};

// The forward pass of mlp_forward (same packed weights, same operation order, so the mode-0 error bound of the policy
// kernels applies) that also hands out the hidden activations h0[j * st] (128 units) and h1[k * st] (64 units).
R6_HD void ppo_forward(const float *W, const float *x, float *h0, float *h1s, int st, float (&out)[4])
{
    float h1[kMlpH1];
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) h1[k] = 0.0f;
#pragma unroll 2
    for (int j = 0; j < kMlpH0; j++) {
        const F4 wa = ld4(W + j * 16), wb = ld4(W + j * 16 + 4), wc = ld4(W + j * 16 + 8), wd = ld4(W + j * 16 + 12);
        float s = wa.x * x[0];
        s = f32_fma(wa.y, x[1], s); s = f32_fma(wa.z, x[2], s); s = f32_fma(wa.w, x[3], s);
        s = f32_fma(wb.x, x[4], s); s = f32_fma(wb.y, x[5], s); s = f32_fma(wb.z, x[6], s); s = f32_fma(wb.w, x[7], s);
        s = f32_fma(wc.x, x[8], s); s = f32_fma(wc.y, x[9], s); s = f32_fma(wc.z, x[10], s); s = f32_fma(wc.w, x[11], s);
        s = f32_fma(wd.x, x[12], s);
        const float h = tanhf(s + wd.y);
        h0[j * st] = h;
        const float *w1 = W + kMlpOffW1 + j * kMlpH1;
#pragma unroll
        for (int k = 0; k < kMlpH1; k += 4) {
            const F4 w = ld4(w1 + k);
            h1[k] = f32_fma(w.x, h, h1[k]); h1[k + 1] = f32_fma(w.y, h, h1[k + 1]);
            h1[k + 2] = f32_fma(w.z, h, h1[k + 2]); h1[k + 3] = f32_fma(w.w, h, h1[k + 3]);
        }
    }
    // layer 1 goes through h1s (pre-activation, then activation): a fully unrolled tanh loop over registers would keep
    // far more than the 64 accumulators live
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) h1s[k * st] = h1[k];
    float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f, o3 = 0.0f;
#pragma unroll 4
    for (int k = 0; k < kMlpH1; k++) {
        const float h = tanhf(h1s[k * st] + W[kMlpOffB1 + k]);
        h1s[k * st] = h;
        o0 = f32_fma(W[kMlpOffW2 + k], h, o0);
        o1 = f32_fma(W[kMlpOffW2 + kMlpH1 + k], h, o1);
        o2 = f32_fma(W[kMlpOffW2 + 2 * kMlpH1 + k], h, o2);
        o3 = f32_fma(W[kMlpOffW2 + 3 * kMlpH1 + k], h, o3);
    }
    out[0] = o0 + W[kMlpOffB2];
    out[1] = o1 + W[kMlpOffB2 + 1];
    out[2] = o2 + W[kMlpOffB2 + 2];
    out[3] = o3 + W[kMlpOffB2 + 3];
}

// A' from the raw advantage: (A - mu) * inv_std in float64, rounded once (stats = NULL: A itself)
R6_HD float ppo_advantage(float A, const double *stats)
{
    return stats != nullptr ? f64_to_f32(((double)A - stats[0]) * stats[1]) : A;
}

// loss terms and output gradients of one sample (out = mean[0..2], value)
R6_HD void ppo_head(const float (&out)[4], const float *a, float old_logp, float adv, float ret, const float *log_std,
                    float clip, float vf_coef, float ent_coef, PpoHead &h)
{
    // division-free: z = (a - mean) / sigma with 1 / sigma = exp(-log_std) (a division's slow path is a call, and
    // everything live across it would spill)
    float z[3], isg[3], logp = 0.0f;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        isg[j] = expf(-log_std[j]);
        z[j] = (a[j] - out[j]) * isg[j];
        logp += -0.5f * (z[j] * z[j]) - log_std[j] - 0.9189385332046727f;      // log sqrt(2 pi)
    }
    const float lr = logp - old_logp;
    const float ratio = expf(lr);
    const float rc = fminf(fmaxf(ratio, 1.0f - clip), 1.0f + clip);
    const float s1 = adv * ratio, s2 = adv * rc;
    h.pg = -fminf(s1, s2);
    const float w = s1 <= s2 ? -s1 : 0.0f;                 // d pg / d logp: the unclipped branch only
#pragma unroll
    for (int j = 0; j < 3; j++) {
        h.g[j] = w * (z[j] * isg[j]);
        h.g[4 + j] = w * f32_fma(z[j], z[j], -1.0f) - ent_coef;
    }
    const float e = out[3] - ret;
    h.g[3] = 2.0f * vf_coef * e;
    h.vloss = e * e;
    h.clipped = fabsf(ratio - 1.0f) > clip ? 1.0f : 0.0f;
    h.kl = (ratio - 1.0f) - lr;
}

// delta1_k = (sum_c W2[c][k] g_c + wv_k g_v) (1 - h1_k^2), from h1[k * st] into d1[k * st]
R6_HD void ppo_delta1(const float *W, const PpoHead &h, const float *h1, float *d1, int st)
{
#pragma unroll 4
    for (int k = 0; k < kMlpH1; k++) {
        float s = W[kMlpOffW2 + k] * h.g[0];
        s = f32_fma(W[kMlpOffW2 + kMlpH1 + k], h.g[1], s);
        s = f32_fma(W[kMlpOffW2 + 2 * kMlpH1 + k], h.g[2], s);
        s = f32_fma(W[kMlpOffW2 + 3 * kMlpH1 + k], h.g[3], s);
        const float hk = h1[k * st];
        d1[k * st] = s * f32_fma(-hk, hk, 1.0f);
    }
}

// delta0_j = (sum_k W1[k][j] delta1_k) (1 - h0_j^2)   (W1 stored transposed in the packed block: row j contiguous)
R6_HD float ppo_delta0(const float *W, int j, const float (&d1)[kMlpH1], float h0)
{
    const float *w1 = W + kMlpOffW1 + j * kMlpH1;
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < kMlpH1; k += 4) {
        const F4 w = ld4(w1 + k);
        s = f32_fma(w.x, d1[k], s); s = f32_fma(w.y, d1[k + 1], s);
        s = f32_fma(w.z, d1[k + 2], s); s = f32_fma(w.w, d1[k + 3], s);
    }
    return s * f32_fma(-h0, h0, 1.0f);
}

// clip_grad_norm_'s factor min(1, max_norm / (norm + 1e-6)) as torch forms it (a float32 tensor); 1 when max_norm <= 0
R6_HD float clip_coef(double max_norm, double norm)
{
    return max_norm > 0.0 ? fminf(f64_to_f32(max_norm / (norm + 1e-6)), 1.0f) : 1.0f;
}

// the per-step constants of adam_element: c = (1 - beta1, beta2, 1 - beta2, lr / (1 - beta1^step),
// sqrt(1 - beta2^step), eps), the bias corrections in float64 like torch's Python scalars
R6_HD void adam_coefs(const R6AdamCoef &a, int64_t step, float (&c)[6])
{
    const double bc1 = 1.0 - pow(a.beta1, (double)step), bc2 = 1.0 - pow(a.beta2, (double)step);
    c[0] = f64_to_f32(1.0 - a.beta1);
    c[1] = f64_to_f32(a.beta2);
    c[2] = f64_to_f32(1.0 - a.beta2);
    c[3] = f64_to_f32(a.lr / bc1);
    c[4] = f64_to_f32(sqrt(bc2));
    c[5] = f64_to_f32(a.eps);
}

// One parameter of torch.optim.Adam (foreach and single-tensor forms compute the same): g already scaled and clipped,
// c from adam_coefs
R6_HD void adam_element(float &p, float &m, float &v, float g, const float (&c)[6])
{
    m = f32_fma(c[0], g - m, m);                         // lerp(m, g, 1 - beta1) for a weight < 0.5
    v = f32_fma(c[2], g * g, v * c[1]);
    const float denom = f32_sqrt(v) / c[4] + c[5];
    p = f32_fma(-c[3], m / denom, p);
}

}  // namespace r6
