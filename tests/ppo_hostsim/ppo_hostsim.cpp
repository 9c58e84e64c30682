// ppo_hostsim.cpp — TEST-ONLY host compilation of rl_rocket_6dof_b200/csrc/r6_ppo.cuh (the per-sample PPO loss and
// gradient, and the Adam step of r6_adam_step), built by tests/ppo_hostsim/__init__.py with g++ into
// tests/ppo_hostsim/_build/.  Lets the CPU test-suite check the kernels' per-sample math against float64 autograd and
// torch Adam; never imported, linked or shipped by the product package.
#include "../../rl_rocket_6dof_b200/csrc/r6_ppo.cuh"

using namespace r6;

extern "C" {

// per-sample gradient over the flat parameters (grad [n][R6_PPO_NPARAMS]; weight entries are the float32 products of
// the kernel's accumulation, unsummed) and loss terms [n][4] (pg, vloss, clipped, kl), for obs13 [n][13], act3 [n][3]
// and old_logp / adv / ret [n]; adv_stats NULL or (mean, inv_std)
int hs_ppo_nparams(void) { return kPpoParams; }
void hs_ppo_sample_grad(const float *params, const float *obs13, const float *act3, const float *old_logp, const float *adv,
                        const float *ret, int64_t n, const double *adv_stats, float clip, float vf_coef, float ent_coef,
                        float *grad, float *terms)
{
    const R6Mlp m = {params + kPpoOffW0, params + kPpoOffB0, params + kPpoOffW1, params + kPpoOffB1, params + kPpoOffW2,
                     params + kPpoOffB2, params + kPpoOffWv, params + kPpoOffBv, params + kPpoOffLogStd};
    static float W[kMlpFloats];
    for (int i = 0; i < kMlpFloats; i++) W[i] = mlp_pack_element(m, i);
    for (int64_t s = 0; s < n; s++) {
        const float *x = obs13 + 13 * s;
        float h0[kMlpH0], h1[kMlpH1], d1[kMlpH1], out[4];
        ppo_forward(W, x, h0, h1, 1, out);
        PpoHead hd;
        ppo_head(out, act3 + 3 * s, old_logp[s], ppo_advantage(adv[s], adv_stats), ret[s], m.log_std, clip, vf_coef, ent_coef, hd);
        ppo_delta1(W, hd, h1, d1, 1);
        float *g = grad + s * kPpoParams;
        for (int j = 0; j < kMlpH0; j++) {
            const float d0 = ppo_delta0(W, j, d1, h0[j]);
            for (int c = 0; c < kMlpIn; c++) g[kPpoOffW0 + j * kMlpIn + c] = d0 * x[c];
            g[kPpoOffB0 + j] = d0;
        }
        for (int k = 0; k < kMlpH1; k++) {
            for (int j = 0; j < kMlpH0; j++) g[kPpoOffW1 + k * kMlpH0 + j] = d1[k] * h0[j];
            g[kPpoOffB1 + k] = d1[k];
            for (int c = 0; c < 3; c++) g[kPpoOffW2 + c * kMlpH1 + k] = hd.g[c] * h1[k];
            g[kPpoOffWv + k] = hd.g[3] * h1[k];
        }
        for (int c = 0; c < 3; c++) {
            g[kPpoOffB2 + c] = hd.g[c];
            g[kPpoOffLogStd + c] = hd.g[4 + c];
        }
        g[kPpoOffBv] = hd.g[3];
        terms[4 * s] = hd.pg; terms[4 * s + 1] = hd.vloss; terms[4 * s + 2] = hd.clipped; terms[4 * s + 3] = hd.kl;
    }
}

// r6_adam_step on the host: the same norm, clip factor and per-parameter update
void hs_adam_step(float *p, const float *grad_sum, float *m, float *v, int64_t P, const R6AdamCoef *coef, int64_t step,
                  double *norm_out)
{
    const float scale = (float)coef->scale;
    double t = 0.0;
    for (int64_t i = 0; i < P; i++) { const double g = (double)(scale * grad_sum[i]); t += g * g; }
    const double norm = sqrt(t);
    const float cc = clip_coef(coef->max_grad_norm, norm);
    float c[6];
    adam_coefs(*coef, step, c);
    for (int64_t i = 0; i < P; i++) adam_element(p[i], m[i], v[i], (scale * grad_sum[i]) * cc, c);
    *norm_out = norm;
}

}  // extern "C"
