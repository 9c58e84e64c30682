// sde_hostsim.cpp — TEST-ONLY host compilation of the gSDE math of rl_rocket_6dof_b200/csrc/r6_core.cuh (the noise draw,
// sde_noise_block) and csrc/r6_ppo.cuh (r6_ppo_grad_sde's per-sample loss and gradient), built by
// tests/sde_hostsim/__init__.py with g++ into tests/sde_hostsim/_build/.  Lets the CPU test-suite check them against
// their NumPy / float64 autograd restatements; never imported, linked or shipped by the product package.
#include "../../rl_rocket_6dof_b200/csrc/r6_ppo.cuh"

using namespace r6;

extern "C" {

// gSDE noise draw per env: xi [n][192] (component c = 3 k + a) for global env ids genv [n] and one draw step
void hs_sde_noise(uint64_t seed, const uint64_t *genv, uint64_t step, int64_t n, float *xi)
{
    for (int64_t i = 0; i < n; i++)
        for (int b = 0; b < kSdeBlocks; b++) {
            float z[4];
            sde_noise_block(seed, genv[i], step, b, z);
            for (int q = 0; q < 4; q++) xi[i * kSdeXi + 4 * b + q] = z[q];
        }
}

// r6_ppo_grad_sde's per-sample math: params [R6_PPO_NPARAMS_SDE], grad [n][R6_PPO_NPARAMS_SDE] (weight entries are the
// float32 products of the kernel's accumulation, unsummed; the log_std entries are sigma^2 (r_a h_k^2)), terms [n][5]
// (pg, vloss, clipped, kl, entropy), for obs13 [n][13], act3 [n][3] and old_logp / adv / ret [n]
int hs_ppo_sde_nparams(void) { return kPpoParamsSde; }
void hs_ppo_sde_sample_grad(const float *params, const float *obs13, const float *act3, const float *old_logp,
                            const float *adv, const float *ret, int64_t n, const double *adv_stats, float clip, float vf_coef,
                            float ent_coef, float *grad, float *terms)
{
    const R6Mlp m = {params + kPpoOffW0, params + kPpoOffB0, params + kPpoOffW1, params + kPpoOffB1, params + kPpoOffW2,
                     params + kPpoOffB2, params + kPpoOffWv, params + kPpoOffBv, nullptr};
    static float W[kMlpFloats];
    for (int i = 0; i < kMlpFloats; i++) W[i] = mlp_pack_element(m, i);
    float sig2[kSdeXi];
    for (int c = 0; c < kSdeXi; c++) { const float sg = expf(params[kPpoOffLogStd + c]); sig2[c] = sg * sg; }
    for (int64_t s = 0; s < n; s++) {
        const float *x = obs13 + 13 * s;
        float h0[kMlpH0], h1[kMlpH1], d1[kMlpH1], out[4], var[3];
        ppo_forward(W, x, h0, h1, 1, out);
        sde_latent_var(h1, 1, sig2, var);
        PpoHeadSde hd;
        ppo_head_sde(out, act3 + 3 * s, old_logp[s], ppo_advantage(adv[s], adv_stats), ret[s], var, clip, vf_coef, ent_coef, hd);
        ppo_delta1(W, hd, h1, d1, 1);
        float *g = grad + s * kPpoParamsSde;
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
            for (int c = 0; c < 3; c++) g[kPpoOffLogStd + 3 * k + c] = sig2[3 * k + c] * (hd.g[4 + c] * (h1[k] * h1[k]));
        }
        for (int c = 0; c < 3; c++) g[kPpoOffB2 + c] = hd.g[c];
        g[kPpoOffBv] = hd.g[3];
        float *t = terms + 5 * s;
        t[0] = hd.pg; t[1] = hd.vloss; t[2] = hd.clipped; t[3] = hd.kl; t[4] = hd.ent;
    }
}

}  // extern "C"
