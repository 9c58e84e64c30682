// sepsde_hostsim.cpp — TEST-ONLY host compilation of the per-sample math of ppo_grad_sep_sde_kernel
// (rl_rocket_6dof_b200/csrc/r6_ppo.cuh: ppo_forward_sep, sde_latent_var on the policy latent, ppo_head_sde, ppo_value_clip,
// ppo_delta1_sep, ppo_delta0), built by tests/sepsde_hostsim/__init__.py with g++ into tests/sepsde_hostsim/_build/.
// Never imported, linked or shipped by the product package.
#include "../../rl_rocket_6dof_b200/csrc/r6_ppo.cuh"

using namespace r6;

extern "C" {

int hs_sepsde_nparams(void) { return kPpoParamsSepSde; }

// params [R6_PPO_NPARAMS_SEP_SDE]; grad [n][R6_PPO_NPARAMS_SEP_SDE] (the float32 products of the kernel's accumulation,
// unsummed; log_std entries sigma^2 (r_a hp_k^2)), terms [n][5] (pg, vloss, clipped, kl, entropy), for obs13 [n][13],
// act3 [n][3], old_logp / adv / ret [n]; vfc > 0 clips the value around vold [n] (nullable otherwise)
void hs_sepsde_sample_grad(const float *params, const float *obs13, const float *act3, const float *old_logp,
                           const float *adv, const float *ret, const float *vold, int64_t n, const double *adv_stats,
                           float clip, float vf_coef, float ent_coef, float vfc, float *grad, float *terms)
{
    R6Mlp m = {params + kSepOffW0, params + kSepOffB0, params + kSepOffW1, params + kSepOffB1, params + kSepOffW2,
               params + kSepOffB2, params + kSepOffWv, params + kSepOffBv, nullptr};
    m.vf_w0 = params + kSepOffVw0; m.vf_b0 = params + kSepOffVb0; m.vf_w1 = params + kSepOffVw1; m.vf_b1 = params + kSepOffVb1;
    static float W[kMlpFloatsSep];
    for (int i = 0; i < kMlpFloatsSep; i++) W[i] = mlp_pack_element_sep(m, i);
    float sig2[kSdeXi];
    for (int c = 0; c < kSdeXi; c++) { const float sg = expf(params[kSepOffLogStd + c]); sig2[c] = sg * sg; }
    for (int64_t s = 0; s < n; s++) {
        const float *x = obs13 + 13 * s;
        float h0[kMlpH0], hp[kMlpH1], hv[kMlpH1], out[4], var[3];
        ppo_forward_sep(W, x, h0, hp, hv, 1, out);
        sde_latent_var(hp, 1, sig2, var);
        PpoHeadSde hd;
        ppo_head_sde(out, act3 + 3 * s, old_logp[s], ppo_advantage(adv[s], adv_stats), ret[s], var, clip, vf_coef, ent_coef, hd);
        if (vfc > 0.0f) ppo_value_clip(out[3], vold[s], ret[s], vfc, vf_coef, hd);
        float *g = grad + s * kPpoParamsSepSde;
        for (int k = 0; k < kMlpH1; k++) {
            for (int c = 0; c < 3; c++) g[kSepOffW2 + c * kMlpH1 + k] = hd.g[c] * hp[k];
            g[kSepOffWv + k] = hd.g[3] * hv[k];
            for (int c = 0; c < 3; c++) g[kSepOffLogStd + 3 * k + c] = sig2[3 * k + c] * (hd.g[4 + c] * (hp[k] * hp[k]));
        }
        ppo_delta1_sep(W, hd, hp, hv, 1);
        for (int j = 0; j < kMlpH0; j++) {
            const float d0 = ppo_delta0(W, j, j < kMlpH1 ? hp : hv, h0[j]);
            for (int c = 0; c < kMlpIn; c++) g[kSepOffW0 + j * kMlpIn + c] = d0 * x[c];
            g[kSepOffB0 + j] = d0;
        }
        for (int k = 0; k < kMlpH1; k++) {
            for (int j = 0; j < kMlpH1; j++) {
                g[kSepOffW1 + k * kMlpH1 + j] = hp[k] * h0[j];
                g[kSepOffVw1 + k * kMlpH1 + j] = hv[k] * h0[kMlpH1 + j];
            }
            g[kSepOffB1 + k] = hp[k];
            g[kSepOffVb1 + k] = hv[k];
        }
        for (int c = 0; c < 3; c++) g[kSepOffB2 + c] = hd.g[c];
        g[kSepOffBv] = hd.g[3];
        float *t = terms + 5 * s;
        t[0] = hd.pg; t[1] = hd.vloss; t[2] = hd.clipped; t[3] = hd.kl; t[4] = hd.ent;
    }
}

}  // extern "C"
