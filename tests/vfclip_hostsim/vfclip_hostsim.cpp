// vfclip_hostsim.cpp — TEST-ONLY host compilation of the value clipping of rl_rocket_6dof_b200/csrc/r6_ppo.cuh
// (ppo_value_clip after ppo_head / ppo_head_sde, as the kVfClip instantiations of the PPO gradient kernels run it),
// built by tests/vfclip_hostsim/__init__.py with g++ into tests/vfclip_hostsim/_build/.  Never imported, linked or
// shipped by the product package.
#include "../../rl_rocket_6dof_b200/csrc/r6_ppo.cuh"

using namespace r6;

extern "C" {

// the head of one sample and its value clipping: out4 [n][4] (mean 0..2, V), ls [3] (Gaussian log_std) or, with sde,
// var [n][3] (gSDE latent variances); g [n][7], vloss [n]
void hs_vf_head(int sde, const float *out4, const float *act3, const float *old_logp, const float *adv, const float *ret,
                const float *vold, int64_t n, const float *ls_or_var, float clip, float vf_coef, float ent_coef, float vfc,
                float *g, float *vloss)
{
    for (int64_t s = 0; s < n; s++) {
        const float out[4] = {out4[4 * s], out4[4 * s + 1], out4[4 * s + 2], out4[4 * s + 3]};
        PpoHeadSde hd;
        if (sde) {
            const float var[3] = {ls_or_var[3 * s], ls_or_var[3 * s + 1], ls_or_var[3 * s + 2]};
            ppo_head_sde(out, act3 + 3 * s, old_logp[s], adv[s], ret[s], var, clip, vf_coef, ent_coef, hd);
        } else {
            ppo_head(out, act3 + 3 * s, old_logp[s], adv[s], ret[s], ls_or_var, clip, vf_coef, ent_coef, hd);
        }
        ppo_value_clip(out[3], vold[s], ret[s], vfc, vf_coef, hd);
        for (int c = 0; c < 7; c++) g[7 * s + c] = hd.g[c];
        vloss[s] = hd.vloss;
    }
}

// ppo_grad_kernel<true>'s per-sample math (shared trunk): grad [n][R6_PPO_NPARAMS] unsummed, terms [n][4]
void hs_vf_shared_grad(const float *params, const float *obs13, const float *act3, const float *old_logp, const float *adv,
                       const float *ret, const float *vold, int64_t n, const double *adv_stats, float clip, float vf_coef,
                       float ent_coef, float vfc, float *grad, float *terms)
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
        ppo_value_clip(out[3], vold[s], ret[s], vfc, vf_coef, hd);
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

// ppo_grad_sep_kernel<true>'s per-sample math (separate towers): grad [n][R6_PPO_NPARAMS_SEP] unsummed, terms [n][4]
void hs_vf_sep_grad(const float *params, const float *obs13, const float *act3, const float *old_logp, const float *adv,
                    const float *ret, const float *vold, int64_t n, const double *adv_stats, float clip, float vf_coef,
                    float ent_coef, float vfc, float *grad, float *terms)
{
    R6Mlp m = {params + kSepOffW0, params + kSepOffB0, params + kSepOffW1, params + kSepOffB1, params + kSepOffW2,
               params + kSepOffB2, params + kSepOffWv, params + kSepOffBv, params + kSepOffLogStd};
    m.vf_w0 = params + kSepOffVw0; m.vf_b0 = params + kSepOffVb0; m.vf_w1 = params + kSepOffVw1; m.vf_b1 = params + kSepOffVb1;
    static float W[kMlpFloatsSep];
    for (int i = 0; i < kMlpFloatsSep; i++) W[i] = mlp_pack_element_sep(m, i);
    for (int64_t s = 0; s < n; s++) {
        const float *x = obs13 + 13 * s;
        float h0[kMlpH0], hp[kMlpH1], hv[kMlpH1], out[4];
        ppo_forward_sep(W, x, h0, hp, hv, 1, out);
        PpoHead hd;
        ppo_head(out, act3 + 3 * s, old_logp[s], ppo_advantage(adv[s], adv_stats), ret[s], m.log_std, clip, vf_coef, ent_coef, hd);
        ppo_value_clip(out[3], vold[s], ret[s], vfc, vf_coef, hd);
        float *g = grad + s * kPpoParamsSep;
        for (int k = 0; k < kMlpH1; k++) {
            for (int c = 0; c < 3; c++) g[kSepOffW2 + c * kMlpH1 + k] = hd.g[c] * hp[k];
            g[kSepOffWv + k] = hd.g[3] * hv[k];
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
        for (int c = 0; c < 3; c++) {
            g[kSepOffB2 + c] = hd.g[c];
            g[kSepOffLogStd + c] = hd.g[4 + c];
        }
        g[kSepOffBv] = hd.g[3];
        terms[4 * s] = hd.pg; terms[4 * s + 1] = hd.vloss; terms[4 * s + 2] = hd.clipped; terms[4 * s + 3] = hd.kl;
    }
}

}  // extern "C"
