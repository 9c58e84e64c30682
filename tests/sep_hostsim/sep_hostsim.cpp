// sep_hostsim.cpp — TEST-ONLY host compilation of the separate-tower math of rl_rocket_6dof_b200/csrc/r6_core.cuh
// (mlp_forward_sep, the mode-0 policy kernel's network) and csrc/r6_ppo.cuh (r6_ppo_grad's per-sample loss and gradient
// for SB3 1.6's separate policy / value towers), built by tests/sep_hostsim/__init__.py with g++ into
// tests/sep_hostsim/_build/.  Never imported, linked or shipped by the product package.
#include "../../rl_rocket_6dof_b200/csrc/r6_ppo.cuh"

using namespace r6;

namespace {
R6Mlp sep_mlp(const float *p)
{
    R6Mlp m = {p + kSepOffW0, p + kSepOffB0, p + kSepOffW1, p + kSepOffB1, p + kSepOffW2, p + kSepOffB2, p + kSepOffWv,
               p + kSepOffBv, p + kSepOffLogStd};
    m.vf_w0 = p + kSepOffVw0; m.vf_b0 = p + kSepOffVb0; m.vf_w1 = p + kSepOffVw1; m.vf_b1 = p + kSepOffVb1;
    return m;
}
}  // namespace

extern "C" {

int hs_sep_nparams(void) { return kPpoParamsSep; }

// mlp_forward_sep: out [n][4] (mean 0..2, value) for obs13 [n][13], params in the R6_PPO_NPARAMS_SEP layout
void hs_sep_forward(const float *params, const float *obs13, int64_t n, float *out)
{
    const R6Mlp m = sep_mlp(params);
    static float W[kMlpFloatsSep];
    for (int i = 0; i < kMlpFloatsSep; i++) W[i] = mlp_pack_element_sep(m, i);
    for (int64_t s = 0; s < n; s++) {
        float o[4];
        mlp_forward_sep(W, obs13 + 13 * s, o);
        for (int c = 0; c < 4; c++) out[4 * s + c] = o[c];
    }
}

// ppo_grad_sep_kernel's per-sample math: grad [n][R6_PPO_NPARAMS_SEP] (the float32 products the kernel accumulates,
// unsummed), terms [n][4] (pg, vloss, clipped, kl)
void hs_sep_sample_grad(const float *params, const float *obs13, const float *act3, const float *old_logp, const float *adv,
                        const float *ret, int64_t n, const double *adv_stats, float clip, float vf_coef, float ent_coef,
                        float *grad, float *terms)
{
    const R6Mlp m = sep_mlp(params);
    static float W[kMlpFloatsSep];
    for (int i = 0; i < kMlpFloatsSep; i++) W[i] = mlp_pack_element_sep(m, i);
    for (int64_t s = 0; s < n; s++) {
        const float *x = obs13 + 13 * s;
        float h0[kMlpH0], hp[kMlpH1], hv[kMlpH1], out[4];
        ppo_forward_sep(W, x, h0, hp, hv, 1, out);
        PpoHead hd;
        ppo_head(out, act3 + 3 * s, old_logp[s], ppo_advantage(adv[s], adv_stats), ret[s], m.log_std, clip, vf_coef, ent_coef, hd);
        float *g = grad + s * kPpoParamsSep;
        for (int k = 0; k < kMlpH1; k++) {
            for (int c = 0; c < 3; c++) g[kSepOffW2 + c * kMlpH1 + k] = hd.g[c] * hp[k];
            g[kSepOffWv + k] = hd.g[3] * hv[k];
        }
        ppo_delta1_sep(W, hd, hp, hv, 1);          // hp, hv now hold the deltas
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
