// hostsim.cpp — TEST-ONLY host compilation of rl_rocket_6dof_b200/csrc/r6_core.cuh.
//
// Lets the CPU test-suite (-m "not gpu") run the exact per-environment code of the CUDA kernels
// against the oracle before any GPU time is spent (SURVEY.md §7 step 3).  It is built by
// tests/hostsim/__init__.py with g++ into tests/hostsim/_build/ and is never imported, linked or
// shipped by the product package, which has no CPU path and fails without its CUDA library.
#include <string.h>

#include "../../rl_rocket_6dof_b200/csrc/r6_core.cuh"

using namespace r6;

extern "C" {

struct HsEnv {
    double y[14];
    float m0, v0;
    int32_t k;
    uint32_t episode;
    double ep_return;
    float tgo, pad;      // warm start of the t_go iteration, carried from step to step like R6Buffers.tgo
};
struct HsOut {
    double state[14];
    float obs[14];
    double reward;
    double terms[7];
    int32_t flags, finished, natt, status, tgo_missing;
};

int hs_sizeof_env(void) { return (int)sizeof(HsEnv); }
int hs_sizeof_out(void) { return (int)sizeof(HsOut); }

void hs_step(const R6Params *p, const double *t_table, HsEnv *envs, int64_t n, const float *actions, HsOut *outs)
{
    const Derived dv = make_derived(*p);
    KLocal K;
    for (int64_t i = 0; i < n; i++) {
        Env e;
        memcpy(e.y, envs[i].y, sizeof e.y);
        e.m0 = envs[i].m0; e.v0 = envs[i].v0; e.k = envs[i].k; e.episode = envs[i].episode;
        e.ep_return = envs[i].ep_return;
        e.tgo = envs[i].tgo;
        StepOut o;
        if (p->dt <= kMaxDtSeries) env_step<false>(*p, dv, t_table, e, actions[3 * i], actions[3 * i + 1], actions[3 * i + 2], o, K);
        else env_step<true>(*p, dv, t_table, e, actions[3 * i], actions[3 * i + 1], actions[3 * i + 2], o, K);
        memcpy(envs[i].y, e.y, sizeof e.y);
        envs[i].k = e.k; envs[i].ep_return = e.ep_return; envs[i].tgo = e.tgo;
        HsOut &r = outs[i];
        memcpy(r.state, e.y, sizeof e.y);
        for (int c = 0; c < 14; c++) r.obs[c] = obs_component(*p, dv, e.y, c);
        r.reward = o.reward;
        memcpy(r.terms, o.post.terms, sizeof r.terms);
        r.flags = (int32_t)o.flags; r.finished = o.finished; r.natt = o.natt; r.status = o.status;
        r.tgo_missing = o.post.tgo_missing;
    }
}

void hs_reset(const R6Params *p, const R6Buffers *b, HsEnv *envs, int64_t n, int64_t env_offset, uint64_t seed)
{
    for (int64_t i = 0; i < n; i++) {
        Env e;
        e.episode = envs[i].episode;
        env_reset(*p, *b, seed, env_offset + i, e);
        memcpy(envs[i].y, e.y, sizeof e.y);
        envs[i].m0 = e.m0; envs[i].v0 = e.v0; envs[i].k = e.k; envs[i].episode = e.episode;
        envs[i].ep_return = e.ep_return; envs[i].tgo = e.tgo;
    }
}

int hs_sim_step_raw(double *y, const double *u, double m0, double t, double dt, int *natt)
{
    StepConst c;
    consts_raw_mode(c, m0, u[0], u[1], u[2], y[10]);
    KLocal K;
    int st = (dt <= kMaxDtSeries) ? integrate<false>(c, y, t, dt, *natt, K) : integrate<true>(c, y, t, dt, *natt, K);
    normalize_quat(y);
    return st;
}

// The same solve_ivp call cut at RK-attempt boundaries the way integrate_first_kernel / integrate_resume_kernel do:
// one attempt per pass, and between passes NOTHING survives but y and the PassCtx (fresh constants, fresh stage
// storage), which is exactly what the work lists carry on the device.
int hs_sim_step_raw_passes(double *y, const double *u, double m0, double t, double dt, int *natt, int *passes)
{
    PassCtx<double> px;
    px.budget = 1;
    int st;
    {
        StepConst c;
        consts_raw_mode(c, m0, u[0], u[1], u[2], y[10]);
        KLocal K;
        st = (dt <= kMaxDtSeries) ? integrate<false, KLocal, double, 1>(c, y, t, dt, *natt, K, px)
                                  : integrate<true, KLocal, double, 1>(c, y, t, dt, *natt, K, px);
    }
    *passes = 1;
    while (st == -2) {
        StepConst c;
        consts_raw_mode(c, m0, u[0], u[1], u[2], y[10]);
        KLocal K;
        memset(&K, 0, sizeof K);
        px.budget = 1;
        st = (dt <= kMaxDtSeries) ? integrate<false, KLocal, double, 2>(c, y, t, dt, *natt, K, px)
                                  : integrate<true, KLocal, double, 2>(c, y, t, dt, *natt, K, px);
        (*passes)++;
    }
    normalize_quat(y);
    return st;
}

double hs_tgo(double c0, double c2, double c3, double c4) { return tgo_largest_root(c0, c2, c3, c4); }
double hs_tgo_warm(double c0, double c2, double c3, double c4, double guess) { return tgo_largest_root(c0, c2, c3, c4, guess); }

void hs_euler_tests(const double viol[3], const double land[3], const double q[4], int *violated, int *land_ok)
{
    const AngleTests at = make_angle_tests(viol, land);
    bool v, l;
    euler_limit_tests(at, q[0], q[1], q[2], q[3], v, l);
    *violated = v; *land_ok = l;
}

void hs_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4])
{
    U4 r = philox4x32_10(U4{c0, c1, c2, c3}, k0, k1);
    out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

// fused-policy network on packed weights (W has kMlpFloats floats, built with mlp_pack_element)
int hs_mlp_floats(void) { return kMlpFloats; }
void hs_mlp_pack(const R6Mlp *m, float *W) { for (int i = 0; i < kMlpFloats; i++) W[i] = mlp_pack_element(*m, i); }
void hs_mlp(const float *W, const float *obs13, int64_t n, float *actions)
{
    for (int64_t i = 0; i < n; i++) mlp_policy(W, obs13 + 13 * i, actions[3 * i], actions[3 * i + 1], actions[3 * i + 2]);
}

// raw network outputs (out[4 i .. 4 i + 3] = unclipped mean, value) of the float32 FMA network
void hs_mlp_forward(const float *W, const float *obs13, int64_t n, float *out4)
{
    for (int64_t i = 0; i < n; i++) {
        float o[4];
        mlp_forward(W, obs13 + 13 * i, o);
        for (int c = 0; c < 4; c++) out4[4 * i + c] = o[c];
    }
}

// Gaussian policy head per row: mean4 [n][4] (value column ignored), genv / step [n], log_std [3] or NULL
void hs_gaussian_head(const float *mean4, const float *log_std, int32_t stochastic, uint64_t seed, const uint64_t *genv,
                      const uint64_t *step, int64_t n, float *raw3, float *logp)
{
    for (int64_t i = 0; i < n; i++) {
        const float m[4] = {mean4[4 * i], mean4[4 * i + 1], mean4[4 * i + 2], mean4[4 * i + 3]};
        float raw[3];
        gaussian_head(m, log_std, stochastic != 0, seed, genv[i], step[i], raw, logp[i]);
        for (int c = 0; c < 3; c++) raw3[3 * i + c] = raw[c];
    }
}

void hs_philox_action(uint64_t seed, uint64_t genv, uint64_t step, float a[3]) { philox_action(seed, genv, step, a[0], a[1], a[2]); }

}  // extern "C"
