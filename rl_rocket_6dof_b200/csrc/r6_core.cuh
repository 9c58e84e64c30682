// r6_core.cuh — per-environment math of the batched 6DOF env step (one thread = one environment).
//
// Restates, B200-first, the hot path of Tuxliri/RL_Rocket_6DOF:
//   Rocket6DOF.step            my_environment/envs/rocket_env.py:201-231
//   Simulator6DOF.step / RHS   my_environment/utils/simulator.py:69-143
//   SciPy solve_ivp RK45       scipy/integrate/_ivp/rk.py:14-180, common.py:63-134, ivp.py:52-158,646-716
//   reward / flags / obs       rocket_env.py:317-402, 503-566, 591-617
// following the verified precision map of SURVEY.md Appendix A (float32 where the reference is
// float32, float64 elsewhere).  It is NOT a transliteration: the right-hand side is algebraically
// de-duplicated (one rotation matrix, un-normalised quaternion scaled by 1/|q|^2, gyroscopic term
// of the axisymmetric body folded), the position rows of the Runge–Kutta stages are eliminated with
// the squared tableau (A·A, Bᵀ·A, Eᵀ·A) so a stage stores 9 instead of 14 doubles, the air density is
// expanded around the step's initial height, and the Euler-angle limit tests are done on cosines
// instead of atan2.  All of these change results at the 1e-16 level only (tolerance is 1e-9).
//
// The file compiles for the device (nvcc, sm_100a) and — for tests/hostsim only — for the host with
// g++ (R6_HOST_BUILD).  The product never uses the host build.
#pragma once

#include <math.h>
#include <stdint.h>

#include "../../include/r6dof.h"

#if defined(__CUDACC__)
#define R6_HD __host__ __device__ __forceinline__
#define R6_HD_NOINLINE __host__ __device__ __noinline__
#else
#define R6_HD inline
#define R6_HD_NOINLINE inline
#endif

namespace r6 {

// ------------------------------------------------------------------------------------------------
// float32 primitives that must not be contracted / reassociated (SURVEY §A.1)
#if defined(__CUDA_ARCH__)
R6_HD float f32_mul(float a, float b) { return __fmul_rn(a, b); }
R6_HD float f32_add(float a, float b) { return __fadd_rn(a, b); }
R6_HD float f32_sub(float a, float b) { return __fsub_rn(a, b); }
R6_HD float f32_div(float a, float b) { return __fdiv_rn(a, b); }
R6_HD float f32_sqrt(float a) { return __fsqrt_rn(a); }
R6_HD float f32_fma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
R6_HD float f64_to_f32(double a) { return __double2float_rn(a); }
// fast reciprocal / square root: MUFU seed (relative error 2^-20 measured on sm_100a, profiles/microbench/mufu_seed.cu)
// + one third-order step r (1 + e + e^2), e = 1 - x r  =>  <= 1 ulp, three dependent FMAs, no IEEE special cases.
R6_HD double fast_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);
    return fma(r, fma(e, e, e), r);
}
// one Newton step only (~1e-12 relative): for the tolerance-scaled norms of the step-size controller,
// where 1e-12 in a scale moves the next step size by 1e-12 and the solution by < 1e-15 (DESIGN.md §3)
R6_HD double fast_rcp1(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    return fma(r, fma(-x, r, 1.0), r);
}
R6_HD double fast_sqrt(double x)
{
    double r;
    // seed on x + tiny: x = 0 then gives s = 0 * r = 0 without a branch (x + 1e-300 == x for every normal x)
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x + 1e-300));
    // coupled (Goldschmidt) iteration on s ~ sqrt(x), h ~ 1/(2 sqrt(x)): two quadratic steps 2^-20 -> 2^-40 -> 2^-80,
    // i.e. rounding-limited (<= 1 ulp measured); 2 DMUL + 5 DFMA
    double s = x * r, h = 0.5 * r;
    double e = fma(-s, h, 0.5);
    s = fma(s, e, s);
    h = fma(h, e, h);
    e = fma(-s, h, 0.5);
    return fma(s, e, s);
}
#else
R6_HD float f32_mul(float a, float b) { return a * b; }
R6_HD float f32_add(float a, float b) { return a + b; }
R6_HD float f32_sub(float a, float b) { return a - b; }
R6_HD float f32_div(float a, float b) { return a / b; }
R6_HD float f32_sqrt(float a) { return sqrtf(a); }
R6_HD float f32_fma(float a, float b, float c) { return fmaf(a, b, c); }
R6_HD float f64_to_f32(double a) { return (float)a; }
R6_HD double fast_rcp(double x) { return 1.0 / x; }
R6_HD double fast_rcp1(double x) { return 1.0 / x; }
R6_HD double fast_sqrt(double x) { return sqrt(x); }
#endif

// NumPy's float32 cos/sin for |x| < pi/4 (exact polynomial, SURVEY §A.1); simulator.py:204-207
R6_HD float np_cosf_small(float x)
{
    float x2 = f32_mul(x, x), r;
    r = f32_fma(0x1.98e616p-16f, x2, -0x1.6c06dcp-10f);
    r = f32_fma(r, x2, 0x1.55553cp-05f);
    r = f32_fma(r, x2, -0x1p-1f);
    r = f32_fma(r, x2, 1.0f);
    return r;
}
R6_HD float np_sinf_small(float x)
{
    float x2 = f32_mul(x, x), r;
    r = f32_fma(0x1.7d3bbcp-19f, x2, -0x1.a06bbap-13f);
    r = f32_fma(r, x2, 0x1.11119ap-07f);
    r = f32_fma(r, x2, -0x1.555556p-03f);
    r = f32_fma(r, x2, 0.0f);
    r = f32_fma(r, x, x);
    return r;
}
// OpenBLAS sdot (n = 3): float32 products, float64 sequential accumulation, one float32 rounding
R6_HD float sdot3(float a0, float a1, float a2, float b0, float b1, float b2)
{
    double acc = (double)f32_mul(a0, b0);
    acc = acc + (double)f32_mul(a1, b1);
    acc = acc + (double)f32_mul(a2, b2);
    return f64_to_f32(acc);
}

// ------------------------------------------------------------------------------------------------
// Precision of the integrator.  R = double is the parity path (<= 1e-9 against the reference);
// R = float is the optional throughput path with its own stated bound (tests/test_gpu_fp32.py).
// Everything from here to the end of integrate() is generic in R; literals are written R(x) so that a
// float instantiation contains no double arithmetic.
template <class R> struct Real;
template <> struct Real<double> {
    static constexpr double eps = 2.220446049250313e-16;
    static constexpr double tiny = 1e-300;
};
template <> struct Real<float> {
    static constexpr float eps = 1.1920929e-07f;
    static constexpr float tiny = 1e-30f;
};
#if defined(__CUDA_ARCH__)
R6_HD float fast_rcp(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
R6_HD float fast_sqrt(float x)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
#else
R6_HD float fast_rcp(float x) { return 1.0f / x; }
R6_HD float fast_sqrt(float x) { return sqrtf(x); }
#endif
R6_HD float fast_rcp1(float x) { return fast_rcp(x); }
R6_HD double r_nextafter_up(double t) { return nextafter(t, (double)INFINITY); }
R6_HD float r_nextafter_up(float t) { return nextafterf(t, INFINITY); }

// ------------------------------------------------------------------------------------------------
// Dormand–Prince tableau (scipy rk.py:541-565) and the derived "position" tableaus.
template <class R>
struct TabT {
    R A[6][5], B[6], C[6], E[7];
    R AA[6][5];   // AA[s][j] = sum_k A[s][k] A[k][j]   : x_s = x + h C_s v + h^2 sum_j AA[s][j] dv_j
    R BA[6];      // BA[j]    = sum_k B[k] A[k][j]      : r_new = r + h v + h^2 sum_j BA[j] dv_j
    R EA[6];      // EA[j]    = sum_k E[k] A[k][j] + E[6] B[j] : e_r = h^2 sum_j EA[j] dv_j
    // stage-input rows used by the rolled integrator: x = y + h * sum_j SA[row][j] K_j, positions
    // r = r + h SC[row] v + h^2 sum_j SAA[row][j] dv_j.  rows 1..5 = (A, AA, C); row 6 = (B, BA, 1) gives
    // y_new (the 7th Dormand-Prince stage is evaluated AT y_new); row 7 = (e_0, 0, 1) gives y + h f0,
    // the probe point of select_initial_step.
    R SA[8][6], SAA[8][6], SC[8];
    R P[7][4];
    R Psum[4];    // Psum[m]  = sum_j P[j][m]
    R PA[6][4];   // PA[j][m] = sum_k P[k][m] A[k][j] + P[6][m] B[j] : dense output of the position rows
};
using Tab = TabT<double>;
constexpr Tab make_tab()
{
    Tab t{};
    const double A[6][5] = {
        {0, 0, 0, 0, 0},
        {1.0 / 5, 0, 0, 0, 0},
        {3.0 / 40, 9.0 / 40, 0, 0, 0},
        {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
        {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
        {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
    const double B[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
    const double C[6] = {0, 1.0 / 5, 3.0 / 10, 4.0 / 5, 8.0 / 9, 1};
    const double E[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
    const double P[7][4] = {
        {1, -8048581381.0 / 2820520608, 8663915743.0 / 2820520608, -12715105075.0 / 11282082432},
        {0, 0, 0, 0},
        {0, 131558114200.0 / 32700410799, -68118460800.0 / 10900136933, 87487479700.0 / 32700410799},
        {0, -1754552775.0 / 470086768, 14199869525.0 / 1410260304, -10690763975.0 / 1880347072},
        {0, 127303824393.0 / 49829197408, -318862633887.0 / 49829197408, 701980252875.0 / 199316789632},
        {0, -282668133.0 / 205662961, 2019193451.0 / 616988883, -1453857185.0 / 822651844},
        {0, 40617522.0 / 29380423, -110615467.0 / 29380423, 69997945.0 / 29380423}};
    for (int s = 0; s < 6; s++) {
        t.B[s] = B[s];
        t.C[s] = C[s];
        for (int j = 0; j < 5; j++) t.A[s][j] = A[s][j];
    }
    for (int j = 0; j < 7; j++) {
        t.E[j] = E[j];
        for (int m = 0; m < 4; m++) t.P[j][m] = P[j][m];
    }
    for (int s = 0; s < 6; s++)
        for (int j = 0; j < 5; j++) {
            double a = 0;
            for (int k = j + 1; k < s; k++) a += A[s][k] * A[k][j];
            t.AA[s][j] = a;
        }
    for (int j = 0; j < 6; j++) {
        double b = 0, e = 0;
        for (int k = j + 1; k < 6; k++) {
            b += B[k] * A[k][j];
            e += E[k] * A[k][j];
        }
        t.BA[j] = b;
        t.EA[j] = e + E[6] * B[j];
    }
    for (int s = 1; s < 6; s++) {
        t.SC[s] = C[s];
        for (int j = 0; j < 5; j++) { t.SA[s][j] = A[s][j]; t.SAA[s][j] = t.AA[s][j]; }
    }
    for (int j = 0; j < 6; j++) { t.SA[6][j] = B[j]; t.SAA[6][j] = t.BA[j]; }
    t.SC[6] = 1;
    t.SA[7][0] = 1;
    t.SC[7] = 1;
    for (int m = 0; m < 4; m++) {
        double ps = 0;
        for (int j = 0; j < 7; j++) ps += P[j][m];
        t.Psum[m] = ps;
        for (int j = 0; j < 6; j++) {
            double a = 0;
            for (int k = j + 1; k < 6; k++) a += P[k][m] * A[k][j];
            t.PA[j][m] = a + P[6][m] * B[j];
        }
    }
    return t;
}
constexpr TabT<float> make_tab_f32()
{
    const Tab d = make_tab();
    TabT<float> t{};
    for (int s = 0; s < 6; s++) {
        t.B[s] = (float)d.B[s]; t.C[s] = (float)d.C[s]; t.BA[s] = (float)d.BA[s]; t.EA[s] = (float)d.EA[s];
        for (int j = 0; j < 5; j++) { t.A[s][j] = (float)d.A[s][j]; t.AA[s][j] = (float)d.AA[s][j]; }
        for (int m = 0; m < 4; m++) t.PA[s][m] = (float)d.PA[s][m];
    }
    for (int j = 0; j < 7; j++) {
        t.E[j] = (float)d.E[j];
        for (int m = 0; m < 4; m++) t.P[j][m] = (float)d.P[j][m];
    }
    for (int r = 0; r < 8; r++) {
        t.SC[r] = (float)d.SC[r];
        for (int j = 0; j < 6; j++) { t.SA[r][j] = (float)d.SA[r][j]; t.SAA[r][j] = (float)d.SAA[r][j]; }
    }
    for (int m = 0; m < 4; m++) t.Psum[m] = (float)d.Psum[m];
    return t;
}
constexpr Tab kTabHost = make_tab();
constexpr TabT<float> kTabHostF = make_tab_f32();
#if defined(__CUDACC__)
__constant__ Tab kTabDev = make_tab();               // dynamically indexed by the rolled stage loop
__constant__ TabT<float> kTabDevF = make_tab_f32();
#endif
template <class R> R6_HD const TabT<R> &tab();
#if defined(__CUDA_ARCH__)
template <> R6_HD const TabT<double> &tab<double>() { return kTabDev; }
template <> R6_HD const TabT<float> &tab<float>() { return kTabDevF; }
#else
template <> R6_HD const TabT<double> &tab<double>() { return kTabHost; }
template <> R6_HD const TabT<float> &tab<float>() { return kTabHostF; }
#endif

// ------------------------------------------------------------------------------------------------
// Per-step constants consumed by the RHS
template <class R>
struct StepConstT {
    R Tb0, Tb1, Tb2;   // thrust in the body frame (simulator.py:167-175)
    R Ji1;             // 1/J_yy (= 1/J_zz), float32-valued (simulator.py:45-50)
    R gy;              // w0 * (J0 - J1) * Ji1 : gyroscopic coupling (w0 is constant: dw0 = 0)
    R dm;              // mass rate (simulator.py:140-141)
    // air-density expansion around the step's initial height (simulator.py:145-150)
    R h0, rho0, kd;    // rho(h) = rho0 * (1 - d)^p, d = kd*(h - h0), p = -(1 + g0 M / R / L)
    // folded forms consumed by rhs() (set by consts_finish / density_setup):
    R hw0;             // w0 / 2                              (quaternion kinematics)
    R j5, k1, k2;      // 5 Ji1, 20 Ji1 Tb2, -20 Ji1 Tb1      (torques written on the total force F = Tb + A)
    R nkdh0, rhoc;     // -kd h0, -S_ref C_a rho0 / 2         (d = kd h + nkdh0; aero factor = rhoc (1 - d)^p)
};
using StepConst = StepConstT<double>;

// physical constants (simulator.py:39-67)
constexpr double kG0 = 9.81;
constexpr double kRb = 3.66 / 2;
constexpr double kRb2 = kRb * kRb;
constexpr double kLen2 = 40.0 * 40.0 + 3 * kRb2;
constexpr double kSref = 3.14159265358979323846 * kRb2;
constexpr double kRhoExp = 1 + 9.81 * 0.0289644 / 8.3144598 / (-0.0065);   // ~ -4.2559
constexpr double kLapseOverT = 0.0065 / 288.15;
constexpr double kCa = 0.82;
constexpr double kAero = -0.5 * kSref * kCa;     // aerodynamic force = kAero rho |v| v_body (simulator.py:216-219)

// x^e for x > 0 (one call per env-step: the density at the step's initial height)
R6_HD_NOINLINE double pow_pos(double x, double e) { return exp(e * log(x)); }
R6_HD float pow_pos(float x, float e)
{
#if defined(__CUDA_ARCH__)
    return exp2f(e * __log2f(x));       // MUFU pair, ~1e-6 relative: inside the float path's own round-off
#else
    return expf(e * logf(x));
#endif
}

template <class R>
R6_HD R density_exact(R h)
{
    // 1.225 * (T_b/(T_b + h L_b))^e  ==  1.225 * (1 - c h)^(-e),  c = 0.0065/288.15
    return R(1.225) * pow_pos(R(1.0) - R(kLapseOverT) * h, R(-kRhoExp));
}

struct RhoSeries { double c[14]; };
constexpr RhoSeries make_rho_series(double p)
{
    RhoSeries r{};
    r.c[0] = 1.0;
    for (int k = 0; k < 13; k++) r.c[k + 1] = r.c[k] * (-(p - k)) / (k + 1);
    return r;
}
// Density at the step's initial height: rho0 = 1.225 (1 - x)^p, x = c h0, p = 4.2576.  Because p is close to
// an integer the binomial coefficients collapse after k = 5 (|b_13| = 3e-5), so for |x| <= 0.08 (|h0| <= 3.5 km,
// any state inside the reference's bounds box) 13 Horner steps are exact to < 2e-19 and replace a log/exp pair
// (~200 executed, ~500 static instructions).  Outside that range the out-of-line pow is used.
template <class R>
R6_HD void density_setup(StepConstT<R> &c, R h0)
{
    c.h0 = h0;
    const R x = R(kLapseOverT) * h0;
    const R base = R(1.0) - x;
    c.kd = R(kLapseOverT) * fast_rcp(base);
    constexpr double p = -kRhoExp;
    constexpr int kTerms = sizeof(R) == 8 ? 13 : 6;
    if (fabs(x) <= R(0.08)) {
        constexpr RhoSeries b = make_rho_series(p);      // b_k = binom(p, k) (-1)^k, at compile time
        R s = R(b.c[kTerms - 1]);
#pragma unroll
        for (int k = kTerms - 2; k >= 0; k--) s = fma(s, x, R(b.c[k]));
        c.rho0 = R(1.225) * s;
    } else {
        c.rho0 = R(1.225) * pow_pos(base, R(-kRhoExp));
    }
    c.nkdh0 = -(c.kd * h0);
    c.rhoc = R(kAero) * c.rho0;
}

// kExact = false: binomial series of (1 - d)^p around the step's initial height, d = kd (h - h0),
// p = -kRhoExp, to d^6; the next term is 2.6e-3 d^7, i.e. < 3e-17 for |d| <= 0.01 (|h - h0| <= 400 m).
// The launcher picks kExact = true when dt is so large that this cannot be guaranteed (dt > 0.25 s).
// series coefficients b_1..b_6 of (1 - d)^p.  On the device they live in the constant bank so that each Horner
// step is ONE DFMA with a c[bank][offset] operand; as literals ptxas materialises every 64-bit immediate with two
// UMOVs, which doubled the instruction count of this function (it runs in every right-hand-side evaluation).
struct RhoStep { double b[7]; float bf[7]; };
constexpr RhoStep make_rho_step()
{
    constexpr double p = -kRhoExp;
    RhoStep r{};
    r.b[0] = 1.0;
    for (int k = 0; k < 6; k++) r.b[k + 1] = r.b[k] * (-(p - k)) / (k + 1);
    for (int k = 0; k < 7; k++) r.bf[k] = (float)r.b[k];
    return r;
}
constexpr RhoStep kRhoStepHost = make_rho_step();
#if defined(__CUDACC__)
__constant__ RhoStep kRhoStepDev = make_rho_step();
#endif
#if defined(__CUDA_ARCH__)
#define R6_RHO_STEP ::r6::kRhoStepDev
#else
#define R6_RHO_STEP ::r6::kRhoStepHost
#endif
R6_HD double rho_b(int k, double) { return R6_RHO_STEP.b[k]; }
R6_HD float rho_b(int k, float) { return R6_RHO_STEP.bf[k]; }

constexpr double kMaxDtSeries = 0.25;   // (1000 m/s + 60 m/s^2 dt) dt kd <= 0.01 up to here

// folded per-step constants of rhs() from (Tb, Ji1, w0)
template <class R>
R6_HD void consts_finish(StepConstT<R> &c, R w0)
{
    c.hw0 = R(0.5) * w0;
    c.j5 = R(5.0) * c.Ji1;
    c.k1 = R(20.0) * c.Ji1 * c.Tb2;
    c.k2 = R(-20.0) * c.Ji1 * c.Tb1;
}

// env mode constants from the float32 control / initial mass (SURVEY §A.1)
template <class R>
R6_HD void consts_env_mode(StepConstT<R> &c, float m0, float u0, float u1, float u2, R w0)
{
    float J0 = f32_mul(f32_mul(0.5f, m0), (float)kRb2);
    float J1 = f32_mul(f32_mul((float)(1.0 / 12), m0), (float)kLen2);
    float Ji1 = f32_div(1.0f, J1);
    c.Ji1 = (R)Ji1;
    c.gy = w0 * ((R)J0 - (R)J1) * c.Ji1;
    float cy = np_cosf_small(u0), cz = np_cosf_small(u1);
    float sy = np_sinf_small(u0), sz = np_sinf_small(u1);
    R T = (R)u2;
    c.Tb0 = (R)f32_mul(cy, cz) * T;
    c.Tb1 = (R)f32_mul(sy, cz) * T;
    c.Tb2 = (R)sz * T;
    c.dm = (R)f32_div(-u2, (float)(9.81 * 360));
    consts_finish(c, w0);
}
// raw Simulator6DOF mode: python-list inputs => everything float64 (test_6DOF_simulator.py)
R6_HD void consts_raw_mode(StepConst &c, double m0, double u0, double u1, double u2, double w0)
{
    double J0 = .5 * m0 * kRb2, J1 = 1.0 / 12 * m0 * kLen2;
    c.Ji1 = 1.0 / J1;
    c.gy = w0 * (J0 - J1) * c.Ji1;
    double cy = cos(u0), cz = cos(u1), sy = sin(u0), sz = sin(u1);
    c.Tb0 = (cy * cz) * u2;
    c.Tb1 = (sy * cz) * u2;
    c.Tb2 = sz * u2;
    c.dm = -u2 / (9.81 * 360);
    consts_finish(c, w0);
}

// ------------------------------------------------------------------------------------------------
// One stage derivative: dv[3], dq[4], dw1, dw2  (dr = v, dw0 = 0, dm = const are implicit)
template <class R>
struct DerivT {
    R dv0, dv1, dv2, dq0, dq1, dq2, dq3, dw1, dw2;
};
using Deriv = DerivT<double>;

// un-normalised rotation matrix entries of the leading-scalar quaternion (q0,q1,q2,q3); R = M / n2
template <class R>
struct RotUT {
    R m00, m01, m02, m10, m11, m12, m20, m21, m22, n2;
};
using RotU = RotUT<double>;
template <class R>
R6_HD RotUT<R> rot_unnormalised(R q0, R q1, R q2, R q3)
{
    RotUT<R> r;
    R x2 = q1 * q1, y2 = q2 * q2, z2 = q3 * q3, w2 = q0 * q0;
    R xy = q1 * q2, zw = q3 * q0, xz = q1 * q3, yw = q2 * q0, yz = q2 * q3, xw = q1 * q0;
    r.m00 = x2 - y2 - z2 + w2; r.m01 = 2 * (xy - zw);       r.m02 = 2 * (xz + yw);
    r.m10 = 2 * (xy + zw);     r.m11 = -x2 + y2 - z2 + w2;  r.m12 = 2 * (yz - xw);
    r.m20 = 2 * (xz - yw);     r.m21 = 2 * (yz + xw);       r.m22 = -x2 - y2 + z2 + w2;
    r.n2 = x2 + y2 + z2 + w2;
    return r;
}

// simulator.py:106-143 — inputs: height, velocity, quaternion, (w1,w2), mass of the stage state.
// Written for the FP64 pipe (89 instructions, 2/3 of them FMAs):
//   * rotation matrix from the doubled quaternion components and two sums / differences of squares
//     (M = |q|^2 R; 22 operations instead of 34);
//   * the constant factors of the drag (-S C_a / 2) ride on the density constant rhoc, the 1/2 of the quaternion
//     kinematics on the body rates;
//   * torques on the total body force F = Tb + A:  tau_y = 15 Tb2 - 5 A2 = 20 Tb2 - 5 F2 (the subtraction F - Tb that
//     this hides costs < 1e-16 rad/s^2), so A itself is never formed and F comes out of three FMAs.
template <bool kExact, class R>
R6_HD DerivT<R> rhs(const StepConstT<R> &c, R h, R v0, R v1, R v2, R q0, R q1, R q2, R q3, R w1, R w2, R m)
{
    DerivT<R> d;
    R rhoS;                                  // -S_ref C_a rho(h) / 2
    if (kExact) rhoS = R(kAero) * density_exact(h);
    else {
        const R dd = fma(c.kd, h, c.nkdh0);
        // float: d^4 and beyond are below the rounding of the sum (|d| <= 0.01)
        R s = (sizeof(R) == 8) ? fma(fma(fma(rho_b(6, R()), dd, rho_b(5, R())), dd, rho_b(4, R())), dd, rho_b(3, R())) : rho_b(3, R());
        s = fma(s, dd, rho_b(2, R()));
        s = fma(s, dd, rho_b(1, R()));
        s = fma(s, dd, R(1.0));
        rhoS = c.rhoc * s;
    }
    // un-normalised rotation matrix M = |q|^2 R(q), leading-scalar quaternion (simulator.py:177-186)
    const R Q1 = q1 + q1, Q2 = q2 + q2, Q3 = q3 + q3;
    const R ww = q0 * q0, zz = q3 * q3;
    const R s1 = fma(q1, q1, ww), s2 = fma(q2, q2, zz), d1 = fma(-q1, q1, ww), d2 = fma(q2, q2, -zz);
    const R n2 = s1 + s2, m00 = s1 - s2, m11 = d1 + d2, m22 = d1 - d2;
    const R zw = Q3 * q0, yw = Q2 * q0, xw = Q1 * q0;
    const R m01 = fma(Q1, q2, -zw), m10 = fma(Q1, q2, zw);
    const R m02 = fma(Q1, q3, yw), m20 = fma(Q1, q3, -yw);
    const R m12 = fma(Q2, q3, -xw), m21 = fma(Q2, q3, xw);
    const R inv = fast_rcp(n2 * m);          // 1 / (|q|^2 m)
    const R inv_n2 = inv * m;
    // body-frame velocity (R^T v) and aerodynamic force (simulator.py:216-219)
    const R vb0 = fma(m20, v2, fma(m10, v1, m00 * v0));
    const R vb1 = fma(m21, v2, fma(m11, v1, m01 * v0));
    const R vb2 = fma(m22, v2, fma(m12, v1, m02 * v0));
    const R vn = fast_sqrt(fma(v2, v2, fma(v1, v1, v0 * v0)));
    const R ca = rhoS * vn * inv_n2;
    const R F0 = fma(ca, vb0, c.Tb0), F1 = fma(ca, vb1, c.Tb1), F2 = fma(ca, vb2, c.Tb2);
    // simulator.py:127-130, 156-165
    d.dv0 = fma(fma(m02, F2, fma(m01, F1, m00 * F0)), inv, R(-kG0));
    d.dv1 = fma(m12, F2, fma(m11, F1, m10 * F0)) * inv;
    d.dv2 = fma(m22, F2, fma(m21, F1, m20 * F0)) * inv;
    // simulator.py:136, 221-229 (un-normalised quaternion)
    const R hw0 = c.hw0, hw1 = R(0.5) * w1, hw2 = R(0.5) * w2;
    d.dq0 = fma(-hw0, q1, fma(-hw1, q2, -(hw2 * q3)));
    d.dq1 = fma(hw0, q0, fma(hw2, q2, -(hw1 * q3)));
    d.dq2 = fma(hw1, q0, fma(-hw2, q1, hw0 * q3));
    d.dq3 = fma(hw2, q0, fma(hw1, q1, -(hw0 * q2)));
    // simulator.py:137, 232-244: tau = [0, 15 T2 - 5 A2, -15 T1 + 5 A1];  J = diag(J0, J1, J1)
    d.dw1 = fma(-c.gy, w2, fma(-c.j5, F2, c.k1));
    d.dw2 = fma(c.gy, w1, fma(c.j5, F1, c.k2));
    return d;
}

R6_HD double sq(double x) { return x * x; }
R6_HD float sq(float x) { return x * x; }
R6_HD bool sgn(double x) { return signbit(x); }
R6_HD bool sgn(float x) { return signbit(x); }

// ------------------------------------------------------------------------------------------------
// Stage storage.  The Runge–Kutta stage loop is ROLLED (one copy of the right-hand side in the
// instruction stream, coefficients read from the constant bank) and the six stage derivatives
// K_j = (dv, dq, dw1, dw2) live outside the register file: on the device in shared memory,
// [stage][component][thread] so that a warp touches 32 consecutive values (conflict-free), on the
// host (tests/hostsim) in a local array.
constexpr int kNK = 9;   // stored components per stage
template <class R>
struct Pair {
    R a, b;
};
template <class R>
struct KLocalT {
    R k[6][kNK];
    R6_HD R get(int j, int c) const { return k[j][c]; }
    R6_HD void set(int j, int c, R v) { k[j][c] = v; }
    R6_HD Pair<R> get2(int j, int p) const { return Pair<R>{k[j][2 * p], k[j][2 * p + 1]}; }
    R6_HD void set2(int j, int p, R a, R b) { k[j][2 * p] = a; k[j][2 * p + 1] = b; }
};
using KLocal = KLocalT<double>;
#if defined(__CUDACC__)
// [stage][pair][thread][2] for components 0..7 and [stage][8][thread] for the ninth: a thread's components 2p, 2p+1 are
// adjacent, so a pair moves with ONE 128-bit (float64) shared-memory instruction; a warp's 32 pairs are 512 contiguous
// bytes (conflict-free in four wavefronts, the same data-pipe time as two 64-bit accesses, half the issue slots).
template <class R, int kThreadsPerBlock>
struct KShared {
    R *base;   // smem + 2 * threadIdx.x
    __device__ __forceinline__ int off(int j, int c) const
    {
        return j * kNK * kThreadsPerBlock + (c < 8 ? (c >> 1) * 2 * kThreadsPerBlock + (c & 1) : 8 * kThreadsPerBlock - (int)threadIdx.x);
    }
    __device__ __forceinline__ R get(int j, int c) const { return base[off(j, c)]; }
    __device__ __forceinline__ void set(int j, int c, R v) { base[off(j, c)] = v; }
    __device__ __forceinline__ Pair<R> get2(int j, int p) const
    {
        if constexpr (sizeof(R) == 8) {
            const double2 v = *reinterpret_cast<const double2 *>(base + (j * kNK + 2 * p) * kThreadsPerBlock);
            return Pair<R>{v.x, v.y};
        } else {
            const float2 v = *reinterpret_cast<const float2 *>(base + (j * kNK + 2 * p) * kThreadsPerBlock);
            return Pair<R>{v.x, v.y};
        }
    }
    __device__ __forceinline__ void set2(int j, int p, R a, R b)
    {
        if constexpr (sizeof(R) == 8) *reinterpret_cast<double2 *>(base + (j * kNK + 2 * p) * kThreadsPerBlock) = make_double2(a, b);
        else *reinterpret_cast<float2 *>(base + (j * kNK + 2 * p) * kThreadsPerBlock) = make_float2(a, b);
    }
};
#endif
template <class KS, class R>
R6_HD void k_store(KS &K, int j, const DerivT<R> &d)
{
    K.set2(j, 0, d.dv0, d.dv1); K.set2(j, 1, d.dv2, d.dq0); K.set2(j, 2, d.dq1, d.dq2); K.set2(j, 3, d.dq3, d.dw1);
    K.set(j, 8, d.dw2);
}

// ------------------------------------------------------------------------------------------------
// Terminal height event (ivp.py:52-77, 134-158, 678-699): quartic dense output of the accepted step
// (rk.py:178-180, 715-737) from the stored stages, y[0] = 0 located by Brent's method exactly as
// scipy.optimize.brentq does (xtol = rtol = 4 eps, maxiter 100), then y = sol(t_event).
// Position rows use the PA tableau (their stage derivatives are stage velocities), the mass row is
// dm * Psum, the w0 row is 0.  Rare (at most once per episode) => not inlined.
template <class KS, class R>
R6_HD_NOINLINE void event_resolve(const StepConstT<R> &c, R *y /* in: y_old, out: y(t_event) */, const KS &K,
                                  const DerivT<R> &fn, R t_old, R t_new)
{
    const TabT<R> &T = tab<R>();
    const R h = t_new - t_old;
    R qx[4];   // Q row of the height component
    for (int m = 0; m < 4; m++) {
        R a = 0;
        for (int j = 0; j < 6; j++) a += T.PA[j][m] * K.get(j, 0);
        qx[m] = y[3] * T.Psum[m] + h * a;
    }
    const R x_old = y[0];
    auto ev = [&](R t) {
        const R x = (t - t_old) / h;
        const R p0 = x, p1 = p0 * x, p2 = p1 * x, p3 = p2 * x;
        return h * (qx[0] * p0 + qx[1] * p1 + qx[2] * p2 + qx[3] * p3) + x_old;
    };
    const R eps4 = 4 * Real<R>::eps;
    R xpre = t_old, xcur = t_new, xblk = 0, fblk = 0, spre = 0, scur = 0;
    R fpre = ev(xpre), fcur = ev(xcur);
    R root = xcur;
    if (fpre == 0) root = xpre;
    else if (fcur == 0) root = xcur;
    else if (sgn(fpre) == sgn(fcur)) root = xcur;   // scipy raises; cannot happen after the sign test
    else {
        for (int it = 0; it < 100; it++) {
            if (fpre != 0 && fcur != 0 && (sgn(fpre) != sgn(fcur))) {
                xblk = xpre; fblk = fpre; spre = scur = xcur - xpre;
            }
            if (fabs(fblk) < fabs(fcur)) {
                xpre = xcur; xcur = xblk; xblk = xpre;
                fpre = fcur; fcur = fblk; fblk = fpre;
            }
            const R delta = (eps4 + eps4 * fabs(xcur)) / 2;
            const R sbis = (xblk - xcur) / 2;
            if (fcur == 0 || fabs(sbis) < delta) break;
            if (fabs(spre) > delta && fabs(fcur) < fabs(fpre)) {
                R stry;
                if (xpre == xblk) stry = -fcur * (xcur - xpre) / (fcur - fpre);
                else {
                    const R dpre = (fpre - fcur) / (xpre - xcur);
                    const R dblk = (fblk - fcur) / (xblk - xcur);
                    stry = -fcur * (fblk * dblk - fpre * dpre) / (dblk * dpre * (fblk - fpre));
                }
                const R lim = fmin(fabs(spre), 3 * fabs(sbis) - delta);
                if (2 * fabs(stry) < lim) { spre = scur; scur = stry; }
                else { spre = sbis; scur = sbis; }
            } else { spre = sbis; scur = sbis; }
            xpre = xcur; fpre = fcur;
            if (fabs(scur) > delta) xcur += scur;
            else xcur += (sbis > 0 ? delta : -delta);
            fcur = ev(xcur);
        }
        root = xcur;
    }
    // y = sol(root)
    const R x = (root - t_old) / h;
    R p[4];
    p[0] = x; p[1] = p[0] * x; p[2] = p[1] * x; p[3] = p[2] * x;
    R pp[7];   // pp[j] = sum_m P[j][m] p_m ; ppa[j] for the position rows ; ps = sum_m Psum[m] p_m
    R ppa[6], ps = 0;
    for (int j = 0; j < 7; j++) {
        R a = 0;
        for (int m = 0; m < 4; m++) a += T.P[j][m] * p[m];
        pp[j] = a;
    }
    for (int j = 0; j < 6; j++) {
        R a = 0;
        for (int m = 0; m < 4; m++) a += T.PA[j][m] * p[m];
        ppa[j] = a;
    }
    for (int m = 0; m < 4; m++) ps += T.Psum[m] * p[m];
    const R fnv[kNK] = {fn.dv0, fn.dv1, fn.dv2, fn.dq0, fn.dq1, fn.dq2, fn.dq3, fn.dw1, fn.dw2};
    // positions first (they need the old velocities)
    for (int i = 0; i < 3; i++) {
        R a = 0;
        for (int j = 0; j < 6; j++) a += ppa[j] * K.get(j, i);
        y[i] = y[i] + h * (y[3 + i] * ps + h * a);
    }
    const int comp[kNK] = {3, 4, 5, 6, 7, 8, 9, 11, 12};
    for (int cidx = 0; cidx < kNK; cidx++) {
        R a = pp[6] * fnv[cidx];
        for (int j = 0; j < 6; j++) a += pp[j] * K.get(j, cidx);
        y[comp[cidx]] = y[comp[cidx]] + h * a;
    }
    y[13] = y[13] + h * (c.dm * ps);
}

// ------------------------------------------------------------------------------------------------
// x^(-1/5) for x > 0: the step-size controller's err^(-1/5) (rk.py:149-160) and the initial-step
// (0.01/max(d1,d2))^(1/5) (common.py:129).  Device: single-precision seed from the MUFU log2/exp2
// units, two Newton steps on y^-5 = x (quadratic: 1e-6 -> 1e-12 -> rounding).  Only the magnitude of
// the NEXT step depends on it, so 3 ulp here move the solution by < 1e-18.
R6_HD double inv_root5(double x)
{
#if defined(__CUDA_ARCH__)
    const float xf = fminf(fmaxf(__double2float_rn(x), 1e-30f), 1e30f);
    double y = (double)exp2f(-0.2f * __log2f(xf));
#pragma unroll
    for (int it = 0; it < 2; it++) {
        const double y2 = y * y;
        const double y5 = y2 * y2 * y;
        y = fma(0.2 * y, fma(-x, y5, 1.0), y);
    }
    return y;
#else
    return exp(-0.2 * log(x));
#endif
}
R6_HD float inv_root5(float x)
{
#if defined(__CUDA_ARCH__)
    const float xc = fminf(fmaxf(x, 1e-30f), 1e30f);
    float y = exp2f(-0.2f * __log2f(xc));
    const float y2 = y * y;
    return fmaf(0.2f * y, fmaf(-xc, y2 * y2 * y, 1.0f), y);
#else
    return expf(-0.2f * logf(x));
#endif
}

// ------------------------------------------------------------------------------------------------
// Evaluation point of one right-hand-side call: x = y + h sum_j SA[ROW][j] K_j (rk_step, rk.py:58-66), positions from
// the squared tableau.  One instantiation per row of the extended tableau, fully unrolled: the coefficients are
// constant-bank operands of the FMAs at fixed offsets, the stage loads are all issued up front, and only the height is
// formed for the stage rows (the horizontal positions enter nothing but y_new, row 6).  B[1] = 0: row 6 reads the
// velocity components of stage 1 only (for the position sums).
template <class R>
struct EvalPoint {
    R h, r1, r2, v0, v1, v2, q0, q1, q2, q3, w1, w2, m;
};
// The row's newest stage (K_{ROW-1}, rows 2..6) has just been produced and is still in registers: it is taken from
// `dn` instead of being read back.  Row 6 reads every stage, so it also forms the error-estimate sums
// es = sum_j E[j] K_j, er = sum_j EA[j] K_j[0..2] (rk.py:104-109) on the same loads; only E[6] f(y_new) is added later.
template <class R>
struct ErrSums {
    R es[kNK], er[3];
};
template <int ROW, class KS, class R>
R6_HD void stage_point(const KS &K, const R *y, R hh, R dm, EvalPoint<R> &x, const DerivT<R> &dn, ErrSums<R> &E)
{
    const TabT<R> &T = tab<R>();
    constexpr int cnt = ROW < 6 ? ROW : (ROW == 6 ? 6 : 1);
    constexpr bool kHoriz = ROW == 6;            // horizontal positions only for y_new
    constexpr bool kPos = ROW != 7;              // row 7 (probe) has no h^2 term
    constexpr bool kErr = ROW == 6;
    const R dnv[kNK] = {dn.dv0, dn.dv1, dn.dv2, dn.dq0, dn.dq1, dn.dq2, dn.dq3, dn.dw1, dn.dw2};
    R acc[kNK], ar0 = 0, ar1 = 0, ar2 = 0;
#pragma unroll
    for (int j = 0; j < cnt; j++) {
        const bool skip_a = (ROW == 6 && j == 1);                  // B[1] = E[1] = 0
        const bool newest = ROW >= 2 && ROW <= 6 && j == ROW - 1;
        const R a = T.SA[ROW][j], aa = T.SAA[ROW][j];
        const R e = kErr ? T.E[j] : R(0), ea = kErr ? T.EA[j] : R(0);
        R k[kNK];
        if (newest) {
#pragma unroll
            for (int i = 0; i < kNK; i++) k[i] = dnv[i];
        } else if (skip_a) {                              // velocity components only (position sums of y_new)
            const Pair<R> p0 = K.get2(j, 0), p1 = K.get2(j, 1);
            k[0] = p0.a; k[1] = p0.b; k[2] = p1.a;
#pragma unroll
            for (int i = 3; i < kNK; i++) k[i] = 0;
        } else {
#pragma unroll
            for (int p = 0; p < 4; p++) {
                const Pair<R> v = K.get2(j, p);
                k[2 * p] = v.a; k[2 * p + 1] = v.b;
            }
            k[8] = K.get(j, 8);
        }
        // j = 0 starts the sums with a product (no zeroed accumulators); SAA[ROW][0] = 0 only for ROW = 1 and 7
        if (kPos) ar0 = j == 0 ? aa * k[0] : fma(aa, k[0], ar0);
        if (kHoriz) { ar1 = j == 0 ? aa * k[1] : fma(aa, k[1], ar1); ar2 = j == 0 ? aa * k[2] : fma(aa, k[2], ar2); }
        if (kErr) {
#pragma unroll
            for (int i = 0; i < 3; i++) E.er[i] = j == 0 ? ea * k[i] : fma(ea, k[i], E.er[i]);
        }
        if (!skip_a) {
#pragma unroll
            for (int i = 0; i < kNK; i++) {
                acc[i] = j == 0 ? a * k[i] : fma(a, k[i], acc[i]);
                if (kErr) E.es[i] = j == 0 ? e * k[i] : fma(e, k[i], E.es[i]);
            }
        }
    }
    const R hc = hh * T.SC[ROW], hh2 = hh * hh;
    x.h = kPos ? fma(hh2, ar0, fma(hc, y[3], y[0])) : fma(hc, y[3], y[0]);
    if (kHoriz) {
        x.r1 = fma(hh2, ar1, fma(hc, y[4], y[1]));
        x.r2 = fma(hh2, ar2, fma(hc, y[5], y[2]));
    }
    x.v0 = fma(hh, acc[0], y[3]); x.v1 = fma(hh, acc[1], y[4]); x.v2 = fma(hh, acc[2], y[5]);
    x.q0 = fma(hh, acc[3], y[6]); x.q1 = fma(hh, acc[4], y[7]); x.q2 = fma(hh, acc[5], y[8]); x.q3 = fma(hh, acc[6], y[9]);
    x.w1 = fma(hh, acc[7], y[11]); x.w2 = fma(hh, acc[8], y[12]);
    x.m = fma(hc, dm, y[13]);
}

// ------------------------------------------------------------------------------------------------
// solve_ivp(fun, [t, t+dt], y, events=height) with all defaults.  y in/out (quaternion NOT yet
// re-normalised).  Returns the scipy status (0 / 1 / -1); natt = accepted + rejected RK attempts.
//
// Written as ONE loop around ONE right-hand-side evaluation: every RHS call of the algorithm — f0,
// the probe f(y + h0 f0) of select_initial_step, the stages 2..6 of every attempt and f(y_new) — goes
// through the same instructions, and what happens with the result is selected by `stage`.  The
// evaluation point is always  y + h * sum_j SA[row][j] K_j  (rows of the extended tableau above), built
// by one rolled loop.  This keeps the hot instruction footprint to a few KB (the instruction cache is
// what the unrolled formulation was bound by) at the price of a switch per evaluation.
//
// kPass (multi-pass integration, integrate_pass_kernel): the adaptive step count differs per env (1 attempt for a
// third of them, 2 for most, 3-4 rarely) and a warp pays for its slowest lane, so the step can also be cut at
// attempt boundaries: kPass = 1 starts normally and returns -2 ("unfinished") after px->budget attempts with the
// solver's private state in *px; kPass = 2 resumes from *px.  Only (t, h_abs, rejected, natt) and the height the
// density expansion was set up at are carried: f(y), the first-same-as-last stage, is re-evaluated from the stored y
// (same inputs, same instructions => the same bits).  kPass = 0 is the single-call form.
template <class R>
struct PassCtx {
    R t, h_abs, h_ref, t_bound;     // t_bound rides along so that a resumed pass needs neither step_count nor the time table
    int natt, budget;
    bool rejected;
};
#ifndef R6_ROWS_UNROLLED
#define R6_ROWS_UNROLLED 1      /* 1: stage_point<ROW> per row (switch) in the pass kernels; 0: the rolled loop everywhere */
#endif
template <bool kExact, class KS, class R, int kPass = 0>
R6_HD int integrate(StepConstT<R> &c, R *y, R t, R dt, int &natt, KS &K, PassCtx<R> &px)
{
    const TabT<R> &T = tab<R>();
    constexpr R rtol = R(1e-3), atol = R(1e-6);
    constexpr R inv_sqrt14 = R(0.2672612419124244);   // 1/sqrt(14)
    constexpr int kStageF0 = -1, kStageProbe = 0;        // stage >= 1: Dormand-Prince stage index (6 = f(y_new))
    // The pass kernels (one RK attempt per launch, nothing else in the kernel) take the unrolled per-row stage sums:
    // -11 % instructions, all stage loads in flight at once.  The fused step / rollout kernels keep the rolled loop:
    // their hot footprint (integrator + reward + reset in one kernel) is what the instruction cache bounds, and the
    // unrolled rows (+10 KB) cost them 7 % (rollout_fused 1.73e9 -> 1.61e9 env-steps/s).  Same arithmetic either way.
    constexpr bool kUnroll = R6_ROWS_UNROLLED != 0 && kPass != 0;
    const R t_bound = kPass == 2 ? px.t_bound : t + dt;
    const R L = fabs(t_bound - t);                       // common.py:100 (interval length as SciPy computes it)
    if constexpr (kPass == 2) density_setup(c, px.h_ref);
    else density_setup(c, y[0]);
    // evaluation point (height, v, q, w1, w2, m) + the two horizontal positions of y_new
    EvalPoint<R> x = {y[0], y[1], y[2], y[3], y[4], y[5], y[6], y[7], y[8], y[9], y[11], y[12], y[13]};
    int stage = kStageF0;
    R h = 0, h_abs = 0, t_new = t;
    ErrSums<R> esum;              // written by stage_point<6>, read when f(y_new) comes back (unrolled form only)
    R g = y[0];
    int status = -2;
    bool rejected = false;
    natt = 0;
    int budget = 0;
    if constexpr (kPass != 0) budget = px.budget;
    if constexpr (kPass == 1) { px.h_ref = y[0]; px.t_bound = t_bound; }
    if constexpr (kPass == 2) { t = px.t; t_new = t; h_abs = px.h_abs; rejected = px.rejected; natt = px.natt; }
    for (;;) {
        const DerivT<R> d = rhs<kExact>(c, x.h, x.v0, x.v1, x.v2, x.q0, x.q1, x.q2, x.q3, x.w1, x.w2, x.m);
        bool begin_attempt = false;
        int row;
        R hh;
        if (stage >= 1 && stage <= 5) {
            k_store(K, stage, d);
            stage += 1;
            row = stage; hh = h;
        } else if (stage == 6) {
            // ---- d = f(y_new): error estimate (rk.py:104-109, 141-142), accept / reject (rk.py:144-163) ----
            R es[kNK], er[3];
#pragma unroll
            for (int i = 0; i < kNK; i++) es[i] = 0;
#pragma unroll
            for (int i = 0; i < 3; i++) er[i] = 0;
            if constexpr (kUnroll) {
                // the sums over the six stored stages were formed together with y_new (stage_point<6>)
#pragma unroll
                for (int i = 0; i < kNK; i++) es[i] = esum.es[i];
#pragma unroll
                for (int i = 0; i < 3; i++) er[i] = esum.er[i];
            } else {
#pragma unroll 1
                for (int j = 0; j < 6; j++) {
                    const R e = T.E[j], ea = T.EA[j];
#pragma unroll
                    for (int i = 0; i < kNK; i++) {
                        const R k = K.get(j, i);
                        es[i] = fma(e, k, es[i]);
                        if (i < 3) er[i] = fma(ea, k, er[i]);
                    }
                }
            }
            const R e6 = T.E[6];
            const R fnv[kNK] = {d.dv0, d.dv1, d.dv2, d.dq0, d.dq1, d.dq2, d.dq3, d.dw1, d.dw2};
            const R yo[12] = {y[0], y[1], y[2], y[3], y[4], y[5], y[6], y[7], y[8], y[9], y[11], y[12]};
            const R yw[12] = {x.h, x.r1, x.r2, x.v0, x.v1, x.v2, x.q0, x.q1, x.q2, x.q3, x.w1, x.w2};
            // err^2 14 = sum_i (e_i / sc_i)^2 with e_i = h^2 er_i (positions), h (es_i + E6 fn_i) (the rest): the powers of
            // h are factored out of the sums; the w0 and mass rows contribute exactly 0 to the error norm
            R sr = 0, so = 0;
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const R isc = fast_rcp1(fma(fmax(fabs(yo[i]), fabs(yw[i])), rtol, atol));
                const R q = (i < 3 ? er[i] : fma(e6, fnv[i < 3 ? 0 : i - 3], es[i < 3 ? 0 : i - 3])) * isc;
                if (i < 3) sr = fma(q, q, sr);
                else so = fma(q, q, so);
            }
            const R err = fabs(h) * fast_sqrt(fma(h * h, sr, so)) * inv_sqrt14;
            const R raw = (err == 0) ? R(10.0) : R(0.9) * inv_root5(err);        // SAFETY * err^(-1/5)
            if (err < 1) {
                R factor = fmin(R(10.0), raw);
                if (rejected) factor = fmin(R(1.0), factor);
                h_abs *= factor;
                // accepted: ivp.py:659-699
                const R t_old = t;
                const R g_new = x.h;
                const bool ev = (g <= 0 && g_new >= 0) || (g >= 0 && g_new <= 0);
                t = t_new;
                if (t - t_bound >= 0) status = 0;
                if (ev) {
                    const DerivT<R> fn = d;                         // the address-taken copy exists on this rare path only
                    event_resolve(c, y, K, fn, t_old, t_new);
                    status = 1;
                } else {
                    y[0] = x.h; y[1] = x.r1; y[2] = x.r2; y[3] = x.v0; y[4] = x.v1; y[5] = x.v2;
                    y[6] = x.q0; y[7] = x.q1; y[8] = x.q2; y[9] = x.q3; y[11] = x.w1; y[12] = x.w2; y[13] = x.m;
                }
                if (status != -2) break;
                k_store(K, 0, d);                                   // first-same-as-last
                g = g_new;
                rejected = false;
            } else {
                h_abs *= fmax(R(0.2), raw);
                rejected = true;
            }
            if constexpr (kPass != 0) {
                if (--budget == 0) {                                // hand the env to the next pass
                    px.t = t; px.h_abs = h_abs; px.rejected = rejected; px.natt = natt;
                    break;
                }
            }
            begin_attempt = true;
        } else if (kPass == 2 && stage == kStageF0) {
            k_store(K, 0, d);                                       // f(y) again: the first-same-as-last stage
            begin_attempt = true;
        } else if (stage == kStageF0) {
            // ---- d = f0 (rk.py:96); select_initial_step part 1 (common.py:105-119), order 4 ----
            k_store(K, 0, d);
            R s0 = 0, s1 = 0;
            const R fv[14] = {y[3], y[4], y[5], d.dv0, d.dv1, d.dv2, d.dq0, d.dq1, d.dq2, d.dq3, R(0), d.dw1, d.dw2, c.dm};
#pragma unroll
            for (int i = 0; i < 14; i++) {
                const R isc = fast_rcp1(fma(fabs(y[i]), rtol, atol));
                s0 += sq(y[i] * isc);
                if (i != 10) s1 += sq(fv[i] * isc);
                // the 12 scales the probe needs again (all rows but w0 and the mass) wait in the still unused slots of
                // stages 1 and 2
                if (i != 10 && i != 13) { const int s = i < 10 ? i : i - 1; K.set(1 + s / kNK, s % kNK, isc); }
            }
            const R d0 = fast_sqrt(s0) * inv_sqrt14, d1 = fast_sqrt(s1) * inv_sqrt14;
            R h0 = (d0 < R(1e-5) || d1 < R(1e-5)) ? R(1e-6) : R(0.01) * d0 * fast_rcp(d1);
            h0 = fmin(h0, L);
            h = h0;            // probe step; d1 is parked in h_abs until the probe comes back
            h_abs = d1;
            stage = kStageProbe;
            row = 7; hh = h0;
        } else {
            // ---- d = f(y + h0 f0); select_initial_step part 2 (common.py:121-134) ----
            const R h0 = h, d1 = h_abs;
            // (f1 - f0)/scale: position rows are h0*dv, the w0 and mass rows are 0
            const R f1v[kNK] = {d.dv0, d.dv1, d.dv2, d.dq0, d.dq1, d.dq2, d.dq3, d.dw1, d.dw2};
            R sp = 0, so = 0;
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const R isc = K.get(1 + i / kNK, i % kNK);
                const R q = (i < 3 ? K.get(0, i) : f1v[i < 3 ? 0 : i - 3] - K.get(0, i < 3 ? 0 : i - 3)) * isc;
                if (i < 3) sp = fma(q, q, sp);
                else so = fma(q, q, so);
            }
            const R d2 = fast_sqrt(fma(h0 * h0, sp, so)) * inv_sqrt14 * fast_rcp(h0);
            const R tiny15 = R(1e-15);
            const R h1 = (d1 <= tiny15 && d2 <= tiny15) ? fmax(R(1e-6), h0 * R(1e-3)) : inv_root5(R(100.0) * fmax(d1, d2));
            h_abs = fmin(fmin(100 * h0, h1), L);
            begin_attempt = true;
        }
        if (begin_attempt) {
            // ---- RungeKutta._step_impl entry (rk.py:111-131) ----
            const R min_step = 10 * fabs(r_nextafter_up(t) - t);
            if (h_abs < min_step) {
                if (rejected) { status = -1; break; }
                h_abs = min_step;
            }
            t_new = t + h_abs;
            if (t_new - t_bound > 0) t_new = t_bound;
            h = t_new - t;
            h_abs = fabs(h);
            natt++;
            stage = 1;
            row = 1; hh = h;
        }
        // ---- evaluation point of the next RHS call: rk_step (rk.py:58-66) with the row's coefficients ----
        if constexpr (kUnroll) {
            switch (row) {
            case 1: stage_point<1>(K, y, hh, c.dm, x, d, esum); break;
            case 2: stage_point<2>(K, y, hh, c.dm, x, d, esum); break;
            case 3: stage_point<3>(K, y, hh, c.dm, x, d, esum); break;
            case 4: stage_point<4>(K, y, hh, c.dm, x, d, esum); break;
            case 5: stage_point<5>(K, y, hh, c.dm, x, d, esum); break;
            case 6: stage_point<6>(K, y, hh, c.dm, x, d, esum); break;
            default: stage_point<7>(K, y, hh, c.dm, x, d, esum); break;
            }
        } else {
            R acc[kNK], ar0 = 0, ar1 = 0, ar2 = 0;
#pragma unroll
            for (int i = 0; i < kNK; i++) acc[i] = 0;
            const int cnt = row < 6 ? row : (row == 6 ? 6 : 1);
#pragma unroll 1
            for (int j = 0; j < cnt; j++) {
                const R a = T.SA[row][j], aa = T.SAA[row][j];
                const R k0 = K.get(j, 0), k1 = K.get(j, 1), k2 = K.get(j, 2);
                acc[0] = fma(a, k0, acc[0]); acc[1] = fma(a, k1, acc[1]); acc[2] = fma(a, k2, acc[2]);
                ar0 = fma(aa, k0, ar0); ar1 = fma(aa, k1, ar1); ar2 = fma(aa, k2, ar2);
#pragma unroll
                for (int i = 3; i < kNK; i++) acc[i] = fma(a, K.get(j, i), acc[i]);
            }
            const R hc = hh * T.SC[row], hh2 = hh * hh;
            x.h = fma(hh2, ar0, fma(hc, y[3], y[0]));
            x.r1 = fma(hh2, ar1, fma(hc, y[4], y[1]));
            x.r2 = fma(hh2, ar2, fma(hc, y[5], y[2]));
            x.v0 = fma(hh, acc[0], y[3]); x.v1 = fma(hh, acc[1], y[4]); x.v2 = fma(hh, acc[2], y[5]);
            x.q0 = fma(hh, acc[3], y[6]); x.q1 = fma(hh, acc[4], y[7]); x.q2 = fma(hh, acc[5], y[8]); x.q3 = fma(hh, acc[6], y[9]);
            x.w1 = fma(hh, acc[7], y[11]); x.w2 = fma(hh, acc[8], y[12]);
            x.m = fma(hc, c.dm, y[13]);
        }
    }
    return status;
}

// the single-call form (kPass = 0)
template <bool kExact, class KS, class R>
R6_HD int integrate(StepConstT<R> &c, R *y, R t, R dt, int &natt, KS &K)
{
    PassCtx<R> px{};
    return integrate<kExact, KS, R, 0>(c, y, t, dt, natt, K, px);
}

// ------------------------------------------------------------------------------------------------
// t_go of rocket_env.py:528-546: largest positive real root of f(t) = c0 t^4 + c2 t^2 + c3 t + c4
// (np.roots' first eigenvalue with imag == 0 and real > 0 is the largest positive real root,
// SURVEY §A.4).  Bracketing strategy (f''' > 0 on t > 0 so f' is convex there):
//   * t_i = sqrt(-c2/(6 c0)) is the inflection point; f is convex on (t_i, inf).
//   * if f(t_i) <= 0 the largest root lies in the convex region: Newton from an upper bound is monotone.
//   * else if f' >= 0 at t_i, f is increasing on t > 0: single root in (0, t_i), f concave there:
//     Newton from the left is monotone.
//   * else f has a local minimum at s2 > t_i (found by monotone Newton on the convex f'); the largest
//     root is right of s2 if f(s2) <= 0, otherwise it is the single root left of t_i.
// Every Newton step is safeguarded by the bracket (falls back to bisection), so it terminates.
template <class W>
R6_HD W quartic_f(W c0, W c2, W c3, W c4, W t)
{
    W t2 = t * t;
    return fma(fma(c0, t2, c2), t2, fma(c3, t, c4));
}
template <class W>
R6_HD W quartic_df(W c0, W c2, W c3, W t)
{
    return fma(fma(4 * c0, t * t, 2 * c2), t, c3);
}
// Cold start of tgo_largest_root (no usable warm start): bracketing by the convexity analysis above + safeguarded Newton.
// Out of line: with R6Buffers.tgo the step kernels take it for freshly reset envs and the rare third sign pattern only.
template <class W>
R6_HD_NOINLINE W tgo_cold_start(W c0, W c2, W c3, W c4, W ic0, W ti)
{
    // Fujiwara bound on the root moduli; float32 is plenty for a bound (inflated by 1e-4)
    const float a2 = (float)(fabs(c2) * ic0), a1 = (float)(fabs(c3) * ic0), a0 = (float)(fabs(c4) * ic0);
    const W B = (W)(2.0002f * fmaxf(sqrtf(a2), fmaxf(cbrtf(a1), sqrtf(sqrtf(0.5f * a0)))));
    if (!(B > 0) || !isfinite(B)) return W(NAN);
    W lo = 0, hi = B;
    bool from_right = true;
    if (ti > 0 && ti < B) {
        const W fi = quartic_f(c0, c2, c3, c4, ti);
        if (fi <= 0) { lo = ti; }
        else {
            const W gi = quartic_df(c0, c2, c3, ti);
            if (gi >= 0) { hi = ti; from_right = false; }
            else {
                // local minimum s2 > ti: monotone Newton on f' (convex on t > 0) from the right
                W s = B;
                for (int it = 0; it < 60; it++) {
                    const W d1 = quartic_df(c0, c2, c3, s);
                    const W d2 = fma(12 * c0, s * s, 2 * c2);
                    if (!(d2 > 0)) break;
                    const W sn = s - d1 * fast_rcp(d2);
                    if (!(sn < s) || sn <= ti) { break; }
                    s = sn;
                }
                const W fs = quartic_f(c0, c2, c3, c4, s);
                if (fs <= 0) { lo = s; }
                else { hi = ti; from_right = false; }   // f > 0 on [ti, inf): the root is left of ti
            }
        }
    }
    const W flo = quartic_f(c0, c2, c3, c4, lo), fhi = quartic_f(c0, c2, c3, c4, hi);
    if (flo == 0 && lo > 0) return lo;
    if (!(flo < 0) || !(fhi > 0)) {
        if (fhi == 0) return hi;
        return W(NAN);
    }
    W hi_s = hi, fhi_s = fhi;
    bool certified = false;      // bracket inside the convex region AND tightened to ~1e-5 by the float32 walk
    if (from_right && sizeof(W) == 8) {
        // The far end of the bracket is the Fujiwara bound, from which Newton on a quartic first creeps in
        // by factors of 3/4.  Walk that stretch in float32 (FP32 pipe, no safeguards needed: the result is
        // only a PROPOSAL for a tighter upper end, accepted if float64 confirms lo < x < hi and f(x) > 0).
        const float g0 = (float)c0, g2 = (float)c2, g3 = (float)c3, g4 = (float)c4;
        const float g0x4 = 4.0f * g0, g2x2 = 2.0f * g2;
        float xf = (float)hi;
#pragma unroll 1
        for (int it = 0; it < 48; it++) {
            const float x2 = xf * xf;
            const float f = f32_fma(f32_fma(g0, x2, g2), x2, f32_fma(g3, xf, g4));
            const float df = f32_fma(f32_fma(g0x4, x2, g2x2), xf, g3);
            const float xn = xf - f * (float)fast_rcp(df);
            if (!(xf - xn > 2e-6f * xf)) break;
            xf = xn;
        }
        const W xs = (W)xf * W(1.0 + 1e-5);
        if (xs > lo && xs < hi) {
            const W fs = quartic_f(c0, c2, c3, c4, xs);
            if (fs > 0) { hi_s = xs; fhi_s = fs; certified = !(ti >= B); }
        }
    }
    hi = hi_s;
    // start from the upper end in both cases: in the convex case Newton is monotone from there; in the concave case
    // (root left of the inflection point) its first step overshoots to the left of the root and is monotone after
    // that, whereas starting at lo = 0 with f'(0) = c3 <= 0 would fall back to bisection for many iterations
    W x = hi_s;
    W fx = fhi_s;
    if (certified) {
        // f is convex on [lo, hi] with f(lo) <= 0 < f(hi) and hi within ~1e-5 of the root: plain Newton from hi is
        // monotone, cannot leave the bracket and converges quadratically (1e-5 -> 1e-10 -> 1e-20): three bare steps,
        // no bracket bookkeeping.  If the third step still moved, fall through to the safeguarded loop.
        W dx = 0;
#pragma unroll
        for (int it = 0; it < 3; it++) {
            dx = fx * fast_rcp(quartic_df(c0, c2, c3, x));
            x -= dx;
            fx = quartic_f(c0, c2, c3, c4, x);
        }
        if (!(fabs(dx) <= W(1e-11) * fabs(x))) { certified = false; x = hi_s; fx = fhi_s; }
    }
    for (int it = 0; it < 100 && !certified; it++) {
        const W dfx = quartic_df(c0, c2, c3, x);
        W xn = x - fx * fast_rcp(dfx);
        if (fabs(xn - x) <= 2 * Real<W>::eps * fabs(x)) break;   // converged (monotone Newton stalls at the root)
        if (!(xn >= lo && xn <= hi)) xn = W(0.5) * (lo + hi);        // safeguard: bisection
        const W fn_ = quartic_f(c0, c2, c3, c4, xn);
        x = xn; fx = fn_;
        if (fn_ > 0) hi = xn; else if (fn_ < 0) lo = xn; else break;
        if (hi - lo <= Real<W>::eps * hi) break;
    }
    // final polish: one unconditional Newton step with a true division (converged iterates barely move)
    {
        const W dfx = quartic_df(c0, c2, c3, x);
        if (dfx != 0) {
            const W xn = x - quartic_f(c0, c2, c3, c4, x) / dfx;
            if (xn > 0 && fabs(xn - x) <= W(sizeof(W) == 8 ? 1e-9 : 1e-4) * x) x = xn;
        }
    }
    return x;
}

// `guess` (optional warm start, 0 = none): the root found for the same env one step earlier.  t_go moves by about dt
// per env-step, so Newton from the previous root needs 3-4 steps instead of the ~10 + 3 of the cold start from the
// Fujiwara bound.  A warm result is accepted only when it is CERTIFIED to be the largest positive root:
//   (A) f(t_i) <= 0 (or no inflection point): the largest root is the only root right of t_i, where f is convex and
//       tends to +inf — any converged iterate x > t_i with f'(x) > 0 is it;
//   (B) f(t_i) > 0 and f'(t_i) >= 0: f' has its minimum at t_i, so f increases on all of t > 0 and has exactly one
//       positive root, inside (0, t_i) — any converged iterate there is it.
// Anything else — the third sign pattern (a local minimum right of t_i decides), an iterate leaving the interval, a
// non-positive slope, no convergence in 6 steps — falls back to the cold start below.
template <class W>
R6_HD W tgo_largest_root(W c0, W c2, W c3, W c4, W guess = W(0))
{
    if (!(c4 < 0) && !(c3 < 0) && !(c2 < 0)) return W(NAN);       // no sign change => no positive root
    const W ic0 = fast_rcp(c0);
    const W ti = (c2 < 0) ? fast_sqrt(-c2 * ic0 * W(1.0 / 6)) : W(0.0);
    if (guess > 0) {
        W lo = ti, hi = W(INFINITY);                              // case (A)
        bool usable = true;
        if (ti > 0) {
            const W fi = quartic_f(c0, c2, c3, c4, ti);
            if (fi > 0) {
                if (quartic_df(c0, c2, c3, ti) >= 0) { lo = 0; hi = ti; }      // case (B)
                else usable = false;
            }
        }
        W x = fmin(guess, hi);
        if (usable && x > lo) {
            W fx = quartic_f(c0, c2, c3, c4, x), dx = x;
            bool conv = false;
#pragma unroll 1
            for (int it = 0; it < 6; it++) {
                const W dfx = quartic_df(c0, c2, c3, x);
                if (!(dfx > 0)) break;
                dx = fx * fast_rcp(dfx);
                x -= dx;
                if (!(x > lo && x <= hi)) break;
                fx = quartic_f(c0, c2, c3, c4, x);
                // quadratic convergence: a correction below 1e-8 x leaves an error of ~1e-16 x
                if (fabs(dx) <= W(sizeof(W) == 8 ? 1e-8 : 1e-4) * x) { conv = true; break; }
            }
            if (conv) {
                const W dfx = quartic_df(c0, c2, c3, x);
                if (dfx > 0) {
                    const W xn = x - fx * fast_rcp(dfx);          // polish: rounding level
                    if (xn > lo && xn <= hi) return xn;
                }
            }
        }
    }
    return tgo_cold_start(c0, c2, c3, c4, ic0, ti);
}

// ------------------------------------------------------------------------------------------------
// Host-derived thresholds for the Euler-angle limit tests (computed once per call on the host)
struct AngleTests {
    // violation test |e_i| > L_i (rocket_env.py:366-369): mode 0 = never (L >= range), 1 = compare
    int viol_mode[3];
    double viol_thr[3];    // cos(L0), sin(L1), cos(L2)
    // landing test |e_i| < L_i (rocket_env.py:386-388): mode 0 = never (L <= 0), 1 = compare, 2 = always
    int land_mode[3];
    double land_thr[3];
};
inline AngleTests make_angle_tests(const double viol[3], const double land[3])
{
    AngleTests a;
    const double pi = 3.14159265358979323846;
    for (int i = 0; i < 3; i++) {
        const double range = (i == 1) ? pi / 2 : pi;     // |e1| <= pi/2, |e0|,|e2| <= pi
        a.viol_mode[i] = (viol[i] >= range) ? 0 : 1;
        a.viol_thr[i] = (i == 1) ? sin(viol[i]) : cos(viol[i]);
        if (viol[i] < 0) { a.viol_mode[i] = 2; }          // |e| > negative: always
        a.land_mode[i] = (land[i] > range) ? 2 : ((land[i] <= 0) ? 0 : 1);
        a.land_thr[i] = (i == 1) ? sin(land[i]) : cos(land[i]);
    }
    return a;
}

// Everything the kernels need that is derived from R6Params on the host once per call
struct Derived {
    AngleTests at;
    double inv_norm[R6_NSTATE];   // RN(1 / normalizer[i]) for the exact 3-instruction division below
    float inv_norm_f[R6_NSTATE];  // the same in float32 (fp32 path: obs = y * inv_norm_f, 1 ulp)
};
inline Derived make_derived(const R6Params &p)
{
    Derived d;
    d.at = make_angle_tests(p.att_traj_limit, p.land_att_limit);
    for (int i = 0; i < R6_NSTATE; i++) {
        d.inv_norm[i] = 1.0 / p.normalizer[i];
        d.inv_norm_f[i] = (float)d.inv_norm[i];
    }
    return d;
}
// Correctly rounded a / b from r = RN(1/b) (Markstein): q = a r; q' = q + (a - b q) r.
// Bit-identical to the IEEE division of rocket_env.py:503-504 (b is a normal number, no overflow).
R6_HD double div_exact(double a, double b, double rinv)
{
    const double q = a * rinv;
    const double rem = fma(-q, b, a);
    return fma(rem, rinv, q);
}
R6_HD float obs_scalar(const R6Params &p, const Derived &dv, double yi, int i)
{
    return f64_to_f32(div_exact(yi, p.normalizer[i], dv.inv_norm[i]));
}
R6_HD float obs_scalar(const R6Params &, const Derived &dv, float yi, int i) { return yi * dv.inv_norm_f[i]; }
template <class R>
R6_HD float obs_component(const R6Params &p, const Derived &dv, const R *y, int i) { return obs_scalar(p, dv, y[i], i); }

// Extrinsic zyx Euler angles of the float32-cast quaternion (scipy _rotation_xp.py:365-401,
// 1052-1111), reduced to what the env needs: the two limit tests.  With a = w-y, b = z-x, c = y+w,
// d = -x-z:  cos(e0) = (ac+bd)/(|ab||cd|), sin(e1) = (|cd|^2-|ab|^2)/(|ab|^2+|cd|^2),
// cos(e2) = (ac-bd)/(|ab||cd|); gimbal lock (|e1 +- pi/2| <= 1e-7): e0 = 2 hs or -2 hd, e2 = 0.
template <class W>
R6_HD void euler_limit_tests(const AngleTests &at, W w, W x, W y, W z, bool &violated,
                             bool &land_ok)
{
    const W a = w - y, b = z - x, c = y + w, d = -x - z;
    const W Q2 = a * a + b * b, P2 = c * c + d * d;
    constexpr W tan2_lock = W(2.5e-15);     // tan(5e-8)^2
    const bool case1 = P2 <= tan2_lock * Q2;
    const bool case2 = Q2 <= tan2_lock * P2;
    W cos0, cos2;
    if (!(case1 || case2)) {
        const W inv = fast_rcp(fast_sqrt(Q2 * P2));
        cos0 = (a * c + b * d) * inv;
        cos2 = (a * c - b * d) * inv;
    } else if (case1) {
        cos0 = (a * a - b * b) / Q2; cos2 = W(1.0);
    } else {
        cos0 = (c * c - d * d) / P2; cos2 = W(1.0);
    }
    const W sin1 = (P2 - Q2) / (P2 + Q2);
    const W m[3] = {cos0, fabs(sin1), cos2};
    violated = false;
    land_ok = false;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        // |e| > L  <=>  cos e < cos L  (i = 0, 2)   |  |sin e1| > sin L (i = 1)
        bool v = (i == 1) ? (m[i] > (W)at.viol_thr[i]) : (m[i] < (W)at.viol_thr[i]);
        v = (at.viol_mode[i] == 1) ? v : (at.viol_mode[i] == 2);
        bool l = (i == 1) ? (m[i] < (W)at.land_thr[i]) : (m[i] > (W)at.land_thr[i]);
        l = (at.land_mode[i] == 1) ? l : (at.land_mode[i] == 2);
        violated = violated || v;
        land_ok = land_ok || l;
    }
}

// ------------------------------------------------------------------------------------------------
// rocket_env.py:509-521 for a float32 action array
R6_HD void denormalize_action(const R6Params &p, float a0, float a1, float a2, float &u0, float &u1, float &u2)
{
    u0 = f64_to_f32((double)a0 * p.max_gimbal);
    u1 = f64_to_f32((double)a1 * p.max_gimbal);
    u2 = f32_mul(f32_div(f32_add(a2, 1.0f), 2.0f), p.max_thrust);
}

struct PostOut {
    double reward;        // after the out-of-bounds penalty, before ClipReward
    double terms[R6_NTERMS];
    uint32_t flags;       // R6_F_* (EVENT, OOB and the five landing flags)
    bool tgo_missing;
    float tgo;            // the t_go root of this step (warm start of the next step's iteration), 0 when there is none
};

// rocket_env.py:206-231 after the simulator step.  S = post-step state with the quaternion already
// re-normalised in float64 (simulator.py:97).
// W = working precision of the float64 parts of the reference's reward (t_go root, a_targ, thrust rotation, Euler
// tests): double on the parity path (S = the float64 state), float on the float32 path (S = the float32 state; the
// reward then carries float32 round-off, inside that path's own bound).
R6_HD float to_f32(double x) { return f64_to_f32(x); }
R6_HD float to_f32(float x) { return x; }
R6_HD double w_exp(double x) { return exp(x); }
R6_HD float w_exp(float x) { return expf(x); }
template <class RS, class W>
R6_HD void post_step(const R6Params &p, const AngleTests &at, const StepConstT<RS> &cr, const W *S, float u2,
                     float v0_episode, int status, PostOut &o, float tgo_guess = 0.0f)
{
    struct { W Tb0, Tb1, Tb2; } c = {(W)cr.Tb0, (W)cr.Tb1, (W)cr.Tb2};
    float s[14];
#pragma unroll
    for (int i = 0; i < 14; i++) s[i] = to_f32(S[i]);                          // :206
    const float m = s[13];
    const bool oob = !(s[0] >= p.bounds_low[0] && s[0] <= p.bounds_high[0] && s[1] >= p.bounds_low[1] &&
                       s[1] <= p.bounds_high[1] && s[2] >= p.bounds_low[2] && s[2] <= p.bounds_high[2]);   // :591-593
    const float vn = f32_sqrt(sdot3(s[3], s[4], s[5], s[3], s[4], s[5]));
    const float rn = f32_sqrt(sdot3(s[0], s[1], s[2], s[0], s[1], s[2]));
    bool att_viol, att_land;
    euler_limit_tests(at, (W)s[6], (W)s[7], (W)s[8], (W)s[9], att_viol, att_land);
    W shaping;
    o.tgo_missing = false;
    o.tgo = 0.0f;
    if (!p.shaping_velocity) {
        // _compute_atarg (:526-566)
        const W c0 = W((-9.81) * (-9.81));
        const float c2 = f32_mul(-4.0f, f32_mul(vn, vn));
        const float c3 = f32_mul(-24.0f, sdot3(s[0], s[1], s[2], s[3], s[4], s[5]));
        const float c4 = f32_mul(-36.0f, f32_mul(rn, rn));
        W tgo = tgo_largest_root(c0, (W)c2, (W)c3, (W)c4, (W)tgo_guess);
        // no positive real root (the reference raises IndexError at rocket_env.py:545): cannot happen for r != 0 (the
        // quartic is negative at 0 and positive at infinity); for r = 0 exactly the target acceleration is defined as
        // that of t_go -> infinity (a_targ = -g), which keeps the reward finite instead of poisoning the statistics
        o.tgo_missing = !(tgo > 0);
        W itg = fast_rcp(tgo);
        if (o.tgo_missing) itg = W(0.0);
        else o.tgo = to_f32(tgo);
        const W itg2 = itg * itg;
        const W q0 = (W)f32_mul(-6.0f, s[0]) * itg2 - (W)f32_mul(4.0f, s[3]) * itg + W(9.81);
        const W q1 = (W)f32_mul(-6.0f, s[1]) * itg2 - (W)f32_mul(4.0f, s[4]) * itg;
        const W q2 = (W)f32_mul(-6.0f, s[2]) * itg2 - (W)f32_mul(4.0f, s[5]) * itg;
        const W U = (W)f32_div(p.max_thrust, m);
        const W qn = fast_sqrt(q0 * q0 + q1 * q1 + q2 * q2);
        const W k = (qn <= U) ? W(1.0) : U * fast_rcp(qn);
        // thrust acceleration from the float64 post-step quaternion (:339-340, simulator.py:177-186)
        RotUT<W> R = rot_unnormalised(S[6], S[7], S[8], S[9]);
        const W im = fast_rcp(R.n2 * (W)m);
        const W d0 = (R.m00 * c.Tb0 + R.m01 * c.Tb1 + R.m02 * c.Tb2) * im - q0 * k;
        const W d1 = (R.m10 * c.Tb0 + R.m11 * c.Tb1 + R.m12 * c.Tb2) * im - q1 * k;
        const W d2 = (R.m20 * c.Tb0 + R.m21 * c.Tb1 + R.m22 * c.Tb2) * im - q2 * k;
        shaping = (W)p.alfa * fast_sqrt(d0 * d0 + d1 * d1 + d2 * d2);
    } else {
        // _compute_vtarg (:646-674) + :349
        W rh0, rh1, rh2, vh0, tau;
        if ((W)s[0] > (W)p.waypoint) {
            rh0 = (W)s[0] - (W)p.waypoint; rh1 = s[1]; rh2 = s[2];
            vh0 = (W)s[3] + W(2.0); tau = 20;
        } else {
            rh0 = (W)f32_add(s[0], 1.0f); rh1 = 0; rh2 = 0;
            vh0 = (W)s[3] + W(1.0); tau = 100;
        }
        const W rh = sqrt(rh0 * rh0 + rh1 * rh1 + rh2 * rh2);
        const W vh = sqrt(vh0 * vh0 + (W)s[4] * (W)s[4] + (W)s[5] * (W)s[5]);
        const W tg = rh / vh, kk = 1 - w_exp(-tg / tau), den = fmax(W(1e-3), rh);
        const W mv0 = (W)(-v0_episode);
        const W d0 = (W)s[3] - (mv0 * (rh0 / den)) * kk;
        const W d1 = (W)s[4] - (mv0 * (rh1 / den)) * kk;
        const W d2 = (W)s[5] - (mv0 * (rh2 / den)) * kk;
        shaping = (W)p.alfa * sqrt(d0 * d0 + d1 * d1 + d2 * d2);
    }
    const float pen = f32_mul(p.beta, u2);                                     // :355
    const double att = att_viol ? p.gamma : 0.0;                               // :366-369
    // landing conditions (:382-390)
    const bool f_zero = s[0] <= p.zero_height_tol;
    const bool f_vel = vn < p.maximum_v;
    const bool f_rad = rn < p.target_r;
    const bool f_att = att_land;
    const bool f_om = fabs((double)s[10]) < p.omega_lim[0] || fabs((double)s[11]) < p.omega_lim[1] ||
                      fabs((double)s[12]) < p.omega_lim[2];
    const double goal = (f_zero && f_vel && f_rad && f_att && f_om) ? p.kappa : 0.0;
    const float dr = f32_sub(p.max_r_f, rn);
    const double final_pos = dr > 0 ? (double)f32_mul(dr, p.w_r_f) : 0.0;      // :400
    const float dv = f32_sub(p.max_v_f, vn);
    const double final_vel = (rn < p.max_r_f && f_zero) ? (dv > 0 ? (double)f32_mul(dv, p.w_v_f) : 0.0) : 0.0;   // :401
    double reward = 0;
    reward += (double)shaping; reward += (double)pen; reward += p.eta; reward += att; reward += goal;
    reward += final_pos; reward += final_vel;                                  // :362
    if (oob) reward += p.oob_penalty;                                          // :228-229
    o.reward = reward;
    o.terms[0] = (double)shaping; o.terms[1] = (double)pen; o.terms[2] = p.eta; o.terms[3] = att;
    o.terms[4] = goal; o.terms[5] = final_pos; o.terms[6] = final_vel;
    uint32_t fl = 0;
    if (status != 0) fl |= R6_F_EVENT;
    if (oob) fl |= R6_F_OOB;
    if (f_zero) fl |= R6_F_ZERO_HEIGHT;
    if (f_vel) fl |= R6_F_VEL_LIMIT;
    if (f_rad) fl |= R6_F_LAND_RADIUS;
    if (f_att) fl |= R6_F_ATT_LIMIT;
    if (f_om) fl |= R6_F_OMEGA_LIMIT;
    o.flags = fl;
}

template <class R>
R6_HD void normalize_quat(R *y)    // simulator.py:97, 153-154
{
    const R rn = fast_rcp(fast_sqrt(y[6] * y[6] + y[7] * y[7] + y[8] * y[8] + y[9] * y[9]));
    y[6] *= rn; y[7] *= rn; y[8] *= rn; y[9] *= rn;
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter-based: key = seed, counter = (env lo, env hi, a, b)
struct U4 { uint32_t x, y, z, w; };
R6_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32); }
R6_HD U4 philox4x32_10(U4 ctr, uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = mulhi32(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = mulhi32(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        U4 n;
        n.x = hi1 ^ ctr.y ^ k0; n.y = lo1; n.z = hi0 ^ ctr.w ^ k1; n.w = lo0;
        ctr = n;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return ctr;
}
// 53-bit uniform in [0,1) from two 32-bit words (the construction of numpy's random_sample)
R6_HD double u53(uint32_t a, uint32_t b)
{
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}
constexpr uint32_t kStreamReset = 0x52534554u;    // 'RSET' + block index
constexpr uint32_t kStreamAction = 0x41435431u;   // 'ACT1'

// Rocket6DOF.reset (rocket_env.py:180-199): Box.sample (float64 uniform, cast to float32), float32
// quaternion normalisation, float32 initial condition.
R6_HD void sample_initial_condition(const R6Params &p, uint64_t seed, uint64_t genv, uint32_t episode, float *ic)
{
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll 1
    for (int b = 0; b < 7; b++) {
        U4 ctr = {(uint32_t)genv, (uint32_t)(genv >> 32), episode, kStreamReset + (uint32_t)b};
        U4 r = philox4x32_10(ctr, k0, k1);
        const double ua = u53(r.x, r.y), ub = u53(r.z, r.w);
        const int i = 2 * b;
        ic[i] = f64_to_f32((double)p.ic_low[i] + ((double)p.ic_high[i] - (double)p.ic_low[i]) * ua);
        ic[i + 1] = f64_to_f32((double)p.ic_low[i + 1] + ((double)p.ic_high[i + 1] - (double)p.ic_low[i + 1]) * ub);
    }
}
R6_HD void normalize_ic_quaternion(float *ic)      // rocket_env.py:190 (float32, sdot rule)
{
    double acc = (double)f32_mul(ic[6], ic[6]);
    acc = acc + (double)f32_mul(ic[7], ic[7]);
    acc = acc + (double)f32_mul(ic[8], ic[8]);
    acc = acc + (double)f32_mul(ic[9], ic[9]);
    const float n = f32_sqrt(f64_to_f32(acc));
#pragma unroll
    for (int i = 6; i < 10; i++) ic[i] = f32_div(ic[i], n);
}
// synthetic random policy: uniform(-1,1) float32, one Philox block per (env, step)
R6_HD void philox_action(uint64_t seed, uint64_t genv, uint64_t step, float &a0, float &a1, float &a2)
{
    U4 ctr = {(uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)step, kStreamAction ^ (uint32_t)(step >> 32)};
    U4 r = philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double s = 1.0 / 4294967296.0;
    a0 = f64_to_f32(-1.0 + 2.0 * (((double)r.x + 0.5) * s));
    a1 = f64_to_f32(-1.0 + 2.0 * (((double)r.y + 0.5) * s));
    a2 = f64_to_f32(-1.0 + 2.0 * (((double)r.z + 0.5) * s));
    // the float32 cast may round to +-1 exactly; that is inside the action space
}

// ------------------------------------------------------------------------------------------------
// Deterministic SB3 MlpPolicy actor (PPO "MlpPolicy", net_arch [128, 64], tanh; the network of
// best_model_*.zip that montecarlo_script.py:54-64 evaluates):
//     a = clip(W2 tanh(W1 tanh(W0 x + b0) + b1) + b2, -1, 1),   x = obs[0:13] (RemoveMassFromObs)
// all in float32 like torch.  Packed weight block (floats), built once per CTA in shared memory
// (or by the host build in plain memory):
//     [0, 2048)        W0 rows padded to 16: row j = (w0[j][0..12], b0[j], 0, 0)
//     [2048, 10240)    W1 transposed: [in j][out k]  (64 contiguous floats per hidden-0 unit)
//     [10240, 10304)   b1      [10304, 10560)  W2 [4][64] (row 3 = value head)      [10560, 10564)  b2, bv
// One thread evaluates the whole network for its environment: hidden-0 units are produced one at a
// time and immediately scattered into the 64 hidden-1 accumulators, so nothing but those 64 floats
// is live; every weight read is a warp-uniform (broadcast) 16-byte load.
constexpr int kMlpIn = 13, kMlpH0 = 128, kMlpH1 = 64, kMlpOut = 3;
constexpr int kMlpOffW1 = kMlpH0 * 16, kMlpOffB1 = kMlpOffW1 + kMlpH0 * kMlpH1, kMlpOffW2 = kMlpOffB1 + kMlpH1;
constexpr int kMlpRows = 4;       // output rows of the last layer: 3 action means + the value head (0 when absent)
constexpr int kMlpOffB2 = kMlpOffW2 + kMlpRows * kMlpH1, kMlpFloats = kMlpOffB2 + 4;

struct F4 { float x, y, z, w; };
R6_HD F4 ld4(const float *p)
{
#if defined(__CUDA_ARCH__)
    const float4 v = *reinterpret_cast<const float4 *>(p);
    return F4{v.x, v.y, v.z, v.w};
#else
    return F4{p[0], p[1], p[2], p[3]};
#endif
}

// last layer as 4 rows: action_net rows 0..2, value_net as row 3 (zeros when the caller gave no critic)
R6_HD float mlp_w2_row(const R6Mlp &m, int row, int k)
{
    if (row < kMlpOut) return m.w2[row * kMlpH1 + k];
    return (row == kMlpOut && m.wv != nullptr) ? m.wv[k] : 0.0f;
}
R6_HD float mlp_b2_row(const R6Mlp &m, int row)
{
    if (row < kMlpOut) return m.b2[row];
    return (row == kMlpOut && m.bv != nullptr) ? m.bv[0] : 0.0f;
}

// element `idx` of the packed block from the SB3-layout tensors ([out][in] row-major)
R6_HD float mlp_pack_element(const R6Mlp &m, int idx)
{
    if (idx < kMlpOffW1) {
        const int j = idx >> 4, i = idx & 15;
        return i < kMlpIn ? m.w0[j * kMlpIn + i] : (i == kMlpIn ? m.b0[j] : 0.0f);
    }
    if (idx < kMlpOffB1) {
        const int r = idx - kMlpOffW1, j = r / kMlpH1, k = r % kMlpH1;
        return m.w1[k * kMlpH0 + j];
    }
    if (idx < kMlpOffW2) return m.b1[idx - kMlpOffB1];
    if (idx < kMlpOffB2) return mlp_w2_row(m, (idx - kMlpOffW2) / kMlpH1, (idx - kMlpOffW2) % kMlpH1);
    return mlp_b2_row(m, idx - kMlpOffB2);
}

// raw outputs: out[0..2] = Gaussian mean (unclipped), out[3] = value.  latent(k, h) is called with every unit h of
// the last hidden layer (the gSDE head reads it; the plain forward passes a no-op).
template <class Latent>
R6_HD void mlp_forward_latent(const float *W, const float *x, float (&out)[4], Latent &&latent)
{
    float acc[kMlpH1];
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) acc[k] = 0.0f;
#pragma unroll 2
    for (int j = 0; j < kMlpH0; j++) {
        const F4 wa = ld4(W + j * 16), wb = ld4(W + j * 16 + 4), wc = ld4(W + j * 16 + 8), wd = ld4(W + j * 16 + 12);
        float s = wa.x * x[0];
        s = f32_fma(wa.y, x[1], s); s = f32_fma(wa.z, x[2], s); s = f32_fma(wa.w, x[3], s);
        s = f32_fma(wb.x, x[4], s); s = f32_fma(wb.y, x[5], s); s = f32_fma(wb.z, x[6], s); s = f32_fma(wb.w, x[7], s);
        s = f32_fma(wc.x, x[8], s); s = f32_fma(wc.y, x[9], s); s = f32_fma(wc.z, x[10], s); s = f32_fma(wc.w, x[11], s);
        s = f32_fma(wd.x, x[12], s);
        const float h = tanhf(s + wd.y);
        const float *w1 = W + kMlpOffW1 + j * kMlpH1;
#pragma unroll
        for (int k = 0; k < kMlpH1; k += 4) {
            const F4 w = ld4(w1 + k);
            acc[k] = f32_fma(w.x, h, acc[k]); acc[k + 1] = f32_fma(w.y, h, acc[k + 1]);
            acc[k + 2] = f32_fma(w.z, h, acc[k + 2]); acc[k + 3] = f32_fma(w.w, h, acc[k + 3]);
        }
    }
    float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f, o3 = 0.0f;
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) {
        const float h = tanhf(acc[k] + W[kMlpOffB1 + k]);
        latent(k, h);
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
R6_HD void mlp_forward(const float *W, const float *x, float (&out)[4])
{
    mlp_forward_latent(W, x, out, [](int, float) {});
}
// deterministic action of evaluate_policy / predict: the mean clipped to the action space
R6_HD void mlp_policy(const float *W, const float *x, float &a0, float &a1, float &a2)
{
    float out[4];
    mlp_forward(W, x, out);
    a0 = fminf(fmaxf(out[0], -1.0f), 1.0f);
    a1 = fminf(fmaxf(out[1], -1.0f), 1.0f);
    a2 = fminf(fmaxf(out[2], -1.0f), 1.0f);
}

// ------------------------------------------------------------------------------------------------
// SB3 1.6's default MlpPolicy without policy_kwargs: separate tanh towers net_arch [dict(pi=[64, 64], vf=[64, 64])],
// action_net on the policy latent, value_net on the value latent (R6Mlp with vf_w0 set).  The packed block keeps the
// shared layout's offsets with the two towers stacked, plus the value tower's second bias:
//     [0, 2048)        W0 rows: j < 64 the policy tower's w0[j], j >= 64 the value tower's vf_w0[j - 64] (with b0 / vf_b0)
//     [2048, 10240)    W1 transposed [in j][out k]: j < 64 w1[k][j] (policy), j >= 64 vf_w1[k][j - 64] (value)
//     [10240, 10304)   b1 (policy)   [10304, 10560) W2 [4][64]: rows 0..2 action_net, row 3 value_net   [10560, 10564) b2, bv
//     [10564, 10628)   vf_b1
// The same multiply-adds as the shared trunk (13 x 128 + 2 x 64 x 64 = 13 x 128 + 128 x 64), 256 tanh instead of 192.
constexpr int kMlpOffVb1 = kMlpFloats, kMlpFloatsSep = kMlpOffVb1 + kMlpH1;
static_assert(2 * kMlpH1 == kMlpH0, "the two towers stack into the shared trunk's layer 0");

R6_HD bool mlp_separate(const R6Mlp &m) { return m.vf_w0 != nullptr; }

R6_HD float mlp_pack_element_sep(const R6Mlp &m, int idx)
{
    if (idx < kMlpOffW1) {
        const int j = idx >> 4, i = idx & 15;
        const float *w0 = j < kMlpH1 ? m.w0 + j * kMlpIn : m.vf_w0 + (j - kMlpH1) * kMlpIn;
        const float b0 = j < kMlpH1 ? m.b0[j] : m.vf_b0[j - kMlpH1];
        return i < kMlpIn ? w0[i] : (i == kMlpIn ? b0 : 0.0f);
    }
    if (idx < kMlpOffB1) {
        const int r = idx - kMlpOffW1, j = r / kMlpH1, k = r % kMlpH1;
        return j < kMlpH1 ? m.w1[k * kMlpH1 + j] : m.vf_w1[k * kMlpH1 + j - kMlpH1];
    }
    if (idx < kMlpOffVb1) return mlp_pack_element(m, idx);      // b1, W2 rows, b2 / bv: as the shared layout
    return m.vf_b1[idx - kMlpOffVb1];
}

// acc[k] = sum over the 64 layer-0 units j0 .. j0 + 63 of W1T[j][k] tanh(W0[j] x + b0[j]): one tower's layer 1 before
// its bias (mlp_forward_latent's loop over half of the stacked units).  unit0(j, h) sees every layer-0 activation.
template <int j0, class Unit0>
R6_HD void mlp_tower_acc(const float *W, const float *x, float (&acc)[kMlpH1], Unit0 &&unit0)
{
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) acc[k] = 0.0f;
#pragma unroll 2
    for (int j = j0; j < j0 + kMlpH1; j++) {
        const F4 wa = ld4(W + j * 16), wb = ld4(W + j * 16 + 4), wc = ld4(W + j * 16 + 8), wd = ld4(W + j * 16 + 12);
        float s = wa.x * x[0];
        s = f32_fma(wa.y, x[1], s); s = f32_fma(wa.z, x[2], s); s = f32_fma(wa.w, x[3], s);
        s = f32_fma(wb.x, x[4], s); s = f32_fma(wb.y, x[5], s); s = f32_fma(wb.z, x[6], s); s = f32_fma(wb.w, x[7], s);
        s = f32_fma(wc.x, x[8], s); s = f32_fma(wc.y, x[9], s); s = f32_fma(wc.z, x[10], s); s = f32_fma(wc.w, x[11], s);
        s = f32_fma(wd.x, x[12], s);
        const float h = tanhf(s + wd.y);
        unit0(j, h);
        const float *w1 = W + kMlpOffW1 + j * kMlpH1;
#pragma unroll
        for (int k = 0; k < kMlpH1; k += 4) {
            const F4 w = ld4(w1 + k);
            acc[k] = f32_fma(w.x, h, acc[k]); acc[k + 1] = f32_fma(w.y, h, acc[k + 1]);
            acc[k + 2] = f32_fma(w.z, h, acc[k + 2]); acc[k + 3] = f32_fma(w.w, h, acc[k + 3]);
        }
    }
}

// mlp_forward over the separate towers (packed by mlp_pack_element_sep): the value tower first, reduced to the value
// as its latent is formed, then the policy tower in the same 64 accumulators.  out as mlp_forward.
R6_HD void mlp_forward_sep(const float *W, const float *x, float (&out)[4])
{
    float acc[kMlpH1];
    mlp_tower_acc<kMlpH1>(W, x, acc, [](int, float) {});
    float o3 = 0.0f;
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) o3 = f32_fma(W[kMlpOffW2 + 3 * kMlpH1 + k], tanhf(acc[k] + W[kMlpOffVb1 + k]), o3);
    mlp_tower_acc<0>(W, x, acc, [](int, float) {});
    float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f;
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) {
        const float h = tanhf(acc[k] + W[kMlpOffB1 + k]);
        o0 = f32_fma(W[kMlpOffW2 + k], h, o0);
        o1 = f32_fma(W[kMlpOffW2 + kMlpH1 + k], h, o1);
        o2 = f32_fma(W[kMlpOffW2 + 2 * kMlpH1 + k], h, o2);
    }
    out[0] = o0 + W[kMlpOffB2];
    out[1] = o1 + W[kMlpOffB2 + 1];
    out[2] = o2 + W[kMlpOffB2 + 2];
    out[3] = o3 + W[kMlpOffB2 + 3];
}

// mlp_forward_sep with latent(k, h) called on every unit of the POLICY tower's latent (the gSDE head of the separate
// towers reads it): the same operations in the same order, so out is bit-identical to mlp_forward_sep's.  A copy rather
// than a callback added to mlp_forward_sep, so that the kernels built on that keep their register allocation.
template <class Latent>
R6_HD void mlp_forward_sep_latent(const float *W, const float *x, float (&out)[4], Latent &&latent)
{
    float acc[kMlpH1];
    mlp_tower_acc<kMlpH1>(W, x, acc, [](int, float) {});
    float o3 = 0.0f;
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) o3 = f32_fma(W[kMlpOffW2 + 3 * kMlpH1 + k], tanhf(acc[k] + W[kMlpOffVb1 + k]), o3);
    mlp_tower_acc<0>(W, x, acc, [](int, float) {});
    float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f;
#pragma unroll
    for (int k = 0; k < kMlpH1; k++) {
        const float h = tanhf(acc[k] + W[kMlpOffB1 + k]);
        latent(k, h);
        o0 = f32_fma(W[kMlpOffW2 + k], h, o0);
        o1 = f32_fma(W[kMlpOffW2 + kMlpH1 + k], h, o1);
        o2 = f32_fma(W[kMlpOffW2 + 2 * kMlpH1 + k], h, o2);
    }
    out[0] = o0 + W[kMlpOffB2];
    out[1] = o1 + W[kMlpOffB2 + 1];
    out[2] = o2 + W[kMlpOffB2 + 2];
    out[3] = o3 + W[kMlpOffB2 + 3];
}

// sin(pi x), cos(pi x): exact argument reduction, 1 ulp (CUDA math library); the host build in double precision
R6_HD void sincospi_f32(float x, float &s, float &c)
{
#if defined(__CUDA_ARCH__)
    sincospif(x, &s, &c);
#else
    s = (float)sin(3.141592653589793 * (double)x);
    c = (float)cos(3.141592653589793 * (double)x);
#endif
}
R6_HD float cospi_f32(float x)
{
#if defined(__CUDA_ARCH__)
    return cospif(x);
#else
    return (float)cos(3.141592653589793 * (double)x);
#endif
}

// Gaussian policy head (SB3 DiagGaussianDistribution with a state-independent log_std): sample and log-probability.
// eps from one Philox block keyed (seed, global env, step) through Box-Muller, with the accurate logf (1 ulp) and
// sincospif / cospif (1 ulp) on both builds: z is good to 3 ulp everywhere.  Not the MUFU forms __logf / __sincosf:
// their error is absolute, as large as ln u itself where u -> 1 (the radius off by a fifth), and above their
// documented accuracy elsewhere (tests/test_gpu_policy_ref.py measures the noise against a float64 statement).
constexpr uint32_t kStreamPolicy = 0x50414354u;   // 'PACT'
R6_HD void gaussian_head(const float (&mean)[4], const float *log_std, bool stochastic, uint64_t seed, uint64_t genv,
                         uint64_t step, float (&raw)[3], float &logp)
{
    float z[3] = {0.0f, 0.0f, 0.0f};
    if (stochastic) {
        U4 ctr = {(uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)step, kStreamPolicy ^ (uint32_t)(step >> 32)};
        const U4 r = philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
        const float s = 1.0f / 4294967296.0f;
        const float u1 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)r.y * s;
        const float u3 = ((float)(r.z >> 8) + 0.5f) * (1.0f / 16777216.0f), u4 = (float)r.w * s;
        // u1, u3 in (0, 1] (1.0 for the top grid value: k + 0.5 rounds to even): logf <= 0, so the roots are real.
        // The angles 2 pi u2, 2 pi u4 are formed exactly as pi * (2 u).
        const float ra = sqrtf(-2.0f * logf(u1)), rb = sqrtf(-2.0f * logf(u3));
        float sn, cs;
        sincospi_f32(2.0f * u2, sn, cs);
        z[0] = ra * cs;
        z[1] = ra * sn;
        z[2] = rb * cospi_f32(2.0f * u4);
    }
    logp = 0.0f;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const float ls = log_std != nullptr ? log_std[i] : 0.0f;
        raw[i] = mean[i] + expf(ls) * z[i];
        logp += -0.5f * z[i] * z[i] - ls - 0.9189385332046727f;      // 0.5 log(2 pi)
    }
}

// ------------------------------------------------------------------------------------------------
// Generalised state-dependent exploration (SB3 1.6 StateDependentNoiseDistribution, full_std, no expln, latent_sde =
// the 64-unit trunk output h, detached) [memory]:
//     E_i = sigma (.) xi_i,  sigma = exp(log_std) [64][3],  xi_i ~ N(0, 1) drawn per env by reset_noise
//     raw = mean + h E_i,    std_a = sqrt(sum_k h_k^2 sigma_ka^2 + 1e-6),   log_prob / entropy of N(mean, std)
// xi is a component-major [192][n] buffer, component c = 3 k + a (SB3's [64][3] order).  Component block b (c = 4b ..
// 4b + 3) of an env is one Philox block keyed (seed, global env id, draw step), so the buffer does not depend on the
// shard, lane or sub-range that drew it; Box-Muller with the accurate logf / sincospif of gaussian_head (see there).
constexpr int kSdeLatent = 64, kSdeXi = kSdeLatent * kMlpOut, kSdeBlocks = kSdeXi / 4;
constexpr uint32_t kStreamSde = 0x47534445u;      // 'GSDE' ^ (step hi << 8) ^ block
R6_HD void sde_noise_block(uint64_t seed, uint64_t genv, uint64_t step, int b, float (&z)[4])
{
    U4 ctr = {(uint32_t)genv, (uint32_t)(genv >> 32), (uint32_t)step, kStreamSde ^ ((uint32_t)(step >> 32) << 8) ^ (uint32_t)b};
    const U4 r = philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
    const float s = 1.0f / 4294967296.0f;
    const float u1 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)r.y * s;
    const float u3 = ((float)(r.z >> 8) + 0.5f) * (1.0f / 16777216.0f), u4 = (float)r.w * s;
    const float ra = sqrtf(-2.0f * logf(u1)), rb = sqrtf(-2.0f * logf(u3));
    float sn, cs;
    sincospi_f32(2.0f * u2, sn, cs);
    z[0] = ra * cs;
    z[1] = ra * sn;
    sincospi_f32(2.0f * u4, sn, cs);
    z[2] = rb * cs;
    z[3] = rb * sn;
}

// The gSDE policy head of one env from the partial sums of the latent: nz[a] = sum_k h_k E_ka (the noise),
// var[a] = sum_k h_k^2 sigma_ka^2.  stochastic: raw = mean + nz, else the mean; logp of raw under N(mean, std).
R6_HD void sde_head(const float (&mean)[4], const float (&nz)[3], const float (&var)[3], bool stochastic, float (&raw)[3],
                    float &logp)
{
    logp = 0.0f;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const float v = var[a] + 1e-6f;                   // std^2 (SB3: sqrt(variance + epsilon), squared back by Normal)
        raw[a] = stochastic ? mean[a] + nz[a] : mean[a];
        const float d = raw[a] - mean[a];
        logp += -(d * d) / (2.0f * v) - logf(sqrtf(v)) - 0.9189385332046727f;
    }
}

// ------------------------------------------------------------------------------------------------
// Registers carried by the thread that owns an environment, and the glue of one env step
template <class R>
struct EnvT {
    R y[14];
    float m0, v0;
    int k;             // steps taken in the episode
    uint32_t episode;  // episodes started so far (RNG counter)
    double ep_return;
    float tgo;         // t_go root of the previous step (0 = none): warm start of tgo_largest_root
};
using Env = EnvT<double>;

// Rocket6DOF.reset: new initial condition (Philox or replay table), Simulator6DOF re-created.
template <class R>
R6_HD void env_reset(const R6Params &p, const R6Buffers &b, uint64_t seed, int64_t genv, EnvT<R> &e)
{
    float ic[14];
    if (b.ic_table != nullptr && b.ic_table_len > 0) {
        const int64_t row = (genv + b.n_global * (int64_t)e.episode) % b.ic_table_len;
#pragma unroll
        for (int c = 0; c < 14; c++) ic[c] = b.ic_table[row * 14 + c];   // rows are already normalised
    } else {
        sample_initial_condition(p, seed, (uint64_t)genv, e.episode, ic);
        normalize_ic_quaternion(ic);
    }
#pragma unroll
    for (int c = 0; c < 14; c++) e.y[c] = (R)ic[c];
    e.m0 = ic[13];
    e.v0 = f32_sqrt(sdot3(ic[3], ic[4], ic[5], ic[3], ic[4], ic[5]));
    e.k = 0;
    e.episode += 1;
    e.ep_return = 0.0;
    e.tgo = 0.0f;
}

struct StepOut {
    double reward;     // what the (wrapped) env returns
    uint32_t flags;
    bool finished;     // done or truncated
    int natt;
    int status;
    PostOut post;
};

// VerticalAttitudeReward (wrappers.py:143-150): clip(2 deg(acos(q0)) weight, -10, 10).  Touchdown only => out of line.
R6_HD_NOINLINE double vertical_attitude_term(double q0, double weight)
{
    const double deg = acos(q0) * (180.0 / 3.14159265358979323846);
    return fmin(fmax(2 * deg * weight, -10.0), 10.0);
}

// One Rocket6DOF.step on the registers of `e` (no reset here), in two halves so that the step can also run as two
// kernels (integrate | reward, flags, reset, observation).  R = double: the parity path, integrated on the absolute
// simulator clock t_table[k] like the reference.  R = float: the dynamics are autonomous, so the step is
// integrated on the local clock [0, dt] (a float32 absolute time would waste its mantissa on the 150 s range);
// reward / flags are then evaluated by the same float64 code on the widened state.
//
// First half: Simulator6DOF.step (simulator.py:69-104) — action de-normalisation, solve_ivp, quaternion renorm.
template <bool kExact, class KS, class R>
R6_HD void env_integrate(const R6Params &p, const double *__restrict__ t_table, R *y, float m0, int k, float a0, float a1,
                         float a2, KS &K, int &status, int &natt)
{
    float u0, u1, u2;
    denormalize_action(p, a0, a1, a2, u0, u1, u2);
    StepConstT<R> c;
    consts_env_mode(c, m0, u0, u1, u2, y[10]);
    R t = 0;
    if constexpr (sizeof(R) == 8) {
        const int kk = k < p.n_t ? k : p.n_t - 1;
        t = (R)t_table[kk];
    }
    status = integrate<kExact>(c, y, t, (R)p.dt, natt, K);
    normalize_quat(y);
}

// env_integrate cut at attempt boundaries (see integrate<..., kPass>): returns -2 while the env is unfinished.
template <bool kExact, int kPass, class KS, class R>
R6_HD int env_integrate_pass(const R6Params &p, const double *__restrict__ t_table, R *y, float m0, int k, float a0,
                             float a1, float a2, KS &K, PassCtx<R> &px, int &natt)
{
    float u0, u1, u2;
    denormalize_action(p, a0, a1, a2, u0, u1, u2);
    StepConstT<R> c;
    consts_env_mode(c, m0, u0, u1, u2, y[10]);
    R t = 0;
    if constexpr (sizeof(R) == 8 && kPass != 2) {          // a resumed pass carries its own clock (px.t, px.t_bound)
        const int kk = k < p.n_t ? k : p.n_t - 1;
        t = (R)t_table[kk];
    }
    const int status = integrate<kExact, KS, R, kPass>(c, y, t, (R)p.dt, natt, K, px);
    if (status != -2) normalize_quat(y);
    return status;
}

// Second half: rocket_env.py:206-231 on the post-step state + the make_env() / reward wrappers.  e.k is the step
// index BEFORE this step (incremented here).
template <class R>
R6_HD void env_post(const R6Params &p, const Derived &dv, EnvT<R> &e, float a0, float a1, float a2, int status, int natt,
                    StepOut &o)
{
    float u0, u1, u2;
    denormalize_action(p, a0, a1, a2, u0, u1, u2);
    StepConstT<R> c;
    consts_env_mode(c, e.m0, u0, u1, u2, e.y[10]);      // only the body-frame thrust is used below (w0 is conserved)
    o.status = status;
    o.natt = natt;
    e.k += 1;
    post_step(p, dv.at, c, e.y, u2, e.v0, o.status, o.post, e.tgo);      // working precision = R
    e.tgo = o.post.tgo;
    uint32_t fl = o.post.flags;
    const bool done = (fl & (R6_F_EVENT | R6_F_OOB)) != 0;                    // rocket_env.py:213
    const bool trunc = !done && p.max_episode_steps > 0 && e.k >= p.max_episode_steps;   // gym TimeLimit
    if (trunc) fl |= R6_F_TRUNCATED;
    double r = o.post.reward;
    if (p.reward_mode & R6_RW_ANNEALED) {
        // RewardAnnealing.step (wrappers.py:44-61): the env reward is discarded and rebuilt from four
        // terms of rewards_dict plus -xi*(action[2]+1) (float32: python float times np.float32)
        const float tp = f32_mul(-p.xi, f32_add(a2, 1.0f));
        double s = 0;
        s += o.post.terms[3]; s += o.post.terms[4]; s += o.post.terms[5]; s += o.post.terms[6]; s += (double)tp;
        r = s;
        o.post.terms[0] = 0; o.post.terms[1] = (double)tp; o.post.terms[2] = 0;
    }
    if (p.reward_mode & R6_RW_VERTICAL) {
        // VerticalAttitudeReward.step (wrappers.py:134-155) on the float64 post-step state
        if ((double)e.y[0] < p.va_threshold && o.post.terms[6] > 0) r += vertical_attitude_term((double)e.y[6], p.va_weight);
    }
    if (p.clip_reward) r = fmin(fmax(r, p.clip_lo), p.clip_hi);               // main_6DOF.py:40-42
    o.reward = r;
    o.flags = fl;
    o.finished = done || trunc;
    e.ep_return += r;
}

template <bool kExact, class KS, class R>
R6_HD void env_step(const R6Params &p, const Derived &dv, const double *__restrict__ t_table, EnvT<R> &e, float a0,
                    float a1, float a2, StepOut &o, KS &K)
{
    int status, natt;
    env_integrate<kExact>(p, t_table, e.y, e.m0, e.k, a0, a1, a2, K, status, natt);
    env_post(p, dv, e, a0, a1, a2, status, natt, o);
}

}  // namespace r6
