// r6_mlp_tcgen05.cuh — the policy MLP (13 -> 128 -> 64 -> 3 (+ value), tanh) on the 5th-generation tensor cores:
// tcgen05.mma (kind::tf32, M = 128 envs per tile), accumulators AND activations in tensor memory, weights in shared
// memory, tcgen05.ld / tcgen05.st for the epilogues, mbarrier completion.  It is its own uniform kernel because a
// tcgen05 MMA is a CTA-wide operation (128 rows per tile, a barrier per layer), which the divergent integrator cannot
// afford but a dedicated policy kernel can.  Two modes of r6_policy share the code (template <bool kFaithful>):
//
//   tensor_cores = 3, FAITHFUL: 3xTF32 error compensation — every operand split x = hi + lo, hi = round_tf32(x),
//     lo = round_tf32(x - hi), and hi*hi + lo*hi + hi*lo chained into ONE TMEM accumulator (three MMAs per K-block, the
//     dropped lo*lo term is 2^-22 relative) — with a float32-accurate tanh: actions agree with the float32 FMA network
//     to ~3e-6 (tests/test_gpu_policy.py).
//   tensor_cores = 2, FAST: single-pass TF32 and tanh.approx: |d action| ~2e-3, for rollouts where the policy's own
//     exploration noise dwarfs that.
//
// Layout.  One CTA per SM carries TWO independent 128-env tile groups (warps 0-7 and 8-15; two threads per env row,
// each taking half of the columns of an epilogue) over one resident copy of the weights.  An epilogue thread owns TMEM
// lane = env row: it reads its 32 accumulator columns (tcgen05.ld), applies bias + tanh, splits, and stores hi IN PLACE
// over the columns it just read and lo into a 64-column side tile (tcgen05.st) — which is exactly the K-major A layout
// the next layer's MMA wants when A comes from tensor memory (row = lane, k = column).  No activation ever touches
// shared memory, so no generic->async proxy fence is needed per layer, and the per-MMA shared-memory read is B only
// (2 KB at N = 64: under the 32-cycle tensor-pipe slot; with A in shared memory the same MMA needed 48 cycles of
// shared-memory bandwidth and the 3xTF32 chain read every activation tile twice).
//   TMEM, per group (256 of the SM's 512 columns):  D0 [0,128)   D1 [128,192)   L [192,256)
//     layer 0 : A = X   hi D1[0:16)  lo L[0:16)            -> D0[0:128)      (2 K-blocks)
//     layer 1a: A = H0a hi D0[0:64)  (in place) lo L[0:64) -> D1             (8 K-blocks)
//     layer 1b: A = H0b hi D0[64:128)           lo L[0:64) -> D1 +=          (8 K-blocks)
//     layer 2 : A = H1  hi D1[0:64)  (in place) lo L[0:64) -> D0[0:16)       (8 K-blocks; D0 is dead by then)
//   shared memory: W0h W0l (8+8 KB) | W1h W1l (32+32) | W2h W2l (4+4) | biases | two mbarriers | TMEM base   = 89 KB
//
// Schedule.  (1) The two groups take turns in the bias + tanh + split arithmetic through an epilogue token (named
// barriers 3 and 4): left alone they fall into lock-step — both on the XU pipe, then both waiting on the tensor pipe.
// With the token one group's MMAs run under the other group's epilogue.  (2) The MMAs of a layer are issued by the
// first warp of the group, CONVERGED, from warp-uniform operands, one elected lane per instruction: issued by a single
// thread under a divergent branch every MMA was wrapped in an ELECT / 4 x R2UR / branch sequence of ~75 cycles, which
// made the issue rate — not the tensor pipe — the pace of a layer.  (3) The next tile's observations are loaded under
// the current tile's three layers and the previous tile's outputs are written out under the next layer-0 MMA.
// Measured (profiles/r02_policy_tcgen05_tmem.md): 2^20 envs in 0.175 ms faithful (XU pipe 57 % busy, tensor pipe
// 38 %); the shared-memory-operand version it replaces took 0.30 ms.
//
// Separate towers (SB3 1.6's net_arch [dict(pi=[64, 64], vf=[64, 64])], policy_tc5_sep_kernel).  Layer 0 is the shared
// kernel's once the two towers' w0 are stacked ([pi; vf], 128 rows), and W1's [64][128] tile holds [w1 | vf_w1] side by
// side, so the two layer-1 chains are the shared kernel's 1a / 1b with their own accumulators.  TMEM is what binds:
// D0, D1 and L take a group's 256 columns and a third 64-column accumulator does not fit with both groups resident.
// So the value chain runs first and is reduced on the CUDA cores:
//     layer 1v: A = H0v hi D0[64:128) lo L[0:64) -> D1     then  value = wv . tanh(D1 + vf_b1) in the epilogue, from the
//               float32 accumulator (32 FMAs per column half; the second half's sum handed over through shared memory)
//     layer 1p: A = H0p hi D0[0:64)  lo L[0:64) -> D1     (overwrites the value chain's accumulator, read by then)
//     layer 2 : as above, W2 row 3 zero (the value is not an MMA output)
// Per tile that is one more epilogue (four: H0v, value, H0p, H1p) and the same four MMA commits; the value never
// needs a TF32 split.  Extra shared memory: vf_b1, wv and per group the second half's value sums (kOffSep..).
// With gSDE (policy_tc5_sep_sde_kernel) the H1p epilogue is epilogue_in_tmem_sde, which forms h E and h^2 sigma^2 over the
// policy latent; sigma, sigma^2 and the second half's sums follow the separate-tower region (kOffSepSde.., ~100 KB in all).
//
// Shared-memory operand layout of the weights (K-major, SWIZZLE_NONE "interleaved" canonical layout): element (row r,
// k) of a tile with K_tot columns lives at byte (r % 8) * 16 + (r / 8) * SBO + (k / 4) * 128 + (k % 4) * 4,
// SBO = (K_tot / 4) * 128: 8-row x 16-byte core matrices, consecutive K chunks 128 B apart (LBO), 8-row groups SBO
// apart.  One MMA consumes K = 8 (two chunks), so K-block kb starts 256 B further.
#pragma once

#include <stdint.h>

#include "r6_core.cuh"

namespace r6 {
namespace tc5 {

constexpr int kTile = 128;                       // envs per tile = MMA M
constexpr int kThreads = 512;                    // two tile groups x (128 rows x 2 column halves)
constexpr uint32_t kTmemCols = 512, kGroupCols = 256;
constexpr uint32_t kColD0 = 0, kColD1 = 128, kColL = 192;
// byte offsets inside the dynamic shared memory block
constexpr int kOffW0h = 0, kOffW0l = 8 << 10, kOffW1h = 16 << 10, kOffW1l = 48 << 10, kOffW2h = 80 << 10, kOffW2l = 84 << 10;
constexpr int kOffBias = 88 << 10;                                   // b0[128] b1[64] b2[4]
constexpr int kOffBar = kOffBias + (128 + 64 + 4) * 4;               // one mbarrier per group
constexpr int kOffTmemPtr = kOffBar + 16;
constexpr int kSmemBytes = kOffTmemPtr + 16;
// gSDE kernels only: sigma [192], sigma^2 [192], and per group the second column half's partial sums [128 rows][6]
constexpr int kOffSde = kSmemBytes, kOffSdePart = kOffSde + 2 * 192 * 4;
constexpr int kSmemBytesSde = kOffSdePart + 2 * kTile * 6 * 4;
// separate-tower kernels only: vf_b1 [64] (pre-scaled like b1), wv [64], per group the second half's value sums [128]
constexpr int kOffSep = kSmemBytes, kOffSepWv = kOffSep + 64 * 4, kOffSepPart = kOffSepWv + 64 * 4;
constexpr int kSmemBytesSep = kOffSepPart + 2 * kTile * 4;
// separate towers with gSDE (policy_tc5_sep_sde_kernel): the separate-tower region, then the gSDE region after it
constexpr int kOffSepSde = kSmemBytesSep, kOffSepSdePart = kOffSepSde + 2 * 192 * 4;
constexpr int kSmemBytesSepSde = kOffSepSdePart + 2 * kTile * 6 * 4;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ int tile_off(int r, int k, int ktot) { return (r & 7) * 16 + (r >> 3) * (ktot * 32) + (k >> 2) * 128 + (k & 3) * 4; }
__device__ __forceinline__ float round_tf32(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
__device__ __forceinline__ void split_tf32(float x, float &hi, float &lo)
{
    hi = round_tf32(x);
    lo = round_tf32(x - hi);
}

// 64-bit shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address, LBO, SBO in 16-byte units,
// version 1 (Blackwell), SWIZZLE_NONE
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           (1ull << 46);
}
// 32-bit instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, M = 128
__device__ __forceinline__ constexpr uint32_t instr_desc(int n) { return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24); }

// D[tmem] (+)= A[tmem] B[smem]^T, A read from tensor memory (8 columns = one K-block of TF32)
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_commit(uint32_t bar) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void bar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra WAIT_%=;\n\t"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void group_sync(int group) { asm volatile("bar.sync %0, 256;" ::"r"(group + 1) : "memory"); }
// one lane of a converged warp
__device__ __forceinline__ bool elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t"
        "}\n" : "=r"(pred));
    return pred != 0;
}

// 32 consecutive columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4])
{
    uint32_t r[4];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 4; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
          "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
          "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
          "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
          "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr),
                 "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
                 "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// FAST mode: tanh on the MUFU unit (tanh.approx.f32, relative error 2^-11: the precision class of the TF32 operand it
// is rounded to right afterwards), one XU instruction instead of two plus FP32 ones
__device__ __forceinline__ float tanh_fast(float x)
{
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// FAITHFUL mode: tanh(x) = 1 - 2 / (exp(2x) + 1) on the exp2 / rcp units: absolute error ~1.5e-7 (the float32 ulp at 1
// is 6e-8), saturates correctly (exp -> inf => 1, exp -> 0 => -1)
constexpr float kTwoLog2e = 2.885390081777927f;
// z = 2 log2(e) x is formed by the caller as fma(acc, kTwoLog2e, kTwoLog2e * bias): one FFMA instead of FADD + FMUL
__device__ __forceinline__ float tanh_exact_scaled(float z)
{
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z));                           // exp(2x) = 2^(2x log2 e)
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}

// Epilogue token of the two tile groups (named barriers 3 and 4, 512 participants: the 256 threads of the group that
// takes the token bar.sync, the 256 of the group that hands it over bar.arrive): strict alternation.
__device__ __forceinline__ void token_take(int group) { asm volatile("bar.sync %0, 512;" ::"r"(group + 3) : "memory"); }
__device__ __forceinline__ void token_pass(int to_group) { asm volatile("bar.arrive %0, 512;" ::"r"(to_group + 3) : "memory"); }

// tanh(D[:, src + 32 half .. + 31] + bias) of this thread's row: hi over the columns just read, lo -> L[32 half ..].
// The token brackets the arithmetic only (the XU / FP32 phase); the TMEM load before it and the TMEM stores after it
// overlap with the other group's turn.
template <bool kFaithful>
__device__ __forceinline__ void epilogue_in_tmem(uint32_t tmem_row, uint32_t src, const float *bias, int half, int group)
{
    const int cc = 32 * half;
    float v[32];
    tmem_ld32(tmem_row + src + cc, v);
    token_take(group);
    if constexpr (kFaithful) {
        float l[32];
#pragma unroll
        for (int q = 0; q < 32; q++) split_tf32(tanh_exact_scaled(fmaf(v[q], kTwoLog2e, bias[cc + q])), v[q], l[q]);   // bias pre-scaled
        token_pass(group ^ 1);
        tmem_st32(tmem_row + src + cc, v);
        tmem_st32(tmem_row + kColL + cc, l);
    } else {
#pragma unroll
        for (int q = 0; q < 32; q++) v[q] = round_tf32(tanh_fast(v[q] + bias[cc + q]));
        token_pass(group ^ 1);
        tmem_st32(tmem_row + src + cc, v);
    }
    tmem_st_wait();
}

// The value tower's last hidden layer (separate towers): sum over this thread's 32 units k = cc .. cc + 31 of
// wv_k tanh(D[:, src + k] + vf_b1_k), from the float32 accumulator.  Nothing is stored back: the value latent feeds no MMA.
template <bool kFaithful>
__device__ __forceinline__ float epilogue_value(uint32_t tmem_row, uint32_t src, const float *bias, const float *wv, int half,
                                                int group)
{
    const int cc = 32 * half;
    float v[32];
    tmem_ld32(tmem_row + src + cc, v);
    token_take(group);
    float s = 0.0f;
#pragma unroll
    for (int q = 0; q < 32; q++) {
        const float h = kFaithful ? tanh_exact_scaled(fmaf(v[q], kTwoLog2e, bias[cc + q])) : tanh_fast(v[q] + bias[cc + q]);
        s = fmaf(wv[cc + q], h, s);
    }
    token_pass(group ^ 1);
    return s;
}

// epilogue_in_tmem of the last hidden layer with the gSDE sums over this thread's 32 units k = cc .. cc + 31 of its env row
// i: nz_a = sum_k h_k (sigma_ka xi_ka) (when draw) and var_a = sum_k h_k^2 sigma_ka^2, h the activation the next MMA
// consumes (hi + lo in faithful mode, hi in fast mode).  Formed after the token is handed over (under the other group's
// arithmetic), from xi read coalesced over the rows and sigma, sigma^2 in shared memory.
template <bool kFaithful>
__device__ __forceinline__ void epilogue_in_tmem_sde(uint32_t tmem_row, uint32_t src, const float *bias, int half, int group,
                                                     const float *sig, const float *sig2, const float *__restrict__ xi,
                                                     int64_t n, int64_t i, bool draw, float (&nz)[3], float (&var)[3])
{
    const int cc = 32 * half;
    float v[32], l[32];
    tmem_ld32(tmem_row + src + cc, v);
    token_take(group);
    if constexpr (kFaithful) {
#pragma unroll
        for (int q = 0; q < 32; q++) split_tf32(tanh_exact_scaled(fmaf(v[q], kTwoLog2e, bias[cc + q])), v[q], l[q]);
        token_pass(group ^ 1);
        tmem_st32(tmem_row + src + cc, v);
        tmem_st32(tmem_row + kColL + cc, l);
    } else {
#pragma unroll
        for (int q = 0; q < 32; q++) v[q] = round_tf32(tanh_fast(v[q] + bias[cc + q]));
        token_pass(group ^ 1);
        tmem_st32(tmem_row + src + cc, v);
    }
#pragma unroll
    for (int a = 0; a < 3; a++) nz[a] = var[a] = 0.0f;
    // xi walked by one pointer bumped n floats per component: precomputed per-component 64-bit offsets (loop invariants
    // across tiles) would not fit the 128 registers of a 512-thread CTA
    const float *px = xi + (int64_t)(3 * cc) * n + i;
    const int64_t stride = n;
#pragma unroll
    for (int q = 0; q < 32; q++) {
        const float h = kFaithful ? v[q] + l[q] : v[q], hh = h * h;
#pragma unroll
        for (int a = 0; a < 3; a++) {
            const int c = 3 * (cc + q) + a;
            if (draw) nz[a] = fmaf(h, sig[c] * __ldg(px), nz[a]);
            var[a] = fmaf(hh, sig2[c], var[a]);
            px += stride;
            asm volatile("" : "+l"(px));
        }
    }
    tmem_st_wait();
}

// nk K-blocks of D (+)= (Ah + Al)(Bh + Bl)^T without lo*lo (faithful) or Ah Bh^T (fast); A tiles are TMEM columns (8
// per K-block), B tiles shared memory (256 B per K-block).  Called by a whole CONVERGED warp with warp-uniform
// arguments: the descriptors are computed on the uniform datapath and each group of MMAs is issued by one elected lane.
template <bool kFaithful>
__device__ __forceinline__ void issue_mmas(uint32_t d_tmem, uint32_t ah, uint32_t al, uint32_t bh, uint32_t bl, uint32_t b_sbo,
                                           int nk, int n, bool accumulate_first)
{
    const uint32_t idesc = instr_desc(n);
#pragma unroll
    for (int kb = 0; kb < nk; kb++) {
        const uint64_t dbh = smem_desc(bh + kb * 256, 128, b_sbo), dbl = smem_desc(bl + kb * 256, 128, b_sbo);
        if (elect_one()) {
            mma_tf32_ts(d_tmem, ah + 8 * kb, dbh, idesc, accumulate_first || kb > 0);
            if constexpr (kFaithful) {
                mma_tf32_ts(d_tmem, al + 8 * kb, dbh, idesc, true);
                mma_tf32_ts(d_tmem, ah + 8 * kb, dbl, idesc, true);
            }
        }
    }
}

}  // namespace tc5
}  // namespace r6
