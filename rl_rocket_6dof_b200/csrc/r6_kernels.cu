// r6_kernels.cu — sm_100a kernels + the C ABI of include/r6dof.h.
//
// One thread owns one environment: its 14 state components are loaded from the component-major (SoA) state array
// with fully coalesced accesses (a warp reads 256 contiguous bytes per float64 component), stay in registers
// through the whole adaptive RK45 step, and are written back the same way.  The dynamics are not a contraction:
// their bound is the FP64 pipe, and no tensor core touches them.  Kernels:
//   integrate_kernel | post_kernel   r6_step as a pair: the divergent integrator (one-warp CTAs, stage storage in
//                                    shared memory) and the uniform reward / flags / reset / observation kernel
//   step_kernel                      the same step fused (small batches, zero-copy host path)
//   rollout_kernel, rollout_tc_kernel  k steps per launch with the state in registers (Philox / buffer / policy)
//   policy_kernel, policy_tc5_kernel   the policy MLP alone: float32 FMAs, mma.sync 3xTF32 tiles, or tcgen05.mma with
//                                    accumulators and activations in TMEM (r6_mlp_tc.cuh, r6_mlp_tcgen05.cuh)
//   ppo_grad_kernel | ppo_reduce_kernel, adam_kernel   the PPO update: minibatch loss gradient, Adam step
//   (policy_sep_kernel, policy_tc5_sep_kernel, ppo_grad_sep_kernel: the same for SB3 1.6's separate policy / value towers)
//   trunc_record_kernel, trunc_bootstrap_kernel   time-limit truncations filed per step, bootstrapped with the critic
//   reset_kernel, sim_raw_kernel, tgo_kernel, gae_kernel, peak_fma_kernel
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo (see build.py).
#include <cuda_runtime.h>

#ifndef R6_PDL
#define R6_PDL 1
#endif

#include <stdio.h>
#include <string.h>

#include <type_traits>

#include "r6_core.cuh"
#include "r6_mlp_tc.cuh"
#include "r6_mlp_tcgen05.cuh"
#include "r6_ppo.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, const char *detail = "")
{
    snprintf(g_err, sizeof g_err, fmt, detail);
    return code;
}
int check_launch(const char *what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString(e));
        return R6_ECUDA;
    }
    return R6_OK;
}

#ifndef R6_THREADS
#define R6_THREADS 128           /* threads (= environments) per CTA */
#endif
constexpr int kThreads = R6_THREADS;
#ifndef R6_MIN_BLOCKS
#define R6_MIN_BLOCKS 3          /* resident CTAs per SM the register allocation is tuned for (float64 path) */
#endif
#ifndef R6_MIN_BLOCKS_F32
#define R6_MIN_BLOCKS_F32 4      /* float32 path: half the registers and half the stage storage */
#endif
template <class R> constexpr int min_blocks() { return sizeof(R) == 4 ? R6_MIN_BLOCKS_F32 : R6_MIN_BLOCKS; }
// The stand-alone integrator uses one-warp CTAs: a CTA's registers and stage storage are held until its slowest
// warp has finished its adaptive steps, so with independent warps nothing waits (measured -2.3 % vs 128 threads).
#ifndef R6_INT_THREADS
#define R6_INT_THREADS 32
#endif
constexpr int kIntThreads = R6_INT_THREADS;
#ifndef R6_INT_CTAS_F64
#define R6_INT_CTAS_F64 (R6_MIN_BLOCKS * R6_THREADS / R6_INT_THREADS)      /* resident integrator CTAs per SM, float64 */
#endif
#ifndef R6_INT_CTAS_F32
#define R6_INT_CTAS_F32 (R6_MIN_BLOCKS_F32 * R6_THREADS / R6_INT_THREADS)
#endif
template <class R> constexpr int int_ctas() { return sizeof(R) == 4 ? R6_INT_CTAS_F32 : R6_INT_CTAS_F64; }
#ifndef R6_FIRST_CTAS_F64
#define R6_FIRST_CTAS_F64 R6_INT_CTAS_F64       /* resident CTAs per SM of the first pass of the multi-pass integrator */
#endif
template <class R> constexpr int first_ctas() { return sizeof(R) == 4 ? R6_INT_CTAS_F32 : R6_FIRST_CTAS_F64; }
// stage storage per CTA: 55,296 B (float64) / 27,648 B (float32); + packed policy weights (42,000 B) for R6_ACT_MLP
template <class R> constexpr int smem_bytes() { return 6 * r6::kNK * kThreads * (int)sizeof(R); }
template <class R> constexpr int smem_int_bytes() { return smem_bytes<R>() * kIntThreads / kThreads; }   // one-warp CTAs
template <class R> constexpr int smem_mlp_bytes() { return smem_bytes<R>() + r6::kMlpFloats * (int)sizeof(float); }
// tensor-core policy: fragment-ordered weights (43,792 B) + one [16][33] float staging tile per warp
template <class R> constexpr int smem_tc_bytes()
{
    return smem_bytes<R>() + r6::kMlpTcFloats * (int)sizeof(float) + (kThreads / 32) * 16 * 33 * (int)sizeof(float);
}
constexpr int kSmemBytes = smem_bytes<double>();

using namespace r6;

// the RK stage storage of this thread in a CTA of kWidth threads (dynamic shared memory)
template <class R, int kWidth = kThreads>
__device__ __forceinline__ KShared<R, kWidth> make_kstore()
{
    extern __shared__ __align__(16) double r6_smem[];
    KShared<R, kWidth> K;
    K.base = reinterpret_cast<R *>(r6_smem) + 2 * threadIdx.x;
    return K;
}

// ---------------------------------------------------------------------------------------------
// Episode statistics.  Env-steps are counted per lane and summed over the warp with one REDUX
// (__reduce_add_sync), lane 0 issuing a single atomic per warp; the per-episode slots are added by the
// lane whose episode just ended (about one lane per warp every four steps), straight to L2 — no
// shuffle tree, no block barrier (warps of a CTA finish their adaptive steps at different times) and
// no accumulator registers carried through the step.
// see launch_pdl: returns once the previous grid on the stream has completed and its writes are visible
// (An explicit early griddepcontrol.launch_dependents was measured too: the dependents' CTAs then sit resident at the wait
// and take register-file slots from the other lane's running kernel — joined step +1 %.  The implicit trigger at CTA exit
// keeps only what is free: the next kernel's launch latency under the previous kernel's drain.)
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void stats_steps(double *stats, int my_steps)
{

    const int tot = __reduce_add_sync(0xffffffffu, my_steps);
    if ((threadIdx.x & 31) == 0 && tot != 0) atomicAdd(&stats[R6_S_STEPS], (double)tot);
}
template <class R>
__device__ __noinline__ void stats_episode(double *stats, uint32_t flags, double ep_return, int length)
{
    atomicAdd(&stats[R6_S_EPISODES], 1.0);
    if (isfinite(ep_return)) atomicAdd(&stats[R6_S_RETURN_SUM], ep_return);     // never poison the batch statistics
    atomicAdd(&stats[R6_S_LENGTH_SUM], (double)length);
    if ((flags & R6_F_LANDING_ALL) == R6_F_LANDING_ALL) atomicAdd(&stats[R6_S_LANDED], 1.0);
    if (flags & R6_F_EVENT) atomicAdd(&stats[R6_S_GROUND], 1.0);
    if (flags & R6_F_OOB) atomicAdd(&stats[R6_S_OOB], 1.0);
    if (flags & R6_F_TRUNCATED) atomicAdd(&stats[R6_S_TRUNCATED], 1.0);
}

// ---------------------------------------------------------------------------------------------
// state / terminal_state are float64 [14][n] for the parity path and float32 [14][n] when p.precision = R6_PREC_F32
template <class R>
__device__ __forceinline__ void env_load(const R6Buffers &b, int64_t n, int64_t i, EnvT<R> &e)
{
    const R *state = reinterpret_cast<const R *>(b.state);
#pragma unroll
    for (int c = 0; c < 14; c++) e.y[c] = state[(int64_t)c * n + i];
    e.m0 = b.m0[i];
    e.v0 = b.v0[i];
    e.k = b.step_count[i];
    e.episode = b.episode_id[i];
    e.ep_return = b.ep_return[i];
    e.tgo = b.tgo != nullptr ? b.tgo[i] : 0.0f;
}
template <class R>
__device__ __forceinline__ void env_store(const R6Buffers &b, int64_t n, int64_t i, const EnvT<R> &e)
{
    R *state = reinterpret_cast<R *>(b.state);
#pragma unroll
    for (int c = 0; c < 14; c++) state[(int64_t)c * n + i] = e.y[c];
    b.m0[i] = e.m0;
    b.v0[i] = e.v0;
    b.step_count[i] = e.k;
    b.episode_id[i] = e.episode;
    b.ep_return[i] = e.ep_return;
    if (b.tgo != nullptr) b.tgo[i] = e.tgo;
}

template <class R>
__device__ __forceinline__ void write_terminal_state(const R6Buffers &b, int64_t n, int64_t i, const R *y)
{
    R *ts = reinterpret_cast<R *>(b.terminal_state);
#pragma unroll
    for (int c = 0; c < 14; c++) ts[(int64_t)c * n + i] = y[c];
}

template <class R>
__device__ __forceinline__ void write_obs(float *obs, int64_t n, int64_t i, const R6Params &p, const Derived &dv,
                                          const R *y)
{
    const int rows = p.obs_rows > 0 ? p.obs_rows : 14;
#pragma unroll
    for (int c = 0; c < 14; c++)
        if (c < rows) obs[(int64_t)c * n + i] = obs_component(p, dv, y, c);   // rocket_env.py:503-504
}

// The outputs of an env-step.  reward_terms is written by the one-step kernels only (step_kernel, post_body): in a
// rollout it would keep the terms live across the step loop.
__device__ __forceinline__ void write_step_out(const R6Buffers &b, int64_t i, const StepOut &o)
{
    if (b.reward) b.reward[i] = o.reward;
    if (b.reward_f32) b.reward_f32[i] = (float)o.reward;
    b.done[i] = o.finished ? 1 : 0;
    b.flags[i] = (uint8_t)o.flags;
    if (b.nattempts) b.nattempts[i] = (uint8_t)o.natt;
    if (b.status) b.status[i] = (int8_t)o.status;
}

// (return, length) of the episode that just ended
template <class R>
__device__ __forceinline__ void write_ep_info(const R6Buffers &b, int64_t n, int64_t i, const EnvT<R> &e)
{
    if (b.ep_info) { b.ep_info[i] = e.ep_return; b.ep_info[n + i] = (double)e.k; }
}

// End of an episode with the post-step state in registers: batch statistics, terminal observation / state
// (DummyVecEnv's terminal_observation, montecarlo_script.py:35) and (return, length)
template <class R>
__device__ __forceinline__ void end_episode(const R6Params &p, const R6Buffers &b, const Derived &dv, int64_t n, int64_t i,
                                            const EnvT<R> &e, uint32_t flags)
{
    if (b.stats) stats_episode<R>(b.stats, flags, e.ep_return, e.k);
    write_obs(b.terminal_obs, n, i, p, dv, e.y);
    write_terminal_state(b, n, i, e.y);
    write_ep_info(b, n, i, e);
}

// ---------------------------------------------------------------------------------------------
template <class R>
__global__ void __launch_bounds__(kThreads)
reset_kernel(const R6Params p, const R6Buffers b, const Derived dv, int64_t n, int64_t env_offset, const uint8_t *mask,
             uint64_t seed)
{
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    if (mask != nullptr && mask[i] == 0) return;
    EnvT<R> e;
    e.episode = b.episode_id[i];
    env_reset(p, b, seed, env_offset + i, e);
    env_store(b, n, i, e);
    write_obs(b.obs, n, i, p, dv, e.y);
    if (b.done) b.done[i] = 0;          // un-freezes the env for one-episode (auto_reset = 0) rollouts
}

// Row-major observation block of one warp: the 32 x rows floats of the warp's envs are contiguous in a [n][rows]
// array.  Each lane parks its row in the warp's (by now dead) stage storage, then the warp streams the block out with
// fully coalesced 128-byte stores.  Warp-collective: call with every lane, `valid` = this lane has an env.
// Staging slot of (component c, lane l): the first 32 entries of the warp's span of pair row (stage c / 4, pair c % 4)
// — with the paired stage layout a warp owns [2 w0, 2 w0 + 64) of every pair row, w0 = its first thread.
template <class R>
__device__ __forceinline__ void write_obs_rows(float *obs, int64_t first_env, int rows, bool valid, const float (&ob)[14],
                                               R *smem /* the CTA's stage storage */)
{
    const int lane = threadIdx.x & 31, w0 = threadIdx.x & ~31;
    auto slot = [&](int c, int l) { return reinterpret_cast<float *>(&smem[(kNK * (c >> 2) + 2 * (c & 3)) * kThreads + 2 * w0 + l]); };
    const unsigned live = __ballot_sync(0xffffffffu, valid);
    const int n_valid = __popc(live);                       // valid lanes are a prefix (contiguous env indices)
    __syncwarp();
#pragma unroll
    for (int c = 0; c < 14; c++)
        if (c < rows) *slot(c, lane) = ob[c];
    __syncwarp();
    float *dst = obs + first_env * rows;
    const int total = n_valid * rows;
#pragma unroll
    for (int k = 0; k < 14; k++) {
        const int el = lane + 32 * k;
        if (k < rows && el < total) {
            const int env = el / rows, c = el - env * rows;
            dst[el] = *slot(c, env);
        }
    }
    __syncwarp();
}

template <class R, bool kExact>
__global__ void __launch_bounds__(kThreads, min_blocks<R>())
step_kernel(const R6Params p, const R6Buffers b, const Derived dv, int64_t n, int64_t env_offset,
            const float *__restrict__ actions, uint64_t seed)
{
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    auto K = make_kstore<R>();
    float ob[14];
    // one-episode semantics (auto_reset = 0): a finished env stays frozen until r6_reset (obs_row_major implies auto_reset)
    const bool live = i < n && (p.auto_reset || b.done[i] == 0);
    if (live) {
        EnvT<R> e;
        env_load(b, n, i, e);
        const float a0 = actions[3 * i], a1 = actions[3 * i + 1], a2 = actions[3 * i + 2];
        StepOut o;
        env_step<kExact>(p, dv, b.t_table, e, a0, a1, a2, o, K);
        write_step_out(b, i, o);
        if (b.reward_terms) {
#pragma unroll
            for (int k = 0; k < R6_NTERMS; k++) b.reward_terms[(int64_t)k * n + i] = o.post.terms[k];
        }
        if (o.finished) {
            end_episode(p, b, dv, n, i, e, o.flags);
            if (p.auto_reset) env_reset(p, b, seed, env_offset + i, e);      // with auto_reset hand back the reset obs
        }
        if (p.obs_row_major) {
#pragma unroll
            for (int c = 0; c < 14; c++) ob[c] = obs_component(p, dv, e.y, c);
        } else
            write_obs(b.obs, n, i, p, dv, e.y);
        env_store(b, n, i, e);
    }
    if (p.obs_row_major)
        write_obs_rows<R>(b.obs, (int64_t)blockIdx.x * kThreads + (threadIdx.x & ~31), p.obs_rows > 0 ? p.obs_rows : 14, i < n, ob,
                          K.base - 2 * threadIdx.x);
    if (b.stats) stats_steps(b.stats, live ? 1 : 0);
}

// the action of env i in the kernel pair: from the [n][3] buffer, or from Philox without one (r6_step_random)
__device__ __forceinline__ void step_action(const float *__restrict__ actions, uint64_t seed, int64_t env_offset,
                                            int64_t step_index, int64_t i, float &a0, float &a1, float &a2)
{
    if (actions != nullptr) { a0 = actions[3 * i]; a1 = actions[3 * i + 1]; a2 = actions[3 * i + 2]; }
    else philox_action(seed, (uint64_t)(env_offset + i), (uint64_t)step_index, a0, a1, a2);
}

// Integrator pass kPass of env i on the state in `state`: 0 = the whole step (env_integrate), 1 = probe + the first
// px.budget attempts, 2 = resumed from px.  Returns true while the env is unfinished (kPass != 0); a finished env's
// status and attempt count go to `scratch` for post_kernel.
template <bool kExact, int kPass, class R, class KS>
__device__ __forceinline__ bool integrate_env(const R6Params &p, const R6Buffers &b, int64_t n, int64_t i,
                                              const float *__restrict__ actions, uint64_t seed, int64_t env_offset,
                                              int64_t step_index, KS &K, PassCtx<R> &px)
{
    R *state = reinterpret_cast<R *>(b.state);
    R y[14];
#pragma unroll
    for (int c = 0; c < 14; c++) y[c] = state[(int64_t)c * n + i];
    float a0, a1, a2;
    step_action(actions, seed, env_offset, step_index, i, a0, a1, a2);
    int status, natt;
    if constexpr (kPass == 0) env_integrate<kExact>(p, b.t_table, y, b.m0[i], b.step_count[i], a0, a1, a2, K, status, natt);
    else status = env_integrate_pass<kExact, kPass>(p, b.t_table, y, b.m0[i], kPass == 1 ? b.step_count[i] : 0, a0, a1, a2, K,
                                                    px, natt);
#pragma unroll
    for (int c = 0; c < 14; c++) state[(int64_t)c * n + i] = y[c];
    const bool unfinished = kPass != 0 && status == -2;
    if (!unfinished) {
        b.scratch[i] = (uint8_t)(int8_t)status;
        b.scratch[n + i] = (uint8_t)natt;
    }
    return unfinished;
}

// The same env-step as two kernels (used by r6_step when R6Buffers.scratch is given): the divergent, register- and
// shared-memory-hungry integrator on its own, with a hot instruction footprint that fits the instruction cache, and
// a uniform post-step kernel (reward, flags, wrappers, statistics, auto-reset, observation) without stage storage
// that runs at twice the occupancy.  Costs one extra read of the state (+128 B per env-step, HBM is at 10 %).
template <class R, bool kExact>
__global__ void __launch_bounds__(kIntThreads, int_ctas<R>())
integrate_kernel(const R6Params p, const R6Buffers b, int64_t n, const float *__restrict__ actions, int64_t env_offset,
                 uint64_t seed, int64_t step_index, int64_t i0, int64_t i1)
{
    const int64_t i = i0 + (int64_t)blockIdx.x * kIntThreads + threadIdx.x;     // this launch steps envs [i0, i1)
    auto K = make_kstore<R, kIntThreads>();
    grid_dependency_wait();
    if (i >= i1) return;
    if (!p.auto_reset && b.done[i] != 0) return;      // one-episode semantics: a finished env stays frozen until r6_reset
    PassCtx<R> px;
    integrate_env<kExact, 0>(p, b, n, i, actions, seed, env_offset, step_index, K, px);
}

// ---- multi-pass integration (R6Buffers.work given): the integrator cut at RK-attempt boundaries -------------------
// A warp pays for the slowest of its 32 envs, and the attempt count of a step is 1 for a third of the envs, 2 for
// most and 3-4 for ~1 %: in one kernel a warp runs 2.26 attempts for a mean of 1.64.  Here every pass runs ONE
// attempt per env (the first one also the initial-step probe) and compacts the unfinished envs into a work list for
// the next pass, so lanes never idle through an attempt they do not need:
//   integrate_first_kernel   all envs of the range: probe + attempt 1            -> list 0
//   integrate_resume_kernel  list 0: attempt 2                                   -> list 1
//   integrate_resume_kernel  list 1: the remaining attempts (budget unlimited)
// Carried per unfinished env: (t, h_abs, reference height of the density series) + (attempts, rejected) — see
// integrate<..., kPass>; y is already in `state`.  The per-env arithmetic is that of integrate_kernel bit for bit.
constexpr int kMaxLanes = R6_MAX_LANES;
struct WorkView {
    int32_t *count;          // [2 * kMaxLanes] entries of list l of lane a: count[2 a + l]
    int32_t *list[2];        // [n] env index; a range [i0, i1) uses the slots [i0, i1) of each array
    int32_t *meta[2];        // [n] attempts | rejected << 8
    double *ctx[2];          // [4][n] t, h_abs, h_ref, t_bound
};
__host__ __device__ inline WorkView work_view(uint8_t *w, int64_t n)
{
    WorkView v;
    v.count = reinterpret_cast<int32_t *>(w);
    int32_t *q = reinterpret_cast<int32_t *>(w + 256);
    v.list[0] = q; v.list[1] = q + n; v.meta[0] = q + 2 * n; v.meta[1] = q + 3 * n;
    double *d = reinterpret_cast<double *>(w + 256 + 16 * n);
    v.ctx[0] = d; v.ctx[1] = d + 4 * n;
    return v;
}

template <class R>
__device__ __forceinline__ void work_append(const WorkView &W, int64_t n, int dst, int lane, int64_t i0, bool unfinished,
                                            int64_t i, const PassCtx<R> &px)
{
    const unsigned m = __ballot_sync(0xffffffffu, unfinished);
    if (m == 0) return;
    const int lid = threadIdx.x & 31, leader = __ffs(m) - 1;
    int base = 0;
    if (lid == leader) base = atomicAdd(&W.count[2 * lane + dst], __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (unfinished) {
        const int64_t slot = i0 + base + __popc(m & ((1u << lid) - 1u));
        W.list[dst][slot] = (int32_t)i;
        W.meta[dst][slot] = px.natt | (px.rejected ? 256 : 0);
        double *c = W.ctx[dst];
        c[slot] = (double)px.t; c[n + slot] = (double)px.h_abs; c[2 * n + slot] = (double)px.h_ref;
        c[3 * n + slot] = (double)px.t_bound;
    }
}

template <class R, bool kExact>
__global__ void __launch_bounds__(kIntThreads, first_ctas<R>())
integrate_first_kernel(const R6Params p, const R6Buffers b, int64_t n, const float *__restrict__ actions, int64_t env_offset,
                       uint64_t seed, int64_t step_index, int64_t i0, int64_t i1, int lane)
{
    const int64_t i = i0 + (int64_t)blockIdx.x * kIntThreads + threadIdx.x;
    auto K = make_kstore<R, kIntThreads>();
    PassCtx<R> px;
    bool unfinished = false;
    grid_dependency_wait();
    if (i < i1 && (p.auto_reset || b.done[i] == 0)) {       // one-episode semantics: finished envs stay frozen
        px.budget = 1;
        unfinished = integrate_env<kExact, 1>(p, b, n, i, actions, seed, env_offset, step_index, K, px);
    }
    work_append<R>(work_view(b.work, n), n, 0, lane, i0, unfinished, i, px);
}

// kLast = false: one attempt per env (pass 0, list 0 -> list 1); kLast = true: the remaining attempts, however many
template <class R, bool kExact, bool kLast>
__global__ void __launch_bounds__(kIntThreads, int_ctas<R>())
integrate_resume_kernel(const R6Params p, const R6Buffers b, int64_t n, const float *__restrict__ actions, int64_t env_offset,
                        uint64_t seed, int64_t step_index, int64_t i0, int lane)
{
    constexpr int src = kLast ? 1 : 0;
    constexpr int budget = kLast ? (1 << 30) : 1;
    auto K = make_kstore<R, kIntThreads>();
    const WorkView W = work_view(b.work, n);
    grid_dependency_wait();
    const int64_t cnt = W.count[2 * lane + src];
    for (int64_t s0 = (int64_t)blockIdx.x * kIntThreads; s0 < cnt; s0 += (int64_t)gridDim.x * kIntThreads) {
        const int64_t slot = s0 + threadIdx.x;
        PassCtx<R> px;
        bool unfinished = false;
        int64_t i = 0;
        if (slot < cnt) {
            i = W.list[src][i0 + slot];
            const int meta = W.meta[src][i0 + slot];
            const double *c = W.ctx[src];
            px.t = (R)c[i0 + slot]; px.h_abs = (R)c[n + i0 + slot]; px.h_ref = (R)c[2 * n + i0 + slot];
            px.t_bound = (R)c[3 * n + i0 + slot];
            px.natt = meta & 255; px.rejected = (meta & 256) != 0; px.budget = budget;
            unfinished = integrate_env<kExact, 2>(p, b, n, i, actions, seed, env_offset, step_index, K, px);
        }
        if constexpr (!kLast) work_append<R>(W, n, 1, lane, i0, unfinished, i, px);
    }
}

#ifndef R6_POST_BLOCKS
#define R6_POST_BLOCKS 7         /* resident post-step CTAs per SM (no stage storage: registers are the only limit);
                                    5 (94 registers, no spills) .. 8 (64 registers) measured within 2 % of each other */
#endif
#ifndef R6_POST_THREADS
#define R6_POST_THREADS R6_THREADS
#endif
constexpr int kPostThreads = R6_POST_THREADS;

// Everything of the post-step after its inputs are in registers
template <class R>
__device__ __forceinline__ void post_body(const R6Params &p, const R6Buffers &b, const Derived &dv, int64_t n, int64_t i,
                                          int64_t env_offset, uint64_t seed, EnvT<R> &e, float a0, float a1, float a2, int status,
                                          int natt)
{
    write_obs(b.obs, n, i, p, dv, e.y);          // first thing: the float64 state is then dead but for q and the casts
    StepOut o;
    env_post(p, dv, e, a0, a1, a2, status, natt, o);
    write_step_out(b, i, o);
    if (b.reward_terms) {
#pragma unroll
        for (int k = 0; k < R6_NTERMS; k++) b.reward_terms[(int64_t)k * n + i] = o.post.terms[k];
    }
    if (o.finished) {
        // rare (one env-step in ~140): the post-step state is read back from `state` (nothing has written it since
        // the integrator) so that the 14 doubles are not kept alive through the reward code for this path's sake.
        // (Moving this path out of line into a __noinline__ function cost 5-8 us: measured, rejected.)
        if (b.stats) stats_episode<R>(b.stats, o.flags, e.ep_return, e.k);
        write_ep_info(b, n, i, e);
        const R *state = reinterpret_cast<const R *>(b.state);
        if (p.auto_reset) {
            R yt[14];
#pragma unroll
            for (int c = 0; c < 14; c++) yt[c] = state[(int64_t)c * n + i];
            write_obs(b.terminal_obs, n, i, p, dv, yt);
            write_terminal_state(b, n, i, yt);
            env_reset(p, b, seed, env_offset + i, e);
            write_obs(b.obs, n, i, p, dv, e.y);          // replaces the terminal observation written above
            env_store(b, n, i, e);
        } else {
#pragma unroll 1
            for (int c = 0; c < 14; c++) {               // one-episode semantics: record the terminal state / observation
                const R yc = state[(int64_t)c * n + i];
                reinterpret_cast<R *>(b.terminal_state)[(int64_t)c * n + i] = yc;
                if (c < (p.obs_rows > 0 ? p.obs_rows : 14)) b.terminal_obs[(int64_t)c * n + i] = obs_scalar(p, dv, yc, c);
            }
        }
    }
    if (!(o.finished && p.auto_reset)) {         // the integrator already stored the state
        b.step_count[i] = e.k;
        b.ep_return[i] = e.ep_return;
        if (b.tgo != nullptr) b.tgo[i] = e.tgo;
    }
}

template <class R>
__global__ void __launch_bounds__(kPostThreads, R6_POST_BLOCKS)
post_kernel(const R6Params p, const R6Buffers b, const Derived dv, int64_t n, int64_t env_offset,
            const float *__restrict__ actions, uint64_t seed, int64_t step_index, int64_t i0, int64_t i1, int lane)
{
    const int64_t i = i0 + (int64_t)blockIdx.x * kPostThreads + threadIdx.x;
    grid_dependency_wait();
    if (b.work != nullptr && blockIdx.x == 0 && threadIdx.x < 2)          // the lane's work lists are consumed: empty them
        reinterpret_cast<int32_t *>(b.work)[2 * lane + threadIdx.x] = 0;
    const bool live = i < i1 && (p.auto_reset || b.done[i] == 0);      // frozen envs (auto_reset = 0, done) are skipped
    if (live) {
        EnvT<R> e;
        env_load(b, n, i, e);
        float a0, a1, a2;
        step_action(actions, seed, env_offset, step_index, i, a0, a1, a2);
        const int status = (int)(int8_t)b.scratch[i], natt = (int)b.scratch[n + i];
        post_body(p, b, dv, n, i, env_offset, seed, e, a0, a1, a2, status, natt);
    }
    if (b.stats) stats_steps(b.stats, live ? 1 : 0);
}

// The trajectory record of a rollout (each pointer nullable): obs [k][13][n], actions [k][n][3], rewards and done [k][n]
struct Traj {
    float *obs, *act, *rew;
    uint8_t *done;
};

// Step j of a rollout on the registers of `e`: record the observation and action, step, record reward and done, count
// the step; at the end of an episode reset the env (auto_reset) or freeze it and pad the rest of the record (reward 0,
// done = 2).  Returns true when the env froze.
template <bool kExact, class R, class KS>
__device__ __forceinline__ bool rollout_step(const R6Params &p, const R6Buffers &b, const Derived &dv, int64_t n, int64_t i,
                                             int64_t env_offset, uint64_t seed, const Traj &tr, int j, int k_steps, float a0,
                                             float a1, float a2, EnvT<R> &e, StepOut &o, KS &K, int &steps)
{
    if (tr.obs) {
#pragma unroll
        for (int c = 0; c < 13; c++) tr.obs[((int64_t)j * 13 + c) * n + i] = obs_component(p, dv, e.y, c);
    }
    if (tr.act) { float *a = tr.act + ((int64_t)j * n + i) * 3; a[0] = a0; a[1] = a1; a[2] = a2; }
    env_step<kExact>(p, dv, b.t_table, e, a0, a1, a2, o, K);
    if (tr.rew) tr.rew[(int64_t)j * n + i] = (float)o.reward;
    if (tr.done) tr.done[(int64_t)j * n + i] = o.finished ? 1 : 0;
    steps++;
    if (o.finished) {
        end_episode(p, b, dv, n, i, e, o.flags);
        if (!p.auto_reset) {
            for (int jj = j + 1; jj < k_steps; jj++) {
                if (tr.rew) tr.rew[(int64_t)jj * n + i] = 0.0f;
                if (tr.done) tr.done[(int64_t)jj * n + i] = 2;
            }
            return true;
        }
        env_reset(p, b, seed, env_offset + i, e);
    }
    return false;
}

// the end of a rollout: the last step's outputs, the observation and the env registers
template <class R>
__device__ __forceinline__ void rollout_store(const R6Params &p, const R6Buffers &b, const Derived &dv, int64_t n, int64_t i,
                                              const EnvT<R> &e, const StepOut &o)
{
    write_step_out(b, i, o);
    write_obs(b.obs, n, i, p, dv, e.y);
    env_store(b, n, i, e);
}

// k fused steps, state in registers; actions from Philox, a [k][n][3] buffer or the fused policy MLP.
// p.auto_reset != 0: finished envs restart (VecEnv semantics).  p.auto_reset == 0: an env that finishes
// is left frozen with done = 1 and its terminal state / observation recorded (evaluate_policy /
// Monte-Carlo semantics: one episode per env), and is skipped by later launches until r6_reset.
template <class R, int kMode, bool kExact>
__global__ void __launch_bounds__(kThreads, kMode == R6_ACT_MLP ? 2 : min_blocks<R>())   // MLP: weights take the 3rd CTA's smem
rollout_kernel(const R6Params p, const R6Buffers b, const Derived dv, int64_t n, int64_t env_offset, int k_steps,
               const float *__restrict__ act_buf, const R6Mlp mlp, uint64_t seed, int64_t step_base, float *traj_obs,
               float *traj_act, float *traj_rew, uint8_t *traj_done)
{
    const Traj tr = {traj_obs, traj_act, traj_rew, traj_done};
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    auto K = make_kstore<R>();
    const float *W = nullptr;
    if (kMode == R6_ACT_MLP) {
        // pack the policy weights into shared memory once per CTA (transposes W1, pads W0 rows)
        extern __shared__ __align__(16) double r6_smem[];
        float *Ws = reinterpret_cast<float *>(reinterpret_cast<char *>(r6_smem) + smem_bytes<R>());
        for (int idx = threadIdx.x; idx < kMlpFloats; idx += kThreads) Ws[idx] = mlp_pack_element(mlp, idx);
        __syncthreads();
        W = Ws;
    }
    int my_steps = 0;
    if (i < n && (p.auto_reset || b.done[i] == 0)) {
        EnvT<R> e;
        env_load(b, n, i, e);
        StepOut o;
        o.reward = 0; o.flags = 0; o.finished = false; o.natt = 0; o.status = 0;
#pragma unroll 1
        for (int j = 0; j < k_steps; j++) {
            float a0, a1, a2;
            if (kMode == R6_ACT_PHILOX) philox_action(seed, (uint64_t)(env_offset + i), (uint64_t)(step_base + j), a0, a1, a2);
            else if (kMode == R6_ACT_MLP) {
                float x[kMlpIn];
#pragma unroll
                for (int c = 0; c < kMlpIn; c++) x[c] = obs_component(p, dv, e.y, c);
                mlp_policy(W, x, a0, a1, a2);
            } else {
                const float *a = act_buf + ((int64_t)j * n + i) * 3;
                a0 = a[0]; a1 = a[1]; a2 = a[2];
            }
            if (rollout_step<kExact>(p, b, dv, n, i, env_offset, seed, tr, j, k_steps, a0, a1, a2, e, o, K, my_steps)) break;
        }
        rollout_store(p, b, dv, n, i, e, o);
    }
    if (b.stats) stats_steps(b.stats, my_steps);
}

// Closed-loop rollout with the policy on the tensor cores (R6_ACT_MLP_TC): same semantics as
// rollout_kernel<R, R6_ACT_MLP, false>, but the network is evaluated warp-collectively (r6_mlp_tc.cuh), so the
// step loop is warp-uniform: lanes without a live env keep taking part in the MMAs and skip the dynamics.
template <class R>
__global__ void __launch_bounds__(kThreads, 2)
rollout_tc_kernel(const R6Params p, const R6Buffers b, const Derived dv, int64_t n, int64_t env_offset, int k_steps,
                  const R6Mlp mlp, uint64_t seed, float *traj_obs, float *traj_act, float *traj_rew, uint8_t *traj_done)
{
    const Traj tr = {traj_obs, traj_act, traj_rew, traj_done};
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    auto K = make_kstore<R>();
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(reinterpret_cast<char *>(r6_smem) + smem_bytes<R>());
    for (int idx = threadIdx.x; idx < kMlpTcFloats; idx += kThreads) Ws[idx] = mlp_tc_pack_element(mlp, idx);
    __syncthreads();
    float *scratch = Ws + kMlpTcFloats + (threadIdx.x >> 5) * (16 * 33);
    int my_steps = 0;
    const bool loaded = i < n && (p.auto_reset || b.done[i] == 0);
    bool live = loaded;
    EnvT<R> e;
    if (loaded) env_load(b, n, i, e);
    else {
#pragma unroll
        for (int c = 0; c < 14; c++) e.y[c] = 0;
        e.m0 = 1; e.v0 = 0; e.k = 0; e.episode = 0; e.ep_return = 0; e.tgo = 0;
    }
    StepOut o;
    o.reward = 0; o.flags = 0; o.finished = false; o.natt = 0; o.status = 0;
#pragma unroll 1
    for (int j = 0; j < k_steps; j++) {
        if (!__any_sync(0xffffffffu, live)) break;
        float x[kMlpIn], a0, a1, a2;
#pragma unroll
        for (int c = 0; c < kMlpIn; c++) x[c] = obs_component(p, dv, e.y, c);
        mlp_policy_tc(Ws, scratch, x, a0, a1, a2);
        if (live && rollout_step<false>(p, b, dv, n, i, env_offset, seed, tr, j, k_steps, a0, a1, a2, e, o, K, my_steps))
            live = false;
    }
    if (loaded) rollout_store(p, b, dv, n, i, e, o);
    if (b.stats) stats_steps(b.stats, my_steps);
}

// Simulator6DOF.step, raw (all-float64) mode
template <bool kExact>
__global__ void __launch_bounds__(kThreads, R6_MIN_BLOCKS)
sim_raw_kernel(double *state, const double *u, const double *m0, const double *t, double dt, int64_t n,
               int8_t *status, uint8_t *nattempts)
{
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    auto K = make_kstore<double>();
    if (i >= n) return;
    double y[14];
#pragma unroll
    for (int c = 0; c < 14; c++) y[c] = state[(int64_t)c * n + i];
    StepConst c;
    consts_raw_mode(c, m0[i], u[i], u[n + i], u[2 * n + i], y[10]);
    int natt;
    const int st = integrate<kExact>(c, y, t[i], dt, natt, K);
    normalize_quat(y);
#pragma unroll
    for (int k = 0; k < 14; k++) state[(int64_t)k * n + i] = y[k];
    status[i] = (int8_t)st;
    if (nattempts) nattempts[i] = (uint8_t)natt;
}

__global__ void __launch_bounds__(kThreads)
tgo_kernel(const double *c2, const double *c3, const double *c4, double c0, int64_t n, const double *guess, double *out)
{
    const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i < n) out[i] = tgo_largest_root(c0, c2[i], c3[i], c4[i], guess != nullptr ? guess[i] : 0.0);
}

// What a policy launch writes besides the env actions, and how the action is chosen (r6_policy_ex)
struct PolicyOut {
    float *actions, *raw, *values, *logp;     // [n][3] clipped, [n][3] nullable, [n] nullable, [n] nullable
    int stochastic;
    uint64_t seed;
    int64_t env_offset, step;
    int64_t i0, i1;                           // env sub-range of this launch (r6_policy_range); n stays the obs stride
};
__device__ __forceinline__ void policy_store(const PolicyOut &po, int64_t i, const float (&raw)[3], float logp, float value)
{
#pragma unroll
    for (int c = 0; c < 3; c++) {
        po.actions[3 * i + c] = fminf(fmaxf(raw[c], -1.0f), 1.0f);
        if (po.raw) po.raw[3 * i + c] = raw[c];
    }
    if (po.values) po.values[i] = value;
    if (po.logp) po.logp[i] = logp;
}
__device__ __forceinline__ void policy_epilogue(const PolicyOut &po, const float *log_std, int64_t i, const float (&out)[4])
{
    float raw[3], logp;
    gaussian_head(out, log_std, po.stochastic != 0, po.seed, (uint64_t)(po.env_offset + i), (uint64_t)po.step, raw, logp);
    policy_store(po, i, raw, logp, out[3]);
}
// the gSDE head from the latent sums nz (h E) and var (h^2 sigma^2) of env i
__device__ __forceinline__ void sde_epilogue(const PolicyOut &po, int64_t i, const float (&out)[4], const float (&nz)[3],
                                             const float (&var)[3])
{
    float raw[3], logp;
    sde_head(out, nz, var, po.stochastic != 0, raw, logp);
    policy_store(po, i, raw, logp, out[3]);
}
// gSDE inputs of a policy launch: log_std [64][3] and the xi [192][n] buffer of r6_sde_noise
struct SdeIn {
    const float *log_std, *xi;
};
// sigma = exp(log_std) and sigma^2 (one float32 product, as SB3's std ** 2) into shared memory
__device__ __forceinline__ void sde_stage(const float *log_std, float *sig, float *sig2, int tid, int nthreads)
{
    for (int c = tid; c < kSdeXi; c += nthreads) {
        const float sg = expf(log_std[c]);
        sig[c] = sg;
        sig2[c] = sg * sg;
    }
}

// StateDependentNoiseDistribution.sample_weights (r6_sde_noise): one thread per (env, Philox block); blockIdx.y = block
__global__ void __launch_bounds__(256)
sde_noise_kernel(uint64_t seed, int64_t env_offset, int64_t step, int64_t n, int64_t i0, int64_t i1, float *__restrict__ xi)
{
    const int64_t i = i0 + (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= i1) return;
    float z[4];
    sde_noise_block(seed, (uint64_t)(env_offset + i), (uint64_t)step, b, z);
#pragma unroll
    for (int q = 0; q < 4; q++) xi[(int64_t)(4 * b + q) * n + i] = z[q];
}

// The policy as its own kernel (r6_policy / r6_policy_ex): uniform work, no integrator state => small code, high
// occupancy.  Persistent: the grid is one wave of CTAs, each packs the weights into shared memory ONCE (the gather
// with its index arithmetic costs as much as one network evaluation) and then walks over its tiles of 128 envs.
template <bool kTc>
__global__ void __launch_bounds__(kThreads, kTc ? 3 : 4)
policy_kernel(const R6Mlp mlp, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(r6_smem);
    const int nW = kTc ? kMlpTcFloats : kMlpFloats;
    for (int idx = threadIdx.x; idx < nW; idx += kThreads) Ws[idx] = kTc ? mlp_tc_pack_element(mlp, idx) : mlp_pack_element(mlp, idx);
    __syncthreads();
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kThreads - 1) / kThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t i = po.i0 + tile * kThreads + threadIdx.x;
        float x[kMlpIn], out[4];
#pragma unroll
        for (int c = 0; c < kMlpIn; c++) x[c] = i < i1 ? obs[(int64_t)c * n + i] : 0.0f;
        if (kTc) mlp_forward_tc(Ws, Ws + kMlpTcFloats + (threadIdx.x >> 5) * (16 * 33), x, out);
        else mlp_forward(Ws, x, out);
        if (i < i1) policy_epilogue(po, mlp.log_std, i, out);
    }
}
constexpr int kSmemPolicyTc = (r6::kMlpTcFloats + (kThreads / 32) * 16 * 33) * (int)sizeof(float);
constexpr int kSmemPolicy = r6::kMlpFloats * (int)sizeof(float);

// The policy with the gSDE head on float32 FMAs (r6_policy_sde_range tensor_cores = 0): policy_kernel<false> plus, per
// unit k of the last hidden layer, nz_a += h_k (sigma_ka xi_ka) and var_a += h_k^2 sigma_ka^2 (xi read coalesced over envs)
__global__ void __launch_bounds__(kThreads, 4)
policy_sde_kernel(const R6Mlp mlp, const SdeIn sde, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(r6_smem);
    float *sig = Ws + kMlpFloats, *sig2 = sig + kSdeXi;
    for (int idx = threadIdx.x; idx < kMlpFloats; idx += kThreads) Ws[idx] = mlp_pack_element(mlp, idx);
    sde_stage(sde.log_std, sig, sig2, threadIdx.x, kThreads);
    __syncthreads();
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kThreads - 1) / kThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t i = po.i0 + tile * kThreads + threadIdx.x;
        const bool in = i < i1, draw = in && po.stochastic != 0;
        float x[kMlpIn], out[4], nz[3] = {0.0f, 0.0f, 0.0f}, var[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int c = 0; c < kMlpIn; c++) x[c] = in ? obs[(int64_t)c * n + i] : 0.0f;
        mlp_forward_latent(Ws, x, out, [&](int k, float h) {
            const float hh = h * h;
#pragma unroll
            for (int a = 0; a < 3; a++) {
                const int c = 3 * k + a;
                if (draw) nz[a] = f32_fma(h, sig[c] * __ldg(sde.xi + (int64_t)c * n + i), nz[a]);
                var[a] = f32_fma(hh, sig2[c], var[a]);
            }
        });
        if (in) sde_epilogue(po, i, out, nz, var);
    }
}
constexpr int kSmemPolicySde = kSmemPolicy + 2 * kSdeXi * (int)sizeof(float);

// The policy on tcgen05 with accumulators and activations in tensor memory (r6_policy tensor_cores = 3: 3xTF32, float32
// accuracy; tensor_cores = 2: single-pass TF32).  Layout, schedule and measurements: r6_mlp_tcgen05.cuh.
template <bool kFaithful>
__global__ void __launch_bounds__(tc5::kThreads, 1)
policy_tc5_kernel(const R6Mlp mlp, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    using namespace tc5;
    extern __shared__ __align__(16) double r6_smem[];
    char *S = reinterpret_cast<char *>(r6_smem);
    const int tid = threadIdx.x, group = tid >> 8, lt = tid & 127, half = (tid >> 7) & 1, warp = tid >> 5;
    // programmatic dependent launch: the previous kernel on the stream may have produced the observations — or the weights
    // (an optimiser step), so the wait comes before the weight staging, not after it
    grid_dependency_wait();
    // ---- one-time per CTA: weights split into TF32 hi / lo parts in canonical K-major tiles, biases, barriers, TMEM ----
    for (int idx = tid; idx < 128 * 16; idx += tc5::kThreads) {
        const int r = idx >> 4, k = idx & 15;
        float hi, lo;
        split_tf32(k < kMlpIn ? mlp.w0[r * kMlpIn + k] : 0.0f, hi, lo);
        *reinterpret_cast<float *>(S + kOffW0h + tile_off(r, k, 16)) = hi;
        *reinterpret_cast<float *>(S + kOffW0l + tile_off(r, k, 16)) = lo;
    }
    // W1 / W2 rows are 16-byte aligned runs of 4 consecutive k = one 16-byte chunk of the canonical tile: vector copies
    // (the staging is a fixed cost per CTA and launch: 11 264 weights)
    for (int idx = tid; idx < 64 * 32; idx += tc5::kThreads) {
        const int r = idx >> 5, k = (idx & 31) * 4;
        const float4 w = *reinterpret_cast<const float4 *>(mlp.w1 + r * kMlpH0 + k);
        float4 h, l;
        split_tf32(w.x, h.x, l.x); split_tf32(w.y, h.y, l.y); split_tf32(w.z, h.z, l.z); split_tf32(w.w, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW1h + tile_off(r, k, 128)) = h;
        *reinterpret_cast<float4 *>(S + kOffW1l + tile_off(r, k, 128)) = l;
    }
    for (int idx = tid; idx < 16 * 16; idx += tc5::kThreads) {
        const int r = idx >> 4, k = (idx & 15) * 4;
        float4 h, l;
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k) : 0.0f, h.x, l.x);
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k + 1) : 0.0f, h.y, l.y);
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k + 2) : 0.0f, h.z, l.z);
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k + 3) : 0.0f, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW2h + tile_off(r, k, 64)) = h;
        *reinterpret_cast<float4 *>(S + kOffW2l + tile_off(r, k, 64)) = l;
    }
    float *bias = reinterpret_cast<float *>(S + kOffBias);
    const float bscale = kFaithful ? kTwoLog2e : 1.0f;      // faithful mode: hidden-layer biases pre-scaled for the exp2 form of tanh
    if (tid < 128) bias[tid] = bscale * mlp.b0[tid];
    if (tid < 64) bias[128 + tid] = bscale * mlp.b1[tid];
    if (tid < 4) bias[192 + tid] = mlp_b2_row(mlp, tid);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar)) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar + 8)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(S + kOffTmemPtr)), "n"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();                      // the weight tiles are read by the async proxy (B operand of the MMAs)
    fence_before();
    __syncthreads();
    fence_after();
    // warp-uniform copies (a shuffle result is uniform to the compiler) of everything the MMA-issuing warp computes with
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t *>(S + kOffTmemPtr), 0);
    const uint32_t tmem_g = tmem_base + (uint32_t)(warp_u >> 3) * kGroupCols;              // this group's columns, lane 0
    const uint32_t tmem_row = tmem_g + ((uint32_t)((warp & 3) * 32) << 16);                // this warp's 32 TMEM lanes
    const uint32_t sbase = __shfl_sync(0xffffffffu, smem_u32(S), 0);
    const uint32_t aW0h = sbase + kOffW0h, aW0l = sbase + kOffW0l, aW1h = sbase + kOffW1h;
    const uint32_t aW1l = sbase + kOffW1l, aW2h = sbase + kOffW2h, aW2l = sbase + kOffW2l;
    const uint32_t bar = sbase + kOffBar + 8 * (uint32_t)(warp_u >> 3);
    const bool issuer = (warp_u & 7) == 0;          // the first warp of each group issues its MMAs (one elected lane each)
    uint32_t phase = 0;
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kTile - 1) / kTile;
    // Both groups run the SAME number of tile slots (a slot past the end is all masked rows) so that the epilogue token
    // is handed over a matching number of times.
    const int64_t slots = (tiles + 2 * (int64_t)gridDim.x - 1) / (2 * (int64_t)gridDim.x);
    // this thread's 8 observation components of one tile, as loaded (split and stored one slot later)
    float xo[8];
    auto load_obs = [&](int64_t tile) {
        const int64_t i = po.i0 + tile * kTile + lt;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int k = 8 * half + q;
            xo[q] = (k < kMlpIn && i < i1) ? __ldg(obs + (int64_t)k * n + i) : 0.0f;
        }
    };
    load_obs(2 * (int64_t)blockIdx.x + group);
    float outv[4] = {0.0f, 0.0f, 0.0f, 0.0f};      // the output layer of the previous tile, written out one slot later
    int64_t out_i = i1;
    if (group == 1) token_pass(0);                 // group 0 takes the first epilogue turn
    for (int64_t slot = 0; slot < slots; slot++) {
        const int64_t tile = 2 * ((int64_t)blockIdx.x + slot * gridDim.x) + group;
        const int64_t i = po.i0 + tile * kTile + lt;
        // ---- observations of this thread's env, split -> row `lt` of the input tile: 8 of its 16 K columns per thread ----
        {
            float h[8], l[8];
#pragma unroll
            for (int q = 0; q < 8; q++) split_tf32(xo[q], h[q], l[q]);
            tmem_st8(tmem_row + kColD1 + 8 * half, h);
            if (kFaithful) tmem_st8(tmem_row + kColL + 8 * half, l);
            tmem_st_wait();
        }
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW0h, aW0l, 512, 2, 128, false); if (elect_one()) mma_commit(bar); }
        load_obs(tile + 2 * (int64_t)gridDim.x);       // next slot's observations: in flight under this tile's three layers
        if (half == 0 && out_i < i1) policy_epilogue(po, mlp.log_std, out_i, outv);   // the previous tile's outputs, under MMA0
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- hidden layer 0, first half of the units -> layer 1 partial product ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0, bias, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0, tmem_g + kColL, aW1h, aW1l, 4096, 8, 64, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- second half ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0 + 64, bias + 64, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0 + 64, tmem_g + kColL, aW1h + 2048, aW1l + 2048, 4096, 8, 64, true); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- hidden layer 1 -> output layer (its 16 accumulator columns reuse the head of the dead D0) ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD1, bias + 128, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW2h, aW2l, 2048, 8, 16, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        out_i = i1;
        if (half == 0) {
            tmem_ld4(tmem_row + kColD0, outv);
#pragma unroll
            for (int q = 0; q < 4; q++) outv[q] += bias[192 + q];
            out_i = i;
        }
        // no barrier here: the next slot's input stores go to D1 / L (their reader, this tile's last MMA, has completed),
        // and the next MMA0, which overwrites the columns just read, is issued behind the group barrier that follows them
    }
    if (half == 0 && out_i < i1) policy_epilogue(po, mlp.log_std, out_i, outv);
    if (group == 0) token_take(0);                 // consume group 1's last hand-over: no barrier is left half-arrived at exit
    fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
}

// policy_kernel<false> for SB3 1.6's separate towers (R6Mlp with the value tower): mlp_forward_sep.  At the shared
// kernel's four CTAs per SM (128 registers) ptxas spills 276 B of it (the shared kernel: 24 B); it asks for 255
// registers unbounded, so fewer CTAs per SM do not remove the spill (three: 168 registers, 220 B).
__global__ void __launch_bounds__(kThreads, 4)
policy_sep_kernel(const R6Mlp mlp, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(r6_smem);
    for (int idx = threadIdx.x; idx < kMlpFloatsSep; idx += kThreads) Ws[idx] = mlp_pack_element_sep(mlp, idx);
    __syncthreads();
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kThreads - 1) / kThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t i = po.i0 + tile * kThreads + threadIdx.x;
        float x[kMlpIn], out[4];
#pragma unroll
        for (int c = 0; c < kMlpIn; c++) x[c] = i < i1 ? obs[(int64_t)c * n + i] : 0.0f;
        mlp_forward_sep(Ws, x, out);
        if (i < i1) policy_epilogue(po, mlp.log_std, i, out);
    }
}
constexpr int kSmemPolicySep = r6::kMlpFloatsSep * (int)sizeof(float);

// policy_tc5_kernel for the separate towers (r6_policy tensor_cores = 2 / 3 with the value tower set): stacked layer 0,
// then the value chain (reduced to the value in its epilogue), then the policy chain and the action head.  Schedule and
// TMEM use: r6_mlp_tcgen05.cuh.  A copy of policy_tc5_kernel rather than a template flag of it, so that the shared-trunk
// kernel keeps its register allocation.
template <bool kFaithful>
__global__ void __launch_bounds__(tc5::kThreads, 1)
policy_tc5_sep_kernel(const R6Mlp mlp, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    using namespace tc5;
    extern __shared__ __align__(16) double r6_smem[];
    char *S = reinterpret_cast<char *>(r6_smem);
    const int tid = threadIdx.x, group = tid >> 8, lt = tid & 127, half = (tid >> 7) & 1, warp = tid >> 5;
    grid_dependency_wait();
    // ---- one-time per CTA: [w0; vf_w0] and [w1 | vf_w1] split into TF32 hi / lo parts in canonical K-major tiles ----
    for (int idx = tid; idx < 128 * 16; idx += tc5::kThreads) {
        const int r = idx >> 4, k = idx & 15;
        const float *w0 = r < kMlpH1 ? mlp.w0 + r * kMlpIn : mlp.vf_w0 + (r - kMlpH1) * kMlpIn;
        float hi, lo;
        split_tf32(k < kMlpIn ? w0[k] : 0.0f, hi, lo);
        *reinterpret_cast<float *>(S + kOffW0h + tile_off(r, k, 16)) = hi;
        *reinterpret_cast<float *>(S + kOffW0l + tile_off(r, k, 16)) = lo;
    }
    for (int idx = tid; idx < 64 * 32; idx += tc5::kThreads) {
        const int r = idx >> 5, k = (idx & 31) * 4;
        const float *src = k < kMlpH1 ? mlp.w1 + r * kMlpH1 + k : mlp.vf_w1 + r * kMlpH1 + (k - kMlpH1);
        const float4 w = *reinterpret_cast<const float4 *>(src);
        float4 h, l;
        split_tf32(w.x, h.x, l.x); split_tf32(w.y, h.y, l.y); split_tf32(w.z, h.z, l.z); split_tf32(w.w, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW1h + tile_off(r, k, 128)) = h;
        *reinterpret_cast<float4 *>(S + kOffW1l + tile_off(r, k, 128)) = l;
    }
    for (int idx = tid; idx < 16 * 16; idx += tc5::kThreads) {        // action_net rows 0..2; row 3 (value) stays zero
        const int r = idx >> 4, k = (idx & 15) * 4;
        float4 h, l;
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k] : 0.0f, h.x, l.x);
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k + 1] : 0.0f, h.y, l.y);
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k + 2] : 0.0f, h.z, l.z);
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k + 3] : 0.0f, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW2h + tile_off(r, k, 64)) = h;
        *reinterpret_cast<float4 *>(S + kOffW2l + tile_off(r, k, 64)) = l;
    }
    float *bias = reinterpret_cast<float *>(S + kOffBias);
    float *vb1 = reinterpret_cast<float *>(S + kOffSep), *wv = reinterpret_cast<float *>(S + kOffSepWv);
    float *vpart = reinterpret_cast<float *>(S + kOffSepPart) + group * kTile;
    const float bscale = kFaithful ? kTwoLog2e : 1.0f;
    if (tid < 64) bias[tid] = bscale * mlp.b0[tid];
    else if (tid < 128) bias[tid] = bscale * mlp.vf_b0[tid - 64];
    if (tid < 64) {
        bias[128 + tid] = bscale * mlp.b1[tid];
        vb1[tid] = bscale * mlp.vf_b1[tid];
        wv[tid] = mlp.wv != nullptr ? mlp.wv[tid] : 0.0f;
    }
    if (tid < 4) bias[192 + tid] = mlp_b2_row(mlp, tid);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar)) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar + 8)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(S + kOffTmemPtr)), "n"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t *>(S + kOffTmemPtr), 0);
    const uint32_t tmem_g = tmem_base + (uint32_t)(warp_u >> 3) * kGroupCols;
    const uint32_t tmem_row = tmem_g + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t sbase = __shfl_sync(0xffffffffu, smem_u32(S), 0);
    const uint32_t aW0h = sbase + kOffW0h, aW0l = sbase + kOffW0l, aW1h = sbase + kOffW1h;
    const uint32_t aW1l = sbase + kOffW1l, aW2h = sbase + kOffW2h, aW2l = sbase + kOffW2l;
    const uint32_t bar = sbase + kOffBar + 8 * (uint32_t)(warp_u >> 3);
    const bool issuer = (warp_u & 7) == 0;
    uint32_t phase = 0;
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kTile - 1) / kTile;
    const int64_t slots = (tiles + 2 * (int64_t)gridDim.x - 1) / (2 * (int64_t)gridDim.x);
    float xo[8];
    auto load_obs = [&](int64_t tile) {
        const int64_t i = po.i0 + tile * kTile + lt;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int k = 8 * half + q;
            xo[q] = (k < kMlpIn && i < i1) ? __ldg(obs + (int64_t)k * n + i) : 0.0f;
        }
    };
    load_obs(2 * (int64_t)blockIdx.x + group);
    float outv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    int64_t out_i = i1;
    if (group == 1) token_pass(0);
    for (int64_t slot = 0; slot < slots; slot++) {
        const int64_t tile = 2 * ((int64_t)blockIdx.x + slot * gridDim.x) + group;
        const int64_t i = po.i0 + tile * kTile + lt;
        {
            float h[8], l[8];
#pragma unroll
            for (int q = 0; q < 8; q++) split_tf32(xo[q], h[q], l[q]);
            tmem_st8(tmem_row + kColD1 + 8 * half, h);
            if (kFaithful) tmem_st8(tmem_row + kColL + 8 * half, l);
            tmem_st_wait();
        }
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW0h, aW0l, 512, 2, 128, false); if (elect_one()) mma_commit(bar); }
        load_obs(tile + 2 * (int64_t)gridDim.x);
        if (half == 0 && out_i < i1) policy_epilogue(po, mlp.log_std, out_i, outv);
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- value tower: layer 0 units 64..127 -> its layer 1 (W1 columns 64..127 = vf_w1) ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0 + 64, bias + 64, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0 + 64, tmem_g + kColL, aW1h + 2048, aW1l + 2048, 4096, 8, 64, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- value = value_net(tanh(D1 + vf_b1)) on the CUDA cores; the second half's sum goes through shared memory ----
        const float vs = epilogue_value<kFaithful>(tmem_row, kColD1, vb1, wv, half, group);
        if (half == 1) vpart[lt] = vs;
        // ---- policy tower: layer 0 units 0..63 -> its layer 1 (W1 columns 0..63 = w1), over the value chain's D1 ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0, bias, half, group);
        fence_before(); group_sync(group);       // also publishes vpart to the first half
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0, tmem_g + kColL, aW1h, aW1l, 4096, 8, 64, false); if (elect_one()) mma_commit(bar); }
        const float value = half == 0 ? vs + vpart[lt] : 0.0f;
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- policy latent -> action_net ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD1, bias + 128, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW2h, aW2l, 2048, 8, 16, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        out_i = i1;
        if (half == 0) {
            tmem_ld4(tmem_row + kColD0, outv);
#pragma unroll
            for (int q = 0; q < 3; q++) outv[q] += bias[192 + q];
            outv[3] = value + bias[195];
            out_i = i;
        }
    }
    if (half == 0 && out_i < i1) policy_epilogue(po, mlp.log_std, out_i, outv);
    if (group == 0) token_take(0);
    fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
}

// policy_tc5_kernel with the gSDE head (r6_policy_sde_range tensor_cores = 2 / 3): the sums h E and h^2 sigma^2 are
// formed in the last hidden layer's epilogue (epilogue_in_tmem_sde), where each of the two threads of an env row holds
// 32 of the 64 activations; the second half hands its sums to the first through shared memory (kOffSdePart), and the
// first writes the env's outputs.  A copy of policy_tc5_kernel rather than a template flag of it, so that the plain
// kernel keeps its register allocation.
template <bool kFaithful>
__global__ void __launch_bounds__(tc5::kThreads, 1)
policy_tc5_sde_kernel(const R6Mlp mlp, const SdeIn sde, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    using namespace tc5;
    extern __shared__ __align__(16) double r6_smem[];
    char *S = reinterpret_cast<char *>(r6_smem);
    const int tid = threadIdx.x, group = tid >> 8, lt = tid & 127, half = (tid >> 7) & 1, warp = tid >> 5;
    // programmatic dependent launch: the previous kernel on the stream may have produced the observations — or the weights
    // (an optimiser step), so the wait comes before the weight staging, not after it
    grid_dependency_wait();
    // ---- one-time per CTA: weights split into TF32 hi / lo parts in canonical K-major tiles, biases, barriers, TMEM ----
    for (int idx = tid; idx < 128 * 16; idx += tc5::kThreads) {
        const int r = idx >> 4, k = idx & 15;
        float hi, lo;
        split_tf32(k < kMlpIn ? mlp.w0[r * kMlpIn + k] : 0.0f, hi, lo);
        *reinterpret_cast<float *>(S + kOffW0h + tile_off(r, k, 16)) = hi;
        *reinterpret_cast<float *>(S + kOffW0l + tile_off(r, k, 16)) = lo;
    }
    // W1 / W2 rows are 16-byte aligned runs of 4 consecutive k = one 16-byte chunk of the canonical tile: vector copies
    // (the staging is a fixed cost per CTA and launch: 11 264 weights)
    for (int idx = tid; idx < 64 * 32; idx += tc5::kThreads) {
        const int r = idx >> 5, k = (idx & 31) * 4;
        const float4 w = *reinterpret_cast<const float4 *>(mlp.w1 + r * kMlpH0 + k);
        float4 h, l;
        split_tf32(w.x, h.x, l.x); split_tf32(w.y, h.y, l.y); split_tf32(w.z, h.z, l.z); split_tf32(w.w, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW1h + tile_off(r, k, 128)) = h;
        *reinterpret_cast<float4 *>(S + kOffW1l + tile_off(r, k, 128)) = l;
    }
    for (int idx = tid; idx < 16 * 16; idx += tc5::kThreads) {
        const int r = idx >> 4, k = (idx & 15) * 4;
        float4 h, l;
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k) : 0.0f, h.x, l.x);
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k + 1) : 0.0f, h.y, l.y);
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k + 2) : 0.0f, h.z, l.z);
        split_tf32(r < kMlpRows ? mlp_w2_row(mlp, r, k + 3) : 0.0f, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW2h + tile_off(r, k, 64)) = h;
        *reinterpret_cast<float4 *>(S + kOffW2l + tile_off(r, k, 64)) = l;
    }
    float *bias = reinterpret_cast<float *>(S + kOffBias);
    const float bscale = kFaithful ? kTwoLog2e : 1.0f;      // faithful mode: hidden-layer biases pre-scaled for the exp2 form of tanh
    if (tid < 128) bias[tid] = bscale * mlp.b0[tid];
    if (tid < 64) bias[128 + tid] = bscale * mlp.b1[tid];
    if (tid < 4) bias[192 + tid] = mlp_b2_row(mlp, tid);
    sde_stage(sde.log_std, reinterpret_cast<float *>(S + kOffSde), reinterpret_cast<float *>(S + kOffSde) + kSdeXi, tid,
              tc5::kThreads);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar)) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar + 8)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(S + kOffTmemPtr)), "n"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();                      // the weight tiles are read by the async proxy (B operand of the MMAs)
    fence_before();
    __syncthreads();
    fence_after();
    // warp-uniform copies (a shuffle result is uniform to the compiler) of everything the MMA-issuing warp computes with
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t *>(S + kOffTmemPtr), 0);
    const uint32_t tmem_g = tmem_base + (uint32_t)(warp_u >> 3) * kGroupCols;              // this group's columns, lane 0
    const uint32_t tmem_row = tmem_g + ((uint32_t)((warp & 3) * 32) << 16);                // this warp's 32 TMEM lanes
    const uint32_t sbase = __shfl_sync(0xffffffffu, smem_u32(S), 0);
    const uint32_t aW0h = sbase + kOffW0h, aW0l = sbase + kOffW0l, aW1h = sbase + kOffW1h;
    const uint32_t aW1l = sbase + kOffW1l, aW2h = sbase + kOffW2h, aW2l = sbase + kOffW2l;
    const uint32_t bar = sbase + kOffBar + 8 * (uint32_t)(warp_u >> 3);
    const bool issuer = (warp_u & 7) == 0;          // the first warp of each group issues its MMAs (one elected lane each)
    uint32_t phase = 0;
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kTile - 1) / kTile;
    // Both groups run the SAME number of tile slots (a slot past the end is all masked rows) so that the epilogue token
    // is handed over a matching number of times.
    const int64_t slots = (tiles + 2 * (int64_t)gridDim.x - 1) / (2 * (int64_t)gridDim.x);
    // this thread's 8 observation components of one tile, as loaded (split and stored one slot later)
    float xo[8];
    auto load_obs = [&](int64_t tile) {
        const int64_t i = po.i0 + tile * kTile + lt;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int k = 8 * half + q;
            xo[q] = (k < kMlpIn && i < i1) ? __ldg(obs + (int64_t)k * n + i) : 0.0f;
        }
    };
    load_obs(2 * (int64_t)blockIdx.x + group);
    float outv[4] = {0.0f, 0.0f, 0.0f, 0.0f};      // the output layer of the previous tile, written out one slot later
    float nzv[3] = {0.0f, 0.0f, 0.0f}, varv[3] = {0.0f, 0.0f, 0.0f};   // and its latent sums
    int64_t out_i = i1;
    if (group == 1) token_pass(0);                 // group 0 takes the first epilogue turn
    for (int64_t slot = 0; slot < slots; slot++) {
        const int64_t tile = 2 * ((int64_t)blockIdx.x + slot * gridDim.x) + group;
        const int64_t i = po.i0 + tile * kTile + lt;
        // ---- observations of this thread's env, split -> row `lt` of the input tile: 8 of its 16 K columns per thread ----
        {
            float h[8], l[8];
#pragma unroll
            for (int q = 0; q < 8; q++) split_tf32(xo[q], h[q], l[q]);
            tmem_st8(tmem_row + kColD1 + 8 * half, h);
            if (kFaithful) tmem_st8(tmem_row + kColL + 8 * half, l);
            tmem_st_wait();
        }
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW0h, aW0l, 512, 2, 128, false); if (elect_one()) mma_commit(bar); }
        load_obs(tile + 2 * (int64_t)gridDim.x);       // next slot's observations: in flight under this tile's three layers
        if (half == 0 && out_i < i1) sde_epilogue(po, out_i, outv, nzv, varv);        // the previous tile's outputs, under MMA0
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- hidden layer 0, first half of the units -> layer 1 partial product ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0, bias, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0, tmem_g + kColL, aW1h, aW1l, 4096, 8, 64, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- second half ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0 + 64, bias + 64, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0 + 64, tmem_g + kColL, aW1h + 2048, aW1l + 2048, 4096, 8, 64, true); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- hidden layer 1 -> output layer (its 16 accumulator columns reuse the head of the dead D0) ----
        float pnz[3], pvar[3];
        float *const sig = reinterpret_cast<float *>(S + kOffSde), *const sig2 = sig + kSdeXi;
        float *const part = reinterpret_cast<float *>(S + kOffSdePart) + (group * kTile + lt) * 6;   // this row's exchange slot
        epilogue_in_tmem_sde<kFaithful>(tmem_row, kColD1, bias + 128, half, group, sig, sig2, sde.xi, n, i,
                                        po.stochastic != 0 && i < i1, pnz, pvar);
        if (half == 1) {                 // read by the row's first half after the group barrier below
#pragma unroll
            for (int a = 0; a < 3; a++) { part[a] = pnz[a]; part[3 + a] = pvar[a]; }
        }
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW2h, aW2l, 2048, 8, 16, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        out_i = i1;
        if (half == 0) {
            tmem_ld4(tmem_row + kColD0, outv);
#pragma unroll
            for (int q = 0; q < 4; q++) outv[q] += bias[192 + q];
#pragma unroll
            for (int a = 0; a < 3; a++) { nzv[a] = pnz[a] + part[a]; varv[a] = pvar[a] + part[3 + a]; }
            out_i = i;
        }
        // no barrier here: the next slot's input stores go to D1 / L (their reader, this tile's last MMA, has completed),
        // and the next MMA0, which overwrites the columns just read, is issued behind the group barrier that follows them
    }
    if (half == 0 && out_i < i1) sde_epilogue(po, out_i, outv, nzv, varv);
    if (group == 0) token_take(0);                 // consume group 1's last hand-over: no barrier is left half-arrived at exit
    fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
}

// policy_sep_kernel with the gSDE head (r6_policy_sde_sep_range tensor_cores = 0): the sums of policy_sde_kernel over the
// POLICY tower's latent (mlp_forward_sep_latent), sigma and sigma^2 staged after the packed weights
__global__ void __launch_bounds__(kThreads, 4)
policy_sep_sde_kernel(const R6Mlp mlp, const SdeIn sde, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(r6_smem);
    float *sig = Ws + kMlpFloatsSep, *sig2 = sig + kSdeXi;
    for (int idx = threadIdx.x; idx < kMlpFloatsSep; idx += kThreads) Ws[idx] = mlp_pack_element_sep(mlp, idx);
    sde_stage(sde.log_std, sig, sig2, threadIdx.x, kThreads);
    __syncthreads();
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kThreads - 1) / kThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int64_t i = po.i0 + tile * kThreads + threadIdx.x;
        const bool in = i < i1, draw = in && po.stochastic != 0;
        float x[kMlpIn], out[4], nz[3] = {0.0f, 0.0f, 0.0f}, var[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int c = 0; c < kMlpIn; c++) x[c] = in ? obs[(int64_t)c * n + i] : 0.0f;
        mlp_forward_sep_latent(Ws, x, out, [&](int k, float h) {
            const float hh = h * h;
#pragma unroll
            for (int a = 0; a < 3; a++) {
                const int c = 3 * k + a;
                if (draw) nz[a] = f32_fma(h, sig[c] * __ldg(sde.xi + (int64_t)c * n + i), nz[a]);
                var[a] = f32_fma(hh, sig2[c], var[a]);
            }
        });
        if (in) sde_epilogue(po, i, out, nz, var);
    }
}
constexpr int kSmemPolicySepSde = kSmemPolicySep + 2 * kSdeXi * (int)sizeof(float);

// policy_tc5_sep_kernel with the gSDE head (r6_policy_sde_sep_range tensor_cores = 2 / 3): the policy latent's epilogue
// (the last hidden-layer epilogue, on D1 after the policy chain) is epilogue_in_tmem_sde, and the second column half hands
// its sums to the first through shared memory as in policy_tc5_sde_kernel.  The value chain is policy_tc5_sep_kernel's.
// Shared memory: the separate-tower region (kOffSep..) and then the gSDE region (kOffSepSde..).
template <bool kFaithful>
__global__ void __launch_bounds__(tc5::kThreads, 1)
policy_tc5_sep_sde_kernel(const R6Mlp mlp, const SdeIn sde, const float *__restrict__ obs, int64_t n, const PolicyOut po)
{
    using namespace tc5;
    extern __shared__ __align__(16) double r6_smem[];
    char *S = reinterpret_cast<char *>(r6_smem);
    const int tid = threadIdx.x, group = tid >> 8, lt = tid & 127, half = (tid >> 7) & 1, warp = tid >> 5;
    grid_dependency_wait();
    // ---- one-time per CTA: [w0; vf_w0] and [w1 | vf_w1] split into TF32 hi / lo parts in canonical K-major tiles ----
    for (int idx = tid; idx < 128 * 16; idx += tc5::kThreads) {
        const int r = idx >> 4, k = idx & 15;
        const float *w0 = r < kMlpH1 ? mlp.w0 + r * kMlpIn : mlp.vf_w0 + (r - kMlpH1) * kMlpIn;
        float hi, lo;
        split_tf32(k < kMlpIn ? w0[k] : 0.0f, hi, lo);
        *reinterpret_cast<float *>(S + kOffW0h + tile_off(r, k, 16)) = hi;
        *reinterpret_cast<float *>(S + kOffW0l + tile_off(r, k, 16)) = lo;
    }
    for (int idx = tid; idx < 64 * 32; idx += tc5::kThreads) {
        const int r = idx >> 5, k = (idx & 31) * 4;
        const float *src = k < kMlpH1 ? mlp.w1 + r * kMlpH1 + k : mlp.vf_w1 + r * kMlpH1 + (k - kMlpH1);
        const float4 w = *reinterpret_cast<const float4 *>(src);
        float4 h, l;
        split_tf32(w.x, h.x, l.x); split_tf32(w.y, h.y, l.y); split_tf32(w.z, h.z, l.z); split_tf32(w.w, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW1h + tile_off(r, k, 128)) = h;
        *reinterpret_cast<float4 *>(S + kOffW1l + tile_off(r, k, 128)) = l;
    }
    for (int idx = tid; idx < 16 * 16; idx += tc5::kThreads) {        // action_net rows 0..2; row 3 (value) stays zero
        const int r = idx >> 4, k = (idx & 15) * 4;
        float4 h, l;
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k] : 0.0f, h.x, l.x);
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k + 1] : 0.0f, h.y, l.y);
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k + 2] : 0.0f, h.z, l.z);
        split_tf32(r < kMlpOut ? mlp.w2[r * kMlpH1 + k + 3] : 0.0f, h.w, l.w);
        *reinterpret_cast<float4 *>(S + kOffW2h + tile_off(r, k, 64)) = h;
        *reinterpret_cast<float4 *>(S + kOffW2l + tile_off(r, k, 64)) = l;
    }
    float *bias = reinterpret_cast<float *>(S + kOffBias);
    float *vb1 = reinterpret_cast<float *>(S + kOffSep), *wv = reinterpret_cast<float *>(S + kOffSepWv);
    float *vpart = reinterpret_cast<float *>(S + kOffSepPart) + group * kTile;
    const float bscale = kFaithful ? kTwoLog2e : 1.0f;
    if (tid < 64) bias[tid] = bscale * mlp.b0[tid];
    else if (tid < 128) bias[tid] = bscale * mlp.vf_b0[tid - 64];
    if (tid < 64) {
        bias[128 + tid] = bscale * mlp.b1[tid];
        vb1[tid] = bscale * mlp.vf_b1[tid];
        wv[tid] = mlp.wv != nullptr ? mlp.wv[tid] : 0.0f;
    }
    if (tid < 4) bias[192 + tid] = mlp_b2_row(mlp, tid);
    sde_stage(sde.log_std, reinterpret_cast<float *>(S + kOffSepSde), reinterpret_cast<float *>(S + kOffSepSde) + kSdeXi, tid,
              tc5::kThreads);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar)) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(S + kOffBar + 8)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(S + kOffTmemPtr)), "n"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const int warp_u = __shfl_sync(0xffffffffu, warp, 0);
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile uint32_t *>(S + kOffTmemPtr), 0);
    const uint32_t tmem_g = tmem_base + (uint32_t)(warp_u >> 3) * kGroupCols;
    const uint32_t tmem_row = tmem_g + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t sbase = __shfl_sync(0xffffffffu, smem_u32(S), 0);
    const uint32_t aW0h = sbase + kOffW0h, aW0l = sbase + kOffW0l, aW1h = sbase + kOffW1h;
    const uint32_t aW1l = sbase + kOffW1l, aW2h = sbase + kOffW2h, aW2l = sbase + kOffW2l;
    const uint32_t bar = sbase + kOffBar + 8 * (uint32_t)(warp_u >> 3);
    const bool issuer = (warp_u & 7) == 0;
    uint32_t phase = 0;
    const int64_t i1 = po.i1;
    const int64_t tiles = (i1 - po.i0 + kTile - 1) / kTile;
    const int64_t slots = (tiles + 2 * (int64_t)gridDim.x - 1) / (2 * (int64_t)gridDim.x);
    float xo[8];
    auto load_obs = [&](int64_t tile) {
        const int64_t i = po.i0 + tile * kTile + lt;
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int k = 8 * half + q;
            xo[q] = (k < kMlpIn && i < i1) ? __ldg(obs + (int64_t)k * n + i) : 0.0f;
        }
    };
    load_obs(2 * (int64_t)blockIdx.x + group);
    float outv[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    float nzv[3] = {0.0f, 0.0f, 0.0f}, varv[3] = {0.0f, 0.0f, 0.0f};
    int64_t out_i = i1;
    if (group == 1) token_pass(0);
    for (int64_t slot = 0; slot < slots; slot++) {
        const int64_t tile = 2 * ((int64_t)blockIdx.x + slot * gridDim.x) + group;
        const int64_t i = po.i0 + tile * kTile + lt;
        {
            float h[8], l[8];
#pragma unroll
            for (int q = 0; q < 8; q++) split_tf32(xo[q], h[q], l[q]);
            tmem_st8(tmem_row + kColD1 + 8 * half, h);
            if (kFaithful) tmem_st8(tmem_row + kColL + 8 * half, l);
            tmem_st_wait();
        }
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW0h, aW0l, 512, 2, 128, false); if (elect_one()) mma_commit(bar); }
        load_obs(tile + 2 * (int64_t)gridDim.x);
        if (half == 0 && out_i < i1) sde_epilogue(po, out_i, outv, nzv, varv);
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- value tower: layer 0 units 64..127 -> its layer 1 (W1 columns 64..127 = vf_w1) ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0 + 64, bias + 64, half, group);
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0 + 64, tmem_g + kColL, aW1h + 2048, aW1l + 2048, 4096, 8, 64, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- value = value_net(tanh(D1 + vf_b1)) on the CUDA cores; the second half's sum goes through shared memory ----
        const float vs = epilogue_value<kFaithful>(tmem_row, kColD1, vb1, wv, half, group);
        if (half == 1) vpart[lt] = vs;
        // ---- policy tower: layer 0 units 0..63 -> its layer 1 (W1 columns 0..63 = w1), over the value chain's D1 ----
        epilogue_in_tmem<kFaithful>(tmem_row, kColD0, bias, half, group);
        fence_before(); group_sync(group);       // also publishes vpart to the first half
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD1, tmem_g + kColD0, tmem_g + kColL, aW1h, aW1l, 4096, 8, 64, false); if (elect_one()) mma_commit(bar); }
        const float value = half == 0 ? vs + vpart[lt] : 0.0f;
        bar_wait(bar, phase); phase ^= 1; fence_after();
        // ---- policy latent -> action_net, with the gSDE sums over this thread's 32 latent units ----
        float pnz[3], pvar[3];
        float *const sig = reinterpret_cast<float *>(S + kOffSepSde), *const sig2 = sig + kSdeXi;
        float *const part = reinterpret_cast<float *>(S + kOffSepSdePart) + (group * kTile + lt) * 6;   // this row's exchange slot
        epilogue_in_tmem_sde<kFaithful>(tmem_row, kColD1, bias + 128, half, group, sig, sig2, sde.xi, n, i,
                                        po.stochastic != 0 && i < i1, pnz, pvar);
        if (half == 1) {                 // read by the row's first half after the group barrier below
#pragma unroll
            for (int a = 0; a < 3; a++) { part[a] = pnz[a]; part[3 + a] = pvar[a]; }
        }
        fence_before(); group_sync(group);
        if (issuer) { fence_after(); issue_mmas<kFaithful>(tmem_g + kColD0, tmem_g + kColD1, tmem_g + kColL, aW2h, aW2l, 2048, 8, 16, false); if (elect_one()) mma_commit(bar); }
        bar_wait(bar, phase); phase ^= 1; fence_after();
        out_i = i1;
        if (half == 0) {
            tmem_ld4(tmem_row + kColD0, outv);
#pragma unroll
            for (int q = 0; q < 3; q++) outv[q] += bias[192 + q];
            outv[3] = value + bias[195];
#pragma unroll
            for (int a = 0; a < 3; a++) { nzv[a] = pnz[a] + part[a]; varv[a] = pvar[a] + part[3 + a]; }
            out_i = i;
        }
    }
    if (half == 0 && out_i < i1) sde_epilogue(po, out_i, outv, nzv, varv);
    if (group == 0) token_take(0);
    fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
}

// GAE scan: one thread per env walks its column of the [T][n] trajectory backwards (every access coalesced over
// envs).  HBM-bound: 17 B per (t, env).  No FMA contraction: the float32 roundings are NumPy's.
__global__ void __launch_bounds__(256)
gae_kernel(const float *__restrict__ rew, const float *__restrict__ values, const uint8_t *__restrict__ done,
           const float *__restrict__ last_values, int T, int64_t n, float gamma, float gl, float *__restrict__ adv,
           float *__restrict__ ret)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    float next_v = last_values[i], last = 0.0f;
    for (int t = T - 1; t >= 0; t--) {
        const int64_t o = (int64_t)t * n + i;
        const float v = values[o];
        const float nnt = done[o] ? 0.0f : 1.0f;
        const float delta = __fsub_rn(__fadd_rn(rew[o], __fmul_rn(__fmul_rn(gamma, next_v), nnt)), v);
        last = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nnt), last));
        adv[o] = last;
        ret[o] = __fadd_rn(last, v);
        next_v = v;
    }
}

// Time-limit bootstrap of a collected rollout (SB3 1.6 OnPolicyAlgorithm.collect_rollouts: rewards[idx] += gamma *
// V(terminal_observation) where TimeLimit.truncated).  After each env step, every env whose step was a truncation files
// the step index and the 13 observation rows of its terminal observation into its first free slot (slot_step < 0); an env
// that did not truncate reads its one flags byte and nothing else.  Every thread waits for the env step first, so that
// this grid never completes ahead of it and a programmatic dependent launched after this one still sees the step's output.
__global__ void __launch_bounds__(256)
trunc_record_kernel(const uint8_t *__restrict__ flags, const float *__restrict__ terminal_obs, int64_t n, int64_t i0, int64_t i1,
                    int step, int slots, int32_t *__restrict__ slot_step, float *__restrict__ slot_obs)
{
    const int64_t i = i0 + (int64_t)blockIdx.x * 256 + threadIdx.x;
    grid_dependency_wait();
    if (i >= i1 || !(flags[i] & R6_F_TRUNCATED)) return;
    for (int s = 0; s < slots; s++) {                    // never past slot slots - 1: a further truncation is dropped
        int32_t *st = slot_step + (int64_t)s * n + i;
        if (*st >= 0) continue;
        *st = step;
        float *o = slot_obs + (int64_t)s * 13 * n + i;
#pragma unroll
        for (int c = 0; c < 13; c++) o[(int64_t)c * n] = terminal_obs[(int64_t)c * n + i];
        return;
    }
}

// rew[t][i] = fl32(rew[t][i] + fl32(gamma * V[s][i])) for every filed slot (s, i) with t = slot_step[s][i] in [0, T):
// float32 reward buffer, float32 value, python-float gamma, two roundings and no FMA, as SB3 computes it.  Two slots of one
// env never hold the same step, so every (t, i) is touched at most once.
__global__ void __launch_bounds__(256)
trunc_bootstrap_kernel(float *__restrict__ rew, int T, int64_t n, int slots, const int32_t *__restrict__ slot_step,
                       const float *__restrict__ slot_values, float gamma)
{
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    for (int s = 0; s < slots; s++) {
        const int t = slot_step[(int64_t)s * n + i];
        if (t < 0 || t >= T) continue;
        float *r = rew + (int64_t)t * n + i;
        *r = __fadd_rn(*r, __fmul_rn(gamma, slot_values[(int64_t)s * n + i]));
    }
}

// PPO minibatch gradient (r6_ppo_grad).  A grid of ppo_ctas(B) CTAs (a function of B only, so the summation order and
// the result do not depend on the device) walks tiles of 128 samples.  Each thread runs the forward pass, loss head
// and deltas of its sample (r6_ppo.cuh) and stages its inputs, activations and deltas in shared memory unit-major,
// [unit][sample]; the CTA then accumulates the weight gradients cooperatively into register accumulators that live
// across all its tiles: dW1 (64 x 128) as an 8 x 8 block per thread, dW0 with db0 (128 x 14) one row per thread, the
// heads (dW2, dwv, db1) on threads 0..63 and the scalar sums on 64..75.  Every accumulator adds its samples in tile
// order, one fma per sample.  The dW1 block is parked in shared memory between tiles (registers would spill).  Each CTA writes one partial [P] and its float64 term sums into the work buffer, and
// ppo_reduce_kernel adds the partials in CTA order.
constexpr int kPpoTS = kThreads + 4;   // row stride of the [unit][sample] tiles: 16-byte rows, conflict-free float4 reads
constexpr int kPpoRowH0 = 0, kPpoRowH1 = 128, kPpoRowD1 = 192, kPpoRowX = 256, kPpoRowG = 272, kPpoRowT = 280;
constexpr int kPpoRows = 284;          // h0 (then delta0) 128, h1 64, delta1 64, x 16, head gradients + bad-index flag 8,
                                       // loss terms 4
constexpr int kPpoAccW1 = kMlpH1 * kMlpH0;     // dW1 accumulators, [r * 8 + c][thread]
constexpr int kSmemPpo = (kMlpFloats + kPpoRows * kPpoTS + kPpoAccW1) * (int)sizeof(float);   // 224,976 B: 1 CTA per SM
constexpr int kPpoMaxCtas = 148;
static_assert(kThreads == 128 && kMlpFloats % 4 == 0 && kPpoRowG + 8 == kPpoRowT, "PPO tile layout");
// gSDE (ppo_grad_sde_kernel): rows G + 4 .. G + 6 carry r_a instead of the log_std gradient, one more row holds the
// per-sample entropy, and sigma^2 [64][3] follows the dW1 accumulators: 226,272 B
constexpr int kPpoRowE = kPpoRowT + 4, kPpoRowsSde = kPpoRows + 1;
constexpr int kSmemPpoSde = (kMlpFloats + kPpoRowsSde * kPpoTS + kPpoAccW1 + kSdeXi) * (int)sizeof(float);
static_assert(kSmemPpoSde <= 232448, "PPO gSDE tile layout");
int64_t ppo_ctas(int64_t B)
{
    const int64_t tiles = (B + kThreads - 1) / kThreads;
    return tiles < kPpoMaxCtas ? tiles : kPpoMaxCtas;
}

// kVfClip: SB3's clip_range_vf = vfc > 0 (ppo_value_clip on every sample, reading ro.old_values); the false
// instantiations are the kernels without it, unchanged
template <bool kSde, bool kVfClip>
__device__ __forceinline__ void ppo_grad_body(const R6Mlp mlp, const float *sde_log_std, const R6PpoRollout ro,
                                              const int64_t *__restrict__ idx, int64_t B, float clip, float vf, float ent,
                                              float vfc, const double *__restrict__ adv_stats, double *__restrict__ part_terms,
                                              float *__restrict__ part)
{
    constexpr int kP = kSde ? kPpoParamsSde : kPpoParams, kNT = kSde ? R6_PPO_NTERMS_SDE : R6_PPO_NTERMS;
    constexpr int kRows = kSde ? kPpoRowsSde : kPpoRows;
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(r6_smem);
    float *S = Ws + kMlpFloats;
    float *A1 = S + kRows * kPpoTS;
    float *sig2 = A1 + kPpoAccW1;            // gSDE only
    const int tid = threadIdx.x, kq = tid & 7, jq = tid >> 3;
    for (int i = tid; i < kMlpFloats; i += kThreads) Ws[i] = mlp_pack_element(mlp, i);
    for (int i = tid; i < kPpoAccW1; i += kThreads) A1[i] = 0.0f;
    if constexpr (kSde) {
        for (int c = tid; c < kSdeXi; c += kThreads) {
            const float sg = expf(sde_log_std[c]);
            sig2[c] = sg * sg;
        }
    }
    float aLs[3] = {0.0f, 0.0f, 0.0f};       // gSDE: sum_s r_a h_tid^2 (threads 0..63)
    const int64_t nsamp = ro.T * ro.n;
    float aW0[14], aHd[5];                   // dW0[tid][0..12], db0[tid]; dW2[0..2][tid], dwv, db1
    double aS = 0.0;                         // thread 64 + r: sum of row kPpoRowG + r
#pragma unroll
    for (int c = 0; c < 14; c++) aW0[c] = 0.0f;
#pragma unroll
    for (int c = 0; c < 5; c++) aHd[c] = 0.0f;
    __syncthreads();
    const int64_t tiles = (B + kThreads - 1) / kThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        {   // this thread's sample: forward, loss head, delta1 (a slot past B or with a bad index contributes zeros)
            const int64_t s = tile * kThreads + tid;
            const int64_t q = s < B ? idx[s] : -1;
            const bool ok = q >= 0 && q < nsamp;
            float x[kMlpIn], out[4];
            if (ok) {
                const int64_t t = q / ro.n, i = q - t * ro.n;
                const float *o = ro.obs + t * ro.obs_stride_step + i * ro.obs_stride_env;
#pragma unroll
                for (int c = 0; c < kMlpIn; c++) x[c] = o[c * ro.obs_stride_comp];
            } else {
#pragma unroll
                for (int c = 0; c < kMlpIn; c++) x[c] = 0.0f;
            }
#pragma unroll
            for (int c = 0; c < kMlpIn; c++) S[(kPpoRowX + c) * kPpoTS + tid] = x[c];
            ppo_forward(Ws, x, S + kPpoRowH0 * kPpoTS + tid, S + kPpoRowH1 * kPpoTS + tid, kPpoTS, out);
            std::conditional_t<kSde, PpoHeadSde, PpoHead> hd = {};
            if (ok) {
                const float a[3] = {ro.actions[3 * q], ro.actions[3 * q + 1], ro.actions[3 * q + 2]};
                if constexpr (kSde) {
                    float var[3];
                    sde_latent_var(S + kPpoRowH1 * kPpoTS + tid, kPpoTS, sig2, var);
                    ppo_head_sde(out, a, ro.log_probs[q], ppo_advantage(ro.advantages[q], adv_stats), ro.returns[q], var, clip,
                                 vf, ent, hd);
                } else
                    ppo_head(out, a, ro.log_probs[q], ppo_advantage(ro.advantages[q], adv_stats), ro.returns[q], mlp.log_std,
                             clip, vf, ent, hd);
                if constexpr (kVfClip) ppo_value_clip(out[3], ro.old_values[q], ro.returns[q], vfc, vf, hd);
            }
            ppo_delta1(Ws, hd, S + kPpoRowH1 * kPpoTS + tid, S + kPpoRowD1 * kPpoTS + tid, kPpoTS);
#pragma unroll
            for (int r = 0; r < 7; r++) S[(kPpoRowG + r) * kPpoTS + tid] = hd.g[r];
            S[(kPpoRowG + 7) * kPpoTS + tid] = (s < B && !ok) ? 1.0f : 0.0f;
            S[(kPpoRowT + 0) * kPpoTS + tid] = hd.pg;
            S[(kPpoRowT + 1) * kPpoTS + tid] = hd.vloss;
            S[(kPpoRowT + 2) * kPpoTS + tid] = hd.clipped;
            S[(kPpoRowT + 3) * kPpoTS + tid] = hd.kl;
            if constexpr (kSde) S[kPpoRowE * kPpoTS + tid] = hd.ent;
        }
        __syncthreads();
        // dW1 += delta1^T h0 (every thread: dW1[kq + 8 r][jq + 16 c], in two halves of r), heads and scalar sums
#pragma unroll 1
        for (int r0 = 0; r0 < 8; r0 += 4) {
            float aW1[4][8];
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 8; c++) aW1[r][c] = A1[((r0 + r) * 8 + c) * kThreads + tid];
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                F4 h[8];
#pragma unroll
                for (int c = 0; c < 8; c++) h[c] = ld4(S + (kPpoRowH0 + jq + 16 * c) * kPpoTS + s4);
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const F4 d = ld4(S + (kPpoRowD1 + kq + 8 * (r0 + r)) * kPpoTS + s4);
#pragma unroll
                    for (int c = 0; c < 8; c++) {
                        float a = aW1[r][c];
                        a = __fmaf_rn(d.x, h[c].x, a); a = __fmaf_rn(d.y, h[c].y, a);
                        a = __fmaf_rn(d.z, h[c].z, a); a = __fmaf_rn(d.w, h[c].w, a);
                        aW1[r][c] = a;
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 8; c++) A1[((r0 + r) * 8 + c) * kThreads + tid] = aW1[r][c];
        }
        if (tid < kMlpH1) {
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                const F4 hv = ld4(S + (kPpoRowH1 + tid) * kPpoTS + s4), dv = ld4(S + (kPpoRowD1 + tid) * kPpoTS + s4);
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const F4 g = ld4(S + (kPpoRowG + c) * kPpoTS + s4);
                    float a = aHd[c];
                    a = __fmaf_rn(g.x, hv.x, a); a = __fmaf_rn(g.y, hv.y, a);
                    a = __fmaf_rn(g.z, hv.z, a); a = __fmaf_rn(g.w, hv.w, a);
                    aHd[c] = a;
                }
                aHd[4] = (((aHd[4] + dv.x) + dv.y) + dv.z) + dv.w;
                if constexpr (kSde) {
                    const F4 hh = {hv.x * hv.x, hv.y * hv.y, hv.z * hv.z, hv.w * hv.w};
#pragma unroll
                    for (int c = 0; c < 3; c++) {
                        const F4 r = ld4(S + (kPpoRowG + 4 + c) * kPpoTS + s4);
                        float a = aLs[c];
                        a = __fmaf_rn(r.x, hh.x, a); a = __fmaf_rn(r.y, hh.y, a);
                        a = __fmaf_rn(r.z, hh.z, a); a = __fmaf_rn(r.w, hh.w, a);
                        aLs[c] = a;
                    }
                }
            }
        } else if (tid < kMlpH1 + (kSde ? 13 : 12)) {
            const float *row = S + (kPpoRowG + tid - kMlpH1) * kPpoTS;
#pragma unroll 4
            for (int s = 0; s < kThreads; s++) aS += (double)row[s];
        }
        __syncthreads();
        {   // delta0 over h0, in place: this thread's column only
            float d1[kMlpH1];
#pragma unroll
            for (int k = 0; k < kMlpH1; k++) d1[k] = S[(kPpoRowD1 + k) * kPpoTS + tid];
#pragma unroll 1
            for (int j = 0; j < kMlpH0; j++) {
                float *p = S + (kPpoRowH0 + j) * kPpoTS + tid;
                *p = ppo_delta0(Ws, j, d1, *p);
            }
        }
        __syncthreads();
        // dW0[tid] += delta0_tid [x, 1]
#pragma unroll 1
        for (int s4 = 0; s4 < kThreads; s4 += 4) {
            const F4 d = ld4(S + (kPpoRowH0 + tid) * kPpoTS + s4);
#pragma unroll
            for (int c = 0; c < kMlpIn; c++) {
                const F4 xv = ld4(S + (kPpoRowX + c) * kPpoTS + s4);
                float a = aW0[c];
                a = __fmaf_rn(d.x, xv.x, a); a = __fmaf_rn(d.y, xv.y, a);
                a = __fmaf_rn(d.z, xv.z, a); a = __fmaf_rn(d.w, xv.w, a);
                aW0[c] = a;
            }
            aW0[13] = (((aW0[13] + d.x) + d.y) + d.z) + d.w;
        }
        __syncthreads();
    }
    float *P = part + (int64_t)blockIdx.x * kP;
#pragma unroll
    for (int r = 0; r < 8; r++)
#pragma unroll
        for (int c = 0; c < 8; c++) P[kPpoOffW1 + (kq + 8 * r) * kMlpH0 + jq + 16 * c] = A1[(r * 8 + c) * kThreads + tid];
#pragma unroll
    for (int c = 0; c < kMlpIn; c++) P[kPpoOffW0 + tid * kMlpIn + c] = aW0[c];
    P[kPpoOffB0 + tid] = aW0[13];
    if (tid < kMlpH1) {
#pragma unroll
        for (int c = 0; c < 3; c++) P[kPpoOffW2 + c * kMlpH1 + tid] = aHd[c];
        P[kPpoOffWv + tid] = aHd[3];
        P[kPpoOffB1 + tid] = aHd[4];
        if constexpr (kSde) {
#pragma unroll
            for (int c = 0; c < 3; c++) P[kPpoOffLogStd + 3 * tid + c] = aLs[c] * sig2[3 * tid + c];
        }
    } else if (tid < kMlpH1 + (kSde ? 13 : 12)) {
        const int r = tid - kMlpH1;          // rows: g0..g2 (db2), g3 (dbv), g4..g6 (dlog_std), bad index, 4 loss terms
        double *T = part_terms + (int64_t)blockIdx.x * kNT;   // (gSDE: r_a sums unused, entropy last)
        if (r < 3) P[kPpoOffB2 + r] = (float)aS;
        else if (r == 3) P[kPpoOffBv] = (float)aS;
        else if (r < 7) { if (!kSde) P[kPpoOffLogStd + r - 4] = (float)aS; }
        else if (r == 7) T[R6_PPO_T_BAD_INDEX] = aS;
        else if (r < 12) T[r - 8] = aS;
        else T[R6_PPO_T_ENTROPY] = aS;
    }
}
template <bool kVfClip>
__global__ void __launch_bounds__(kThreads, 1)
ppo_grad_kernel(const R6Mlp mlp, const R6PpoRollout ro, const int64_t *__restrict__ idx, int64_t B, float clip, float vf,
                float ent, float vfc, const double *__restrict__ adv_stats, double *__restrict__ part_terms,
                float *__restrict__ part)
{
    ppo_grad_body<false, kVfClip>(mlp, nullptr, ro, idx, B, clip, vf, ent, vfc, adv_stats, part_terms, part);
}
template <bool kVfClip>
__global__ void __launch_bounds__(kThreads, 1)
ppo_grad_sde_kernel(const R6Mlp mlp, const float *__restrict__ log_std, const R6PpoRollout ro, const int64_t *__restrict__ idx,
                    int64_t B, float clip, float vf, float ent, float vfc, const double *__restrict__ adv_stats,
                    double *__restrict__ part_terms, float *__restrict__ part)
{
    ppo_grad_body<true, kVfClip>(mlp, log_std, ro, idx, B, clip, vf, ent, vfc, adv_stats, part_terms, part);
}

// r6_ppo_grad for SB3 1.6's separate towers (ppo_grad_sep_kernel).  The same tiles, CTA count, accumulators and
// reduction as ppo_grad_kernel; the [unit][sample] tile keeps its 284 rows by giving the latent rows to the deltas in
// place: rows 128..191 hold the policy latent h1p, rows 192..255 the value latent h1v, both overwritten by their
// delta1 once the head gradients (dW2 from h1p, dwv from h1v) have been accumulated.  The 8 x 8 dW1 block of a thread
// covers dW1p[k][j] for its columns j < 64 and dW1v[k][j - 64] for j >= 64 (the stacked layer-0 units), and delta0 of
// unit j comes from its own tower's delta1.  225,232 B of shared memory (vf_b1 joins the packed weights).
constexpr int kPpoRowHP = 128, kPpoRowHV = 192;
constexpr int kSmemPpoSep = (kMlpFloatsSep + kPpoRows * kPpoTS + kPpoAccW1) * (int)sizeof(float);
static_assert(kMlpFloatsSep % 4 == 0 && kPpoRowHP == kPpoRowH1 && kPpoRowHV == kPpoRowD1 && kSmemPpoSep <= 232448,
              "PPO separate-tower tile layout");

// kVfClip as ppo_grad_body: a clipped sample's g[3] = 0 gives its value tower zero deltas through ppo_delta1_sep
template <bool kVfClip>
__global__ void __launch_bounds__(kThreads, 1)
ppo_grad_sep_kernel(const R6Mlp mlp, const R6PpoRollout ro, const int64_t *__restrict__ idx, int64_t B, float clip, float vf,
                    float ent, float vfc, const double *__restrict__ adv_stats, double *__restrict__ part_terms,
                    float *__restrict__ part)
{
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(r6_smem);
    float *S = Ws + kMlpFloatsSep;
    float *A1 = S + kPpoRows * kPpoTS;
    const int tid = threadIdx.x, kq = tid & 7, jq = tid >> 3;
    for (int i = tid; i < kMlpFloatsSep; i += kThreads) Ws[i] = mlp_pack_element_sep(mlp, i);
    for (int i = tid; i < kPpoAccW1; i += kThreads) A1[i] = 0.0f;
    const int64_t nsamp = ro.T * ro.n;
    float aW0[14], aHd[6];                   // dW0 / dvf_w0 row tid, its bias; dW2[0..2][tid], dwv, db1, dvf_b1
    double aS = 0.0;
#pragma unroll
    for (int c = 0; c < 14; c++) aW0[c] = 0.0f;
#pragma unroll
    for (int c = 0; c < 6; c++) aHd[c] = 0.0f;
    __syncthreads();
    const int64_t tiles = (B + kThreads - 1) / kThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        PpoHead hd = {};
        {   // this thread's sample: forward and loss head
            const int64_t s = tile * kThreads + tid;
            const int64_t q = s < B ? idx[s] : -1;
            const bool ok = q >= 0 && q < nsamp;
            float x[kMlpIn], out[4];
            if (ok) {
                const int64_t t = q / ro.n, i = q - t * ro.n;
                const float *o = ro.obs + t * ro.obs_stride_step + i * ro.obs_stride_env;
#pragma unroll
                for (int c = 0; c < kMlpIn; c++) x[c] = o[c * ro.obs_stride_comp];
            } else {
#pragma unroll
                for (int c = 0; c < kMlpIn; c++) x[c] = 0.0f;
            }
#pragma unroll
            for (int c = 0; c < kMlpIn; c++) S[(kPpoRowX + c) * kPpoTS + tid] = x[c];
            ppo_forward_sep(Ws, x, S + kPpoRowH0 * kPpoTS + tid, S + kPpoRowHP * kPpoTS + tid, S + kPpoRowHV * kPpoTS + tid,
                            kPpoTS, out);
            if (ok) {
                const float a[3] = {ro.actions[3 * q], ro.actions[3 * q + 1], ro.actions[3 * q + 2]};
                ppo_head(out, a, ro.log_probs[q], ppo_advantage(ro.advantages[q], adv_stats), ro.returns[q], mlp.log_std, clip,
                         vf, ent, hd);
                if constexpr (kVfClip) ppo_value_clip(out[3], ro.old_values[q], ro.returns[q], vfc, vf, hd);
            }
#pragma unroll
            for (int r = 0; r < 7; r++) S[(kPpoRowG + r) * kPpoTS + tid] = hd.g[r];
            S[(kPpoRowG + 7) * kPpoTS + tid] = (s < B && !ok) ? 1.0f : 0.0f;
            S[(kPpoRowT + 0) * kPpoTS + tid] = hd.pg;
            S[(kPpoRowT + 1) * kPpoTS + tid] = hd.vloss;
            S[(kPpoRowT + 2) * kPpoTS + tid] = hd.clipped;
            S[(kPpoRowT + 3) * kPpoTS + tid] = hd.kl;
        }
        __syncthreads();
        // heads from the latents (dW2 on h1p, dwv on h1v) and the scalar sums, before the latent rows become deltas
        if (tid < kMlpH1) {
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                const F4 hp = ld4(S + (kPpoRowHP + tid) * kPpoTS + s4), hv = ld4(S + (kPpoRowHV + tid) * kPpoTS + s4);
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const F4 g = ld4(S + (kPpoRowG + c) * kPpoTS + s4);
                    const F4 h = c < 3 ? hp : hv;
                    float a = aHd[c];
                    a = __fmaf_rn(g.x, h.x, a); a = __fmaf_rn(g.y, h.y, a);
                    a = __fmaf_rn(g.z, h.z, a); a = __fmaf_rn(g.w, h.w, a);
                    aHd[c] = a;
                }
            }
        } else if (tid < kMlpH1 + 12) {
            const float *row = S + (kPpoRowG + tid - kMlpH1) * kPpoTS;
#pragma unroll 4
            for (int s = 0; s < kThreads; s++) aS += (double)row[s];
        }
        __syncthreads();
        ppo_delta1_sep(Ws, hd, S + kPpoRowHP * kPpoTS + tid, S + kPpoRowHV * kPpoTS + tid, kPpoTS);
        __syncthreads();
        // dW1p / dW1v += delta1^T h0 (columns jq + 16 c: c < 4 policy units, c >= 4 value units), db1 / dvf_b1
#pragma unroll 1
        for (int r0 = 0; r0 < 8; r0 += 4) {
            float aW1[4][8];
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 8; c++) aW1[r][c] = A1[((r0 + r) * 8 + c) * kThreads + tid];
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                F4 h[8];
#pragma unroll
                for (int c = 0; c < 8; c++) h[c] = ld4(S + (kPpoRowH0 + jq + 16 * c) * kPpoTS + s4);
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const F4 dp = ld4(S + (kPpoRowHP + kq + 8 * (r0 + r)) * kPpoTS + s4);
                    const F4 dv = ld4(S + (kPpoRowHV + kq + 8 * (r0 + r)) * kPpoTS + s4);
#pragma unroll
                    for (int c = 0; c < 8; c++) {
                        const F4 d = c < 4 ? dp : dv;
                        float a = aW1[r][c];
                        a = __fmaf_rn(d.x, h[c].x, a); a = __fmaf_rn(d.y, h[c].y, a);
                        a = __fmaf_rn(d.z, h[c].z, a); a = __fmaf_rn(d.w, h[c].w, a);
                        aW1[r][c] = a;
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 8; c++) A1[((r0 + r) * 8 + c) * kThreads + tid] = aW1[r][c];
        }
        if (tid < kMlpH1) {
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                const F4 dp = ld4(S + (kPpoRowHP + tid) * kPpoTS + s4), dv = ld4(S + (kPpoRowHV + tid) * kPpoTS + s4);
                aHd[4] = (((aHd[4] + dp.x) + dp.y) + dp.z) + dp.w;
                aHd[5] = (((aHd[5] + dv.x) + dv.y) + dv.z) + dv.w;
            }
        }
        __syncthreads();
        {   // delta0 over h0, in place, each tower's units from its own delta1: this thread's column only
            float d1[kMlpH1];
#pragma unroll 1
            for (int t = 0; t < 2; t++) {
                const int row = t == 0 ? kPpoRowHP : kPpoRowHV;
#pragma unroll
                for (int k = 0; k < kMlpH1; k++) d1[k] = S[(row + k) * kPpoTS + tid];
#pragma unroll 1
                for (int j = t * kMlpH1; j < (t + 1) * kMlpH1; j++) {
                    float *p = S + (kPpoRowH0 + j) * kPpoTS + tid;
                    *p = ppo_delta0(Ws, j, d1, *p);
                }
            }
        }
        __syncthreads();
        // dW0[tid] += delta0_tid [x, 1]   (rows 0..63 the policy tower's w0, 64..127 the value tower's: stacked in P)
#pragma unroll 1
        for (int s4 = 0; s4 < kThreads; s4 += 4) {
            const F4 d = ld4(S + (kPpoRowH0 + tid) * kPpoTS + s4);
#pragma unroll
            for (int c = 0; c < kMlpIn; c++) {
                const F4 xv = ld4(S + (kPpoRowX + c) * kPpoTS + s4);
                float a = aW0[c];
                a = __fmaf_rn(d.x, xv.x, a); a = __fmaf_rn(d.y, xv.y, a);
                a = __fmaf_rn(d.z, xv.z, a); a = __fmaf_rn(d.w, xv.w, a);
                aW0[c] = a;
            }
            aW0[13] = (((aW0[13] + d.x) + d.y) + d.z) + d.w;
        }
        __syncthreads();
    }
    float *P = part + (int64_t)blockIdx.x * kPpoParamsSep;
#pragma unroll
    for (int r = 0; r < 8; r++)
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int k = kq + 8 * r, j = jq + 16 * c;
            P[(c < 4 ? kSepOffW1 + k * kMlpH1 + j : kSepOffVw1 + k * kMlpH1 + j - kMlpH1)] = A1[(r * 8 + c) * kThreads + tid];
        }
#pragma unroll
    for (int c = 0; c < kMlpIn; c++) P[kSepOffW0 + tid * kMlpIn + c] = aW0[c];
    P[kSepOffB0 + tid] = aW0[13];
    if (tid < kMlpH1) {
#pragma unroll
        for (int c = 0; c < 3; c++) P[kSepOffW2 + c * kMlpH1 + tid] = aHd[c];
        P[kSepOffWv + tid] = aHd[3];
        P[kSepOffB1 + tid] = aHd[4];
        P[kSepOffVb1 + tid] = aHd[5];
    } else if (tid < kMlpH1 + 12) {
        const int r = tid - kMlpH1;          // rows: g0..g2 (db2), g3 (dbv), g4..g6 (dlog_std), bad index, 4 loss terms
        double *T = part_terms + (int64_t)blockIdx.x * R6_PPO_NTERMS;
        if (r < 3) P[kSepOffB2 + r] = (float)aS;
        else if (r == 3) P[kSepOffBv] = (float)aS;
        else if (r < 7) P[kSepOffLogStd + r - 4] = (float)aS;
        else if (r == 7) T[R6_PPO_T_BAD_INDEX] = aS;
        else T[r - 8] = aS;
    }
}

// r6_ppo_grad_sde_sep: ppo_grad_sep_kernel with the gSDE head of ppo_grad_sde_kernel.  var comes from sde_latent_var over
// the POLICY latent rows (kPpoRowHP), rows G + 4 .. G + 6 carry r_a, one more row (kPpoRowE) the per-sample entropy, and
// sigma^2 [64][3] follows the dW1 accumulators.  The log_std accumulators (threads 0..63, sum_s r_a h_p^2) read the policy
// latent in the head pass, before ppo_delta1_sep overwrites its rows; the tower deltas are ppo_delta1_sep's (the latent is
// detached: no gradient through std).  226,528 B of shared memory: one CTA per SM.
constexpr int kSmemPpoSepSde = (kMlpFloatsSep + kPpoRowsSde * kPpoTS + kPpoAccW1 + kSdeXi) * (int)sizeof(float);
static_assert(kSmemPpoSepSde <= 232448 && kPpoRowE == kPpoRowG + 12, "PPO separate-tower gSDE tile layout");

template <bool kVfClip>
__global__ void __launch_bounds__(kThreads, 1)
ppo_grad_sep_sde_kernel(const R6Mlp mlp, const float *__restrict__ log_std, const R6PpoRollout ro,
                        const int64_t *__restrict__ idx, int64_t B, float clip, float vf, float ent, float vfc,
                        const double *__restrict__ adv_stats, double *__restrict__ part_terms, float *__restrict__ part)
{
    extern __shared__ __align__(16) double r6_smem[];
    float *Ws = reinterpret_cast<float *>(r6_smem);
    float *S = Ws + kMlpFloatsSep;
    float *A1 = S + kPpoRowsSde * kPpoTS;
    float *sig2 = A1 + kPpoAccW1;
    const int tid = threadIdx.x, kq = tid & 7, jq = tid >> 3;
    for (int i = tid; i < kMlpFloatsSep; i += kThreads) Ws[i] = mlp_pack_element_sep(mlp, i);
    for (int i = tid; i < kPpoAccW1; i += kThreads) A1[i] = 0.0f;
    for (int c = tid; c < kSdeXi; c += kThreads) {
        const float sg = expf(log_std[c]);
        sig2[c] = sg * sg;
    }
    const int64_t nsamp = ro.T * ro.n;
    float aW0[14], aHd[6];                   // dW0 / dvf_w0 row tid, its bias; dW2[0..2][tid], dwv, db1, dvf_b1
    float aLs[3] = {0.0f, 0.0f, 0.0f};       // sum_s r_a h_p,tid^2 (threads 0..63)
    double aS = 0.0;
#pragma unroll
    for (int c = 0; c < 14; c++) aW0[c] = 0.0f;
#pragma unroll
    for (int c = 0; c < 6; c++) aHd[c] = 0.0f;
    __syncthreads();
    const int64_t tiles = (B + kThreads - 1) / kThreads;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        PpoHeadSde hd = {};
        {   // this thread's sample: forward and loss head
            const int64_t s = tile * kThreads + tid;
            const int64_t q = s < B ? idx[s] : -1;
            const bool ok = q >= 0 && q < nsamp;
            float x[kMlpIn], out[4];
            if (ok) {
                const int64_t t = q / ro.n, i = q - t * ro.n;
                const float *o = ro.obs + t * ro.obs_stride_step + i * ro.obs_stride_env;
#pragma unroll
                for (int c = 0; c < kMlpIn; c++) x[c] = o[c * ro.obs_stride_comp];
            } else {
#pragma unroll
                for (int c = 0; c < kMlpIn; c++) x[c] = 0.0f;
            }
#pragma unroll
            for (int c = 0; c < kMlpIn; c++) S[(kPpoRowX + c) * kPpoTS + tid] = x[c];
            ppo_forward_sep(Ws, x, S + kPpoRowH0 * kPpoTS + tid, S + kPpoRowHP * kPpoTS + tid, S + kPpoRowHV * kPpoTS + tid,
                            kPpoTS, out);
            if (ok) {
                const float a[3] = {ro.actions[3 * q], ro.actions[3 * q + 1], ro.actions[3 * q + 2]};
                float var[3];
                sde_latent_var(S + kPpoRowHP * kPpoTS + tid, kPpoTS, sig2, var);
                ppo_head_sde(out, a, ro.log_probs[q], ppo_advantage(ro.advantages[q], adv_stats), ro.returns[q], var, clip, vf,
                             ent, hd);
                if constexpr (kVfClip) ppo_value_clip(out[3], ro.old_values[q], ro.returns[q], vfc, vf, hd);
            }
#pragma unroll
            for (int r = 0; r < 7; r++) S[(kPpoRowG + r) * kPpoTS + tid] = hd.g[r];
            S[(kPpoRowG + 7) * kPpoTS + tid] = (s < B && !ok) ? 1.0f : 0.0f;
            S[(kPpoRowT + 0) * kPpoTS + tid] = hd.pg;
            S[(kPpoRowT + 1) * kPpoTS + tid] = hd.vloss;
            S[(kPpoRowT + 2) * kPpoTS + tid] = hd.clipped;
            S[(kPpoRowT + 3) * kPpoTS + tid] = hd.kl;
            S[kPpoRowE * kPpoTS + tid] = hd.ent;
        }
        __syncthreads();
        // heads from the latents (dW2 on h1p, dwv on h1v), log_std from h1p^2, and the scalar sums, before the latent rows
        // become deltas
        if (tid < kMlpH1) {
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                const F4 hp = ld4(S + (kPpoRowHP + tid) * kPpoTS + s4), hv = ld4(S + (kPpoRowHV + tid) * kPpoTS + s4);
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const F4 g = ld4(S + (kPpoRowG + c) * kPpoTS + s4);
                    const F4 h = c < 3 ? hp : hv;
                    float a = aHd[c];
                    a = __fmaf_rn(g.x, h.x, a); a = __fmaf_rn(g.y, h.y, a);
                    a = __fmaf_rn(g.z, h.z, a); a = __fmaf_rn(g.w, h.w, a);
                    aHd[c] = a;
                }
                const F4 hh = {hp.x * hp.x, hp.y * hp.y, hp.z * hp.z, hp.w * hp.w};
#pragma unroll
                for (int c = 0; c < 3; c++) {
                    const F4 r = ld4(S + (kPpoRowG + 4 + c) * kPpoTS + s4);
                    float a = aLs[c];
                    a = __fmaf_rn(r.x, hh.x, a); a = __fmaf_rn(r.y, hh.y, a);
                    a = __fmaf_rn(r.z, hh.z, a); a = __fmaf_rn(r.w, hh.w, a);
                    aLs[c] = a;
                }
            }
        } else if (tid < kMlpH1 + 13) {
            const float *row = S + (kPpoRowG + tid - kMlpH1) * kPpoTS;
#pragma unroll 4
            for (int s = 0; s < kThreads; s++) aS += (double)row[s];
        }
        __syncthreads();
        ppo_delta1_sep(Ws, hd, S + kPpoRowHP * kPpoTS + tid, S + kPpoRowHV * kPpoTS + tid, kPpoTS);
        __syncthreads();
        // dW1p / dW1v += delta1^T h0 (columns jq + 16 c: c < 4 policy units, c >= 4 value units), db1 / dvf_b1
#pragma unroll 1
        for (int r0 = 0; r0 < 8; r0 += 4) {
            float aW1[4][8];
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 8; c++) aW1[r][c] = A1[((r0 + r) * 8 + c) * kThreads + tid];
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                F4 h[8];
#pragma unroll
                for (int c = 0; c < 8; c++) h[c] = ld4(S + (kPpoRowH0 + jq + 16 * c) * kPpoTS + s4);
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const F4 dp = ld4(S + (kPpoRowHP + kq + 8 * (r0 + r)) * kPpoTS + s4);
                    const F4 dv = ld4(S + (kPpoRowHV + kq + 8 * (r0 + r)) * kPpoTS + s4);
#pragma unroll
                    for (int c = 0; c < 8; c++) {
                        const F4 d = c < 4 ? dp : dv;
                        float a = aW1[r][c];
                        a = __fmaf_rn(d.x, h[c].x, a); a = __fmaf_rn(d.y, h[c].y, a);
                        a = __fmaf_rn(d.z, h[c].z, a); a = __fmaf_rn(d.w, h[c].w, a);
                        aW1[r][c] = a;
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 8; c++) A1[((r0 + r) * 8 + c) * kThreads + tid] = aW1[r][c];
        }
        if (tid < kMlpH1) {
#pragma unroll 1
            for (int s4 = 0; s4 < kThreads; s4 += 4) {
                const F4 dp = ld4(S + (kPpoRowHP + tid) * kPpoTS + s4), dv = ld4(S + (kPpoRowHV + tid) * kPpoTS + s4);
                aHd[4] = (((aHd[4] + dp.x) + dp.y) + dp.z) + dp.w;
                aHd[5] = (((aHd[5] + dv.x) + dv.y) + dv.z) + dv.w;
            }
        }
        __syncthreads();
        {   // delta0 over h0, in place, each tower's units from its own delta1: this thread's column only
            float d1[kMlpH1];
#pragma unroll 1
            for (int t = 0; t < 2; t++) {
                const int row = t == 0 ? kPpoRowHP : kPpoRowHV;
#pragma unroll
                for (int k = 0; k < kMlpH1; k++) d1[k] = S[(row + k) * kPpoTS + tid];
#pragma unroll 1
                for (int j = t * kMlpH1; j < (t + 1) * kMlpH1; j++) {
                    float *p = S + (kPpoRowH0 + j) * kPpoTS + tid;
                    *p = ppo_delta0(Ws, j, d1, *p);
                }
            }
        }
        __syncthreads();
        // dW0[tid] += delta0_tid [x, 1]   (rows 0..63 the policy tower's w0, 64..127 the value tower's: stacked in P)
#pragma unroll 1
        for (int s4 = 0; s4 < kThreads; s4 += 4) {
            const F4 d = ld4(S + (kPpoRowH0 + tid) * kPpoTS + s4);
#pragma unroll
            for (int c = 0; c < kMlpIn; c++) {
                const F4 xv = ld4(S + (kPpoRowX + c) * kPpoTS + s4);
                float a = aW0[c];
                a = __fmaf_rn(d.x, xv.x, a); a = __fmaf_rn(d.y, xv.y, a);
                a = __fmaf_rn(d.z, xv.z, a); a = __fmaf_rn(d.w, xv.w, a);
                aW0[c] = a;
            }
            aW0[13] = (((aW0[13] + d.x) + d.y) + d.z) + d.w;
        }
        __syncthreads();
    }
    float *P = part + (int64_t)blockIdx.x * kPpoParamsSepSde;
#pragma unroll
    for (int r = 0; r < 8; r++)
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int k = kq + 8 * r, j = jq + 16 * c;
            P[(c < 4 ? kSepOffW1 + k * kMlpH1 + j : kSepOffVw1 + k * kMlpH1 + j - kMlpH1)] = A1[(r * 8 + c) * kThreads + tid];
        }
#pragma unroll
    for (int c = 0; c < kMlpIn; c++) P[kSepOffW0 + tid * kMlpIn + c] = aW0[c];
    P[kSepOffB0 + tid] = aW0[13];
    if (tid < kMlpH1) {
#pragma unroll
        for (int c = 0; c < 3; c++) P[kSepOffW2 + c * kMlpH1 + tid] = aHd[c];
        P[kSepOffWv + tid] = aHd[3];
        P[kSepOffB1 + tid] = aHd[4];
        P[kSepOffVb1 + tid] = aHd[5];
#pragma unroll
        for (int c = 0; c < 3; c++) P[kSepOffLogStd + 3 * tid + c] = aLs[c] * sig2[3 * tid + c];
    } else if (tid < kMlpH1 + 13) {
        const int r = tid - kMlpH1;          // rows: g0..g2 (db2), g3 (dbv), g4..g6 (r_a sums, unused), bad index, 4 loss
        double *T = part_terms + (int64_t)blockIdx.x * R6_PPO_NTERMS_SDE;   // terms, entropy
        if (r < 3) P[kSepOffB2 + r] = (float)aS;
        else if (r == 3) P[kSepOffBv] = (float)aS;
        else if (r == 7) T[R6_PPO_T_BAD_INDEX] = aS;
        else if (r >= 8 && r < 12) T[r - 8] = aS;
        else if (r == 12) T[R6_PPO_T_ENTROPY] = aS;
    }
}

// ppo_reduce_kernel over the separate-tower gSDE layout
__global__ void __launch_bounds__(256)
ppo_reduce_sep_sde_kernel(const double *__restrict__ part_terms, const float *__restrict__ part, int G, float *__restrict__ grad,
                          double *__restrict__ terms)
{
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p < kPpoParamsSepSde) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += (double)part[(int64_t)g * kPpoParamsSepSde + p];
        grad[p] = (float)s;
    }
    if (blockIdx.x == 0 && threadIdx.x < R6_PPO_NTERMS_SDE) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += part_terms[g * R6_PPO_NTERMS_SDE + threadIdx.x];
        terms[threadIdx.x] = s;
    }
}

// ppo_reduce_kernel over the separate-tower layout
__global__ void __launch_bounds__(256)
ppo_reduce_sep_kernel(const double *__restrict__ part_terms, const float *__restrict__ part, int G, float *__restrict__ grad,
                      double *__restrict__ terms)
{
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p < kPpoParamsSep) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += (double)part[(int64_t)g * kPpoParamsSep + p];
        grad[p] = (float)s;
    }
    if (blockIdx.x == 0 && threadIdx.x < R6_PPO_NTERMS) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += part_terms[g * R6_PPO_NTERMS + threadIdx.x];
        terms[threadIdx.x] = s;
    }
}

// grad[p] = sum of the CTA partials in CTA order (float64, rounded once); terms likewise
__global__ void __launch_bounds__(256)
ppo_reduce_kernel(const double *__restrict__ part_terms, const float *__restrict__ part, int G, float *__restrict__ grad,
                  double *__restrict__ terms)
{
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p < kPpoParams) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += (double)part[(int64_t)g * kPpoParams + p];
        grad[p] = (float)s;
    }
    if (blockIdx.x == 0 && threadIdx.x < R6_PPO_NTERMS) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += part_terms[g * R6_PPO_NTERMS + threadIdx.x];
        terms[threadIdx.x] = s;
    }
}

// ppo_reduce_kernel over the gSDE layout
__global__ void __launch_bounds__(256)
ppo_reduce_sde_kernel(const double *__restrict__ part_terms, const float *__restrict__ part, int G, float *__restrict__ grad,
                      double *__restrict__ terms)
{
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p < kPpoParamsSde) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += (double)part[(int64_t)g * kPpoParamsSde + p];
        grad[p] = (float)s;
    }
    if (blockIdx.x == 0 && threadIdx.x < R6_PPO_NTERMS_SDE) {
        double s = 0.0;
        for (int g = 0; g < G; g++) s += part_terms[g * R6_PPO_NTERMS_SDE + threadIdx.x];
        terms[threadIdx.x] = s;
    }
}


// r6_adam_step: one CTA (P is ~10^4).  The squared norm is summed in float64 in a fixed order (strided per thread,
// then a fixed warp-shuffle tree, then the 32 warp sums in order), so the step is deterministic.
constexpr int kAdamThreads = 1024;
struct AdamArgs {
    float scale, c[6];
    double max_norm;
};
__global__ void __launch_bounds__(kAdamThreads, 1)
adam_kernel(float *__restrict__ p, const float *__restrict__ gs, float *__restrict__ m, float *__restrict__ v, int P,
            const AdamArgs a, double *__restrict__ norm_out)
{
    __shared__ double red[kAdamThreads / 32];
    __shared__ float coef_s;
    double s = 0.0;
    for (int i = threadIdx.x; i < P; i += kAdamThreads) {
        const double g = (double)(a.scale * gs[i]);
        s = fma(g, g, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < kAdamThreads / 32; w++) t += red[w];
        const double norm = sqrt(t);
        coef_s = clip_coef(a.max_norm, norm);
        if (norm_out) *norm_out = norm;
    }
    __syncthreads();
    const float coef = coef_s;
    for (int i = threadIdx.x; i < P; i += kAdamThreads) {
        float pi = p[i], mi = m[i], vi = v[i];
        adam_element(pi, mi, vi, __fmul_rn(a.scale * gs[i], coef), a.c);
        p[i] = pi; m[i] = mi; v[i] = vi;
    }
}

// FMA-pipe micro-benchmark: 8 independent chains per thread
template <typename T>
__global__ void __launch_bounds__(256) peak_fma_kernel(int iters, double *sink)
{
    T a[8];
    const T m = (T)1.0000001, c = (T)1e-9;
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = (T)(threadIdx.x + k) * (T)1e-3;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = a[k] * m + c;
    }
    T s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k];
    if (s == (T)123.456) sink[0] = (double)s;
}

// kernels that keep the RK stages in dynamic shared memory need the > 48 KB opt-in once per process
template <class F>
int enable_smem(F kernel, int bytes = kSmemBytes)
{
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return fail(R6_ECUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return R6_OK;
}
template <class R, bool kExact>
int enable_density()
{
    constexpr int si = smem_int_bytes<R>();
    return enable_smem(step_kernel<R, kExact>, smem_bytes<R>()) | enable_smem(integrate_kernel<R, kExact>, si) |
           enable_smem(integrate_first_kernel<R, kExact>, si) | enable_smem(integrate_resume_kernel<R, kExact, false>, si) |
           enable_smem(integrate_resume_kernel<R, kExact, true>, si) |
           enable_smem(rollout_kernel<R, R6_ACT_PHILOX, kExact>, smem_bytes<R>()) |
           enable_smem(rollout_kernel<R, R6_ACT_BUFFER, kExact>, smem_bytes<R>()) |
           enable_smem(rollout_kernel<R, R6_ACT_MLP, kExact>, smem_mlp_bytes<R>());
}
template <class R>
int enable_all()
{
    return enable_density<R, false>() | enable_density<R, true>() | enable_smem(rollout_tc_kernel<R>, smem_tc_bytes<R>());
}
int ensure_attributes()
{
    static thread_local int device_done = -1;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return fail(R6_ECUDA, "cudaGetDevice failed%s");
    if (dev == device_done) return R6_OK;
    int rc = enable_all<double>() | enable_all<float>();
    rc |= enable_smem(policy_kernel<true>, kSmemPolicyTc);
    rc |= enable_smem(policy_kernel<false>, kSmemPolicy);
    rc |= enable_smem(policy_tc5_kernel<true>, tc5::kSmemBytes);
    rc |= enable_smem(policy_tc5_kernel<false>, tc5::kSmemBytes);
    rc |= enable_smem(ppo_grad_kernel<false>, kSmemPpo);
    rc |= enable_smem(ppo_grad_kernel<true>, kSmemPpo);
    rc |= enable_smem(ppo_grad_sde_kernel<false>, kSmemPpoSde);
    rc |= enable_smem(ppo_grad_sde_kernel<true>, kSmemPpoSde);
    rc |= enable_smem(policy_sde_kernel, kSmemPolicySde);
    rc |= enable_smem(policy_tc5_sde_kernel<true>, tc5::kSmemBytesSde);
    rc |= enable_smem(policy_tc5_sde_kernel<false>, tc5::kSmemBytesSde);
    rc |= enable_smem(policy_sep_kernel, kSmemPolicySep);
    rc |= enable_smem(policy_tc5_sep_kernel<true>, tc5::kSmemBytesSep);
    rc |= enable_smem(policy_tc5_sep_kernel<false>, tc5::kSmemBytesSep);
    rc |= enable_smem(ppo_grad_sep_kernel<false>, kSmemPpoSep);
    rc |= enable_smem(ppo_grad_sep_kernel<true>, kSmemPpoSep);
    rc |= enable_smem(policy_sep_sde_kernel, kSmemPolicySepSde);
    rc |= enable_smem(policy_tc5_sep_sde_kernel<true>, tc5::kSmemBytesSepSde);
    rc |= enable_smem(policy_tc5_sep_sde_kernel<false>, tc5::kSmemBytesSepSde);
    rc |= enable_smem(ppo_grad_sep_sde_kernel<false>, kSmemPpoSepSde);
    rc |= enable_smem(ppo_grad_sep_sde_kernel<true>, kSmemPpoSepSde);
    rc |= enable_smem(sim_raw_kernel<false>);
    rc |= enable_smem(sim_raw_kernel<true>);
    if (rc) return R6_ECUDA;
    device_done = dev;
    return R6_OK;
}

int64_t blocks_for(int64_t n) { return (n + kThreads - 1) / kThreads; }

int validate(const R6Params *p, const R6Buffers *b, int64_t n)
{
    if (!p || !b) return fail(R6_EINVAL, "null params/buffers%s");
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    if (p->precision != R6_PREC_F64 && p->precision != R6_PREC_F32) return fail(R6_EINVAL, "bad precision%s");
    if (!b->state || !b->m0 || !b->v0 || !b->step_count || !b->episode_id || !b->ep_return || !b->obs)
        return fail(R6_EINVAL, "a required state buffer is null%s");
    return R6_OK;
}
int validate_step(const R6Params *p, const R6Buffers *b, int64_t n)
{
    int rc = validate(p, b, n);
    if (rc) return rc;
    if ((!b->reward && !b->reward_f32) || !b->done || !b->flags || !b->terminal_obs || !b->terminal_state || !b->t_table)
        return fail(R6_EINVAL, "a required output buffer is null%s");
    if (p->n_t < 1) return fail(R6_EINVAL, "t_table is empty%s");
    return R6_OK;
}

// Programmatic dependent launch (the four kernels of a multi-pass step, back to back on one stream): the next kernel's
// CTAs may be set up while the previous kernel drains; every such kernel starts with griddepcontrol.wait, which returns
// once the previous grid has completed and its writes are visible (a no-op for an ordinary launch).
template <class... KArgs, class... Args>
void launch_pdl(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = R6_PDL;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// f(R(), std::bool_constant<kExact>()) with the density form dt needs: the series up to kMaxDtSeries, exact beyond
template <class R, class F>
auto dispatch_density(double dt, F &&f)
{
    return dt <= kMaxDtSeries ? f(R(), std::false_type()) : f(R(), std::true_type());
}
// ... and with R the working precision of p
template <class F>
auto dispatch(const R6Params *p, F &&f)
{
    return p->precision == R6_PREC_F32 ? dispatch_density<float>(p->dt, f) : dispatch_density<double>(p->dt, f);
}

int check_mlp(const R6Mlp *mlp)
{
    if (!mlp || !mlp->w0 || !mlp->b0 || !mlp->w1 || !mlp->b1 || !mlp->w2 || !mlp->b2)
        return fail(R6_EINVAL, "policy weights are null%s");
    const int vf = (mlp->vf_w0 != nullptr) + (mlp->vf_b0 != nullptr) + (mlp->vf_w1 != nullptr) + (mlp->vf_b1 != nullptr);
    if (vf != 0 && vf != 4) return fail(R6_EINVAL, "the value tower needs all of vf_w0, vf_b0, vf_w1, vf_b1 (or none)%s");
    return R6_OK;
}
// the entry points without a separate-tower kernel refuse such a network rather than run the shared trunk on it
int reject_separate(const R6Mlp *mlp, const char *what)
{
    if (mlp && mlp_separate(*mlp))
        return fail(R6_EINVAL, "%s does not support the separate policy / value towers (R6Mlp.vf_w0 set)", what);
    return R6_OK;
}

template <class R, bool kExact>
void launch_step(const R6Params *p, const R6Buffers *b, const Derived &dv, int64_t n, int64_t env_offset,
                 const float *actions, uint64_t seed, cudaStream_t s, int64_t step_index = 0, int64_t first = 0,
                 int64_t count = -1, int lane = 0)
{
    if (b->scratch == nullptr) {
        step_kernel<R, kExact><<<(unsigned)blocks_for(n), kThreads, smem_bytes<R>(), s>>>(*p, *b, dv, n, env_offset, actions, seed);
        return;
    }
    // kernel pair over the env sub-range [first, first + count)
    if (count < 0) count = n;
    const int64_t last = first + count;
    const unsigned gi = (unsigned)((count + kIntThreads - 1) / kIntThreads);
    constexpr int si = smem_int_bytes<R>();
    if (b->work != nullptr) {                    // integrator cut at attempt boundaries (see integrate_first_kernel)
        // list 0 holds ~2/3 of the range, list 1 ~1 %; the resume kernels walk longer lists with a grid stride
        const unsigned g1 = gi - gi / 4, g2 = gi / 16 + 1;
        launch_pdl(integrate_first_kernel<R, kExact>, gi, kIntThreads, si, s, *p, *b, n, actions, env_offset, seed, step_index, first, last, lane);
        launch_pdl(integrate_resume_kernel<R, kExact, false>, g1, kIntThreads, si, s, *p, *b, n, actions, env_offset, seed, step_index, first, lane);
        launch_pdl(integrate_resume_kernel<R, kExact, true>, g2, kIntThreads, si, s, *p, *b, n, actions, env_offset, seed, step_index, first, lane);
    } else
        launch_pdl(integrate_kernel<R, kExact>, gi, kIntThreads, si, s, *p, *b, n, actions, env_offset, seed, step_index, first, last);
    launch_pdl(post_kernel<R>, (unsigned)((count + kPostThreads - 1) / kPostThreads), kPostThreads, 0, s, *p, *b, dv, n, env_offset, actions, seed, step_index, first, last, lane);
}

template <class R, bool kExact>
int launch_rollout(const R6Params *p, const R6Buffers *b, const Derived &dv, int64_t n, int64_t env_offset, int32_t k,
                   int32_t mode, const R6Mlp *mlp, const float *act_buf, uint64_t seed, int64_t step_base, const Traj &tr,
                   cudaStream_t s)
{
    const unsigned g = (unsigned)blocks_for(n);
    if (mode == R6_ACT_PHILOX)
        rollout_kernel<R, R6_ACT_PHILOX, kExact><<<g, kThreads, smem_bytes<R>(), s>>>(*p, *b, dv, n, env_offset, k, nullptr, R6Mlp{}, seed,
                                                                                     step_base, tr.obs, tr.act, tr.rew, tr.done);
    else if (mode == R6_ACT_BUFFER) {
        if (!act_buf) return fail(R6_EINVAL, "act_buf is null%s");
        rollout_kernel<R, R6_ACT_BUFFER, kExact><<<g, kThreads, smem_bytes<R>(), s>>>(*p, *b, dv, n, env_offset, k, act_buf, R6Mlp{}, seed,
                                                                                     step_base, tr.obs, tr.act, tr.rew, tr.done);
    } else if (mode == R6_ACT_MLP || mode == R6_ACT_MLP_TC) {
        if (int rc = check_mlp(mlp)) return rc;
        // rollout_tc_kernel has the series density only: at dt > kMaxDtSeries the float32 network runs instead
        if (mode == R6_ACT_MLP_TC && !kExact)
            rollout_tc_kernel<R><<<g, kThreads, smem_tc_bytes<R>(), s>>>(*p, *b, dv, n, env_offset, k, *mlp, seed, tr.obs, tr.act,
                                                                       tr.rew, tr.done);
        else
            rollout_kernel<R, R6_ACT_MLP, kExact><<<g, kThreads, smem_mlp_bytes<R>(), s>>>(*p, *b, dv, n, env_offset, k, nullptr, *mlp, seed,
                                                                                         step_base, tr.obs, tr.act, tr.rew, tr.done);
    } else
        return fail(R6_EINVAL, "unsupported action mode%s");
    return R6_OK;
}

}  // namespace

extern "C" {

int r6_abi_version(void) { return R6_ABI_VERSION; }
const char *r6_last_error(void) { return g_err; }
int r6_params_size(void) { return (int)sizeof(R6Params); }
int r6_buffers_size(void) { return (int)sizeof(R6Buffers); }

int r6_reset(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset, const uint8_t *mask, uint64_t seed,
             void *stream)
{
    int rc = validate(p, b, n);
    if (rc) return rc;
    if (n == 0) return R6_OK;
    const Derived dv = make_derived(*p);
    if (p->precision == R6_PREC_F32)
        reset_kernel<float><<<(unsigned)blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(*p, *b, dv, n, env_offset, mask, seed);
    else
        reset_kernel<double><<<(unsigned)blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(*p, *b, dv, n, env_offset, mask, seed);
    return check_launch("r6_reset");
}

int r6_step(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset, const float *actions, uint64_t seed,
            void *stream)
{
    int rc = validate_step(p, b, n);
    if (rc) return rc;
    if (!actions) return fail(R6_EINVAL, "actions is null%s");
    if (n == 0) return R6_OK;
    if ((rc = ensure_attributes())) return rc;
    const Derived dv = make_derived(*p);
    dispatch(p, [&](auto r, auto exact) { launch_step<decltype(r), exact>(p, b, dv, n, env_offset, actions, seed, (cudaStream_t)stream); });
    return check_launch("r6_step");
}

int r6_step_random(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset, uint64_t seed, int64_t step_index,
                   void *stream)
{
    int rc = validate_step(p, b, n);
    if (rc) return rc;
    if (!b->scratch) return fail(R6_EINVAL, "r6_step_random needs R6Buffers.scratch%s");
    if (n == 0) return R6_OK;
    if ((rc = ensure_attributes())) return rc;
    const Derived dv = make_derived(*p);
    dispatch(p, [&](auto r, auto exact) {
        launch_step<decltype(r), exact>(p, b, dv, n, env_offset, nullptr, seed, (cudaStream_t)stream, step_index);
    });
    return check_launch("r6_step_random");
}

int64_t r6_work_bytes(int64_t n) { return n < 0 ? 0 : 256 + 80 * n; }

int r6_step_range(const R6Params *p, const R6Buffers *b, int64_t n, int64_t first, int64_t count, int32_t lane,
                  int64_t env_offset, const float *actions, uint64_t seed, int64_t step_index, void *stream)
{
    int rc = validate_step(p, b, n);
    if (rc) return rc;
    if (!b->scratch) return fail(R6_EINVAL, "r6_step_range needs R6Buffers.scratch%s");
    if (first < 0 || count < 0 || first + count > n) return fail(R6_EINVAL, "env sub-range outside [0, n)%s");
    if (lane < 0 || lane >= R6_MAX_LANES) return fail(R6_EINVAL, "lane outside [0, R6_MAX_LANES)%s");
    if (count == 0) return R6_OK;
    if ((rc = ensure_attributes())) return rc;
    const Derived dv = make_derived(*p);
    dispatch(p, [&](auto r, auto exact) {
        launch_step<decltype(r), exact>(p, b, dv, n, env_offset, actions, seed, (cudaStream_t)stream, step_index, first, count, lane);
    });
    return check_launch("r6_step_range");
}

int r6_rollout(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset, int32_t k, int32_t mode,
               const R6Mlp *mlp, const float *act_buf, uint64_t seed, int64_t step_base, float *traj_obs,
               float *traj_act, float *traj_rew, uint8_t *traj_done, void *stream)
{
    if (mode == R6_ACT_MLP || mode == R6_ACT_MLP_TC)
        if (int rc = reject_separate(mlp, "r6_rollout with R6_ACT_MLP / R6_ACT_MLP_TC")) return rc;
    int rc = validate_step(p, b, n);
    if (rc) return rc;
    if (k < 0) return fail(R6_EINVAL, "k < 0%s");
    if (n == 0 || k == 0) return R6_OK;
    if ((rc = ensure_attributes())) return rc;
    const Derived dv = make_derived(*p);
    const Traj tr = {traj_obs, traj_act, traj_rew, traj_done};
    rc = dispatch(p, [&](auto r, auto exact) {
        return launch_rollout<decltype(r), exact>(p, b, dv, n, env_offset, k, mode, mlp, act_buf, seed, step_base, tr,
                                                  (cudaStream_t)stream);
    });
    if (rc) return rc;
    return check_launch("r6_rollout");
}

int r6_sim_step_raw(double *state, const double *u, const double *m0, const double *t, double dt, int64_t n,
                    int8_t *status, uint8_t *nattempts, void *stream)
{
    if (!state || !u || !m0 || !t || !status) return fail(R6_EINVAL, "null pointer%s");
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    if (n == 0) return R6_OK;
    int rc = ensure_attributes();
    if (rc) return rc;
    dispatch_density<double>(dt, [&](double, auto exact) {
        sim_raw_kernel<exact><<<(unsigned)blocks_for(n), kThreads, kSmemBytes, (cudaStream_t)stream>>>(state, u, m0, t, dt, n, status,
                                                                                                      nattempts);
    });
    return check_launch("r6_sim_step_raw");
}

int r6_tgo(const double *c2, const double *c3, const double *c4, double c0, int64_t n, const double *guess, double *tgo,
           void *stream)
{
    if (!c2 || !c3 || !c4 || !tgo) return fail(R6_EINVAL, "null pointer%s");
    if (n <= 0) return n == 0 ? R6_OK : fail(R6_EINVAL, "n < 0%s");
    tgo_kernel<<<(unsigned)blocks_for(n), kThreads, 0, (cudaStream_t)stream>>>(c2, c3, c4, c0, n, guess, tgo);
    return check_launch("r6_tgo");
}

int r6_policy_range(const R6Mlp *mlp, const float *obs, int64_t n, int64_t first, int64_t count, int32_t tensor_cores,
                    int32_t stochastic, uint64_t seed, int64_t env_offset, int64_t step_index, float *actions,
                    float *actions_raw, float *values, float *log_prob, void *stream)
{
    if (int rc = check_mlp(mlp)) return rc;
    if (!obs || !actions) return fail(R6_EINVAL, "null pointer%s");
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    if (first < 0 || count < 0 || first + count > n) return fail(R6_EINVAL, "env sub-range outside [0, n)%s");
    if (tensor_cores < 0 || tensor_cores > 3) return fail(R6_EINVAL, "tensor_cores must be 0, 1, 2 or 3%s");
    const bool sep = mlp_separate(*mlp);
    if (sep && tensor_cores == 1) return reject_separate(mlp, "r6_policy with tensor_cores = 1 (mma.sync)");
    if (sep && tensor_cores >= 2 && (reinterpret_cast<uintptr_t>(mlp->vf_w1) & 15u) != 0)
        return fail(R6_EINVAL, "tensor_cores = 2 / 3 need vf_w1 16-byte aligned%s");
    if (count == 0) return R6_OK;
    int rc = ensure_attributes();
    if (rc) return rc;
    // one resident wave: SM count x resident CTAs per SM
    static thread_local int sm_count = 0;
    if (sm_count == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count <= 0) sm_count = 148;
    }
    const PolicyOut po = {actions, actions_raw, values, log_prob, stochastic, seed, env_offset, step_index, first, first + count};
    const int64_t wave = (int64_t)sm_count * (tensor_cores ? 3 : 4);
    const unsigned g = (unsigned)(blocks_for(count) < wave ? blocks_for(count) : wave);
    if (tensor_cores >= 2) {
        if ((reinterpret_cast<uintptr_t>(mlp->w1) & 15u) != 0) return fail(R6_EINVAL, "tensor_cores = 2 / 3 need w1 16-byte aligned%s");
        const int64_t pairs = (blocks_for(count) + 1) / 2;                 // one CTA per SM, two tile groups per CTA
        const unsigned g5 = (unsigned)(pairs < sm_count ? pairs : sm_count);
        if (sep && tensor_cores == 3) launch_pdl(policy_tc5_sep_kernel<true>, g5, tc5::kThreads, tc5::kSmemBytesSep, (cudaStream_t)stream, *mlp, obs, n, po);
        else if (sep) launch_pdl(policy_tc5_sep_kernel<false>, g5, tc5::kThreads, tc5::kSmemBytesSep, (cudaStream_t)stream, *mlp, obs, n, po);
        else if (tensor_cores == 3) launch_pdl(policy_tc5_kernel<true>, g5, tc5::kThreads, tc5::kSmemBytes, (cudaStream_t)stream, *mlp, obs, n, po);
        else launch_pdl(policy_tc5_kernel<false>, g5, tc5::kThreads, tc5::kSmemBytes, (cudaStream_t)stream, *mlp, obs, n, po);
    }
    else if (sep) policy_sep_kernel<<<g, kThreads, kSmemPolicySep, (cudaStream_t)stream>>>(*mlp, obs, n, po);
    else if (tensor_cores) policy_kernel<true><<<g, kThreads, kSmemPolicyTc, (cudaStream_t)stream>>>(*mlp, obs, n, po);
    else policy_kernel<false><<<g, kThreads, kSmemPolicy, (cudaStream_t)stream>>>(*mlp, obs, n, po);
    return check_launch("r6_policy");
}

int r6_sde_size(void) { return (int)sizeof(R6Sde); }

int r6_sde_noise(int64_t n, int64_t first, int64_t count, uint64_t seed, int64_t env_offset, int64_t step_index, float *xi,
                 void *stream)
{
    if (!xi) return fail(R6_EINVAL, "null pointer%s");
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    if (first < 0 || count < 0 || first + count > n) return fail(R6_EINVAL, "env sub-range outside [0, n)%s");
    if (count == 0) return R6_OK;
    sde_noise_kernel<<<dim3((unsigned)((count + 255) / 256), kSdeBlocks), 256, 0, (cudaStream_t)stream>>>(
        seed, env_offset, step_index, n, first, first + count, xi);
    return check_launch("r6_sde_noise");
}

int r6_policy_sde_range(const R6Mlp *mlp, const R6Sde *sde, const float *obs, int64_t n, int64_t first, int64_t count,
                        int32_t tensor_cores, int32_t stochastic, float *actions, float *actions_raw, float *values,
                        float *log_prob, void *stream)
{
    if (int rc = check_mlp(mlp)) return rc;
    if (int rc = reject_separate(mlp, "r6_policy_sde_range (gSDE; r6_policy_sde_sep_range runs the separate towers)")) return rc;
    if (!sde || !sde->log_std || !sde->xi || !obs || !actions) return fail(R6_EINVAL, "null pointer%s");
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    if (first < 0 || count < 0 || first + count > n) return fail(R6_EINVAL, "env sub-range outside [0, n)%s");
    if (tensor_cores == 1) return fail(R6_EINVAL, "gSDE has no mma.sync policy kernel (tensor_cores = 1): use 0, 2 or 3%s");
    if (tensor_cores < 0 || tensor_cores > 3) return fail(R6_EINVAL, "tensor_cores must be 0, 2 or 3%s");
    if (count == 0) return R6_OK;
    int rc = ensure_attributes();
    if (rc) return rc;
    int dev = 0, sm_count = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count <= 0) sm_count = 148;
    const PolicyOut po = {actions, actions_raw, values, log_prob, stochastic, 0, 0, 0, first, first + count};
    const SdeIn si = {sde->log_std, sde->xi};
    cudaStream_t s = (cudaStream_t)stream;
    if (tensor_cores >= 2) {
        if ((reinterpret_cast<uintptr_t>(mlp->w1) & 15u) != 0) return fail(R6_EINVAL, "tensor_cores = 2 / 3 need w1 16-byte aligned%s");
        const int64_t pairs = (blocks_for(count) + 1) / 2;
        const unsigned g5 = (unsigned)(pairs < sm_count ? pairs : sm_count);
        if (tensor_cores == 3) launch_pdl(policy_tc5_sde_kernel<true>, g5, tc5::kThreads, tc5::kSmemBytesSde, s, *mlp, si, obs, n, po);
        else launch_pdl(policy_tc5_sde_kernel<false>, g5, tc5::kThreads, tc5::kSmemBytesSde, s, *mlp, si, obs, n, po);
    } else {
        const int64_t wave = (int64_t)sm_count * 4;
        const unsigned g = (unsigned)(blocks_for(count) < wave ? blocks_for(count) : wave);
        policy_sde_kernel<<<g, kThreads, kSmemPolicySde, s>>>(*mlp, si, obs, n, po);
    }
    return check_launch("r6_policy_sde_range");
}

int r6_policy_sde_sep_range(const R6Mlp *mlp, const R6Sde *sde, const float *obs, int64_t n, int64_t first, int64_t count,
                            int32_t tensor_cores, int32_t stochastic, float *actions, float *actions_raw, float *values,
                            float *log_prob, void *stream)
{
    if (int rc = check_mlp(mlp)) return rc;
    if (!mlp_separate(*mlp))
        return fail(R6_EINVAL, "r6_policy_sde_sep_range needs the separate towers (R6Mlp.vf_w0 set): the shared trunk's gSDE "
                               "policy is r6_policy_sde_range%s");
    if (!sde || !sde->log_std || !sde->xi || !obs || !actions) return fail(R6_EINVAL, "null pointer%s");
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    if (first < 0 || count < 0 || first + count > n) return fail(R6_EINVAL, "env sub-range outside [0, n)%s");
    if (tensor_cores == 1) return fail(R6_EINVAL, "gSDE has no mma.sync policy kernel (tensor_cores = 1): use 0, 2 or 3%s");
    if (tensor_cores < 0 || tensor_cores > 3) return fail(R6_EINVAL, "tensor_cores must be 0, 2 or 3%s");
    if (tensor_cores >= 2 && ((reinterpret_cast<uintptr_t>(mlp->w1) | reinterpret_cast<uintptr_t>(mlp->vf_w1)) & 15u) != 0)
        return fail(R6_EINVAL, "tensor_cores = 2 / 3 need w1 and vf_w1 16-byte aligned%s");
    if (count == 0) return R6_OK;
    int rc = ensure_attributes();
    if (rc) return rc;
    int dev = 0, sm_count = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count <= 0) sm_count = 148;
    const PolicyOut po = {actions, actions_raw, values, log_prob, stochastic, 0, 0, 0, first, first + count};
    const SdeIn si = {sde->log_std, sde->xi};
    cudaStream_t s = (cudaStream_t)stream;
    if (tensor_cores >= 2) {
        const int64_t pairs = (blocks_for(count) + 1) / 2;
        const unsigned g5 = (unsigned)(pairs < sm_count ? pairs : sm_count);
        if (tensor_cores == 3) launch_pdl(policy_tc5_sep_sde_kernel<true>, g5, tc5::kThreads, tc5::kSmemBytesSepSde, s, *mlp, si, obs, n, po);
        else launch_pdl(policy_tc5_sep_sde_kernel<false>, g5, tc5::kThreads, tc5::kSmemBytesSepSde, s, *mlp, si, obs, n, po);
    } else {
        const int64_t wave = (int64_t)sm_count * 4;
        const unsigned g = (unsigned)(blocks_for(count) < wave ? blocks_for(count) : wave);
        policy_sep_sde_kernel<<<g, kThreads, kSmemPolicySepSde, s>>>(*mlp, si, obs, n, po);
    }
    return check_launch("r6_policy_sde_sep_range");
}

int r6_policy_ex(const R6Mlp *mlp, const float *obs, int64_t n, int32_t tensor_cores, int32_t stochastic, uint64_t seed,
                 int64_t env_offset, int64_t step_index, float *actions, float *actions_raw, float *values,
                 float *log_prob, void *stream)
{
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    return r6_policy_range(mlp, obs, n, 0, n, tensor_cores, stochastic, seed, env_offset, step_index, actions, actions_raw,
                           values, log_prob, stream);
}

int r6_policy(const R6Mlp *mlp, const float *obs, int64_t n, int32_t tensor_cores, float *actions, void *stream)
{
    return r6_policy_ex(mlp, obs, n, tensor_cores, 0, 0, 0, 0, actions, nullptr, nullptr, nullptr, stream);
}

int r6_gae(const float *rew, const float *values, const uint8_t *done, const float *last_values, int32_t T, int64_t n,
           double gamma, double gae_lambda, float *adv, float *ret, void *stream)
{
    if (!rew || !values || !done || !last_values || !adv || !ret) return fail(R6_EINVAL, "null pointer%s");
    if (T < 0 || n < 0) return fail(R6_EINVAL, "negative size%s");
    if (T == 0 || n == 0) return R6_OK;
    gae_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rew, values, done, last_values, T, n, (float)gamma,
                                                                          (float)(gamma * gae_lambda), adv, ret);
    return check_launch("r6_gae");
}

int r6_trunc_record(const uint8_t *flags, const float *terminal_obs, int64_t n, int64_t first, int64_t count, int32_t step,
                    int32_t slots, int32_t *slot_step, float *slot_obs, void *stream)
{
    if (!flags || !terminal_obs || !slot_step || !slot_obs) return fail(R6_EINVAL, "null pointer%s");
    if (n < 0) return fail(R6_EINVAL, "n < 0%s");
    if (first < 0 || count < 0 || first + count > n) return fail(R6_EINVAL, "env sub-range outside [0, n)%s");
    if (step < 0 || slots < 0) return fail(R6_EINVAL, "step and slots must be >= 0%s");
    if (count == 0 || slots == 0) return R6_OK;
    launch_pdl(trunc_record_kernel, (unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream, flags, terminal_obs, n, first,
               first + count, step, slots, slot_step, slot_obs);
    return check_launch("r6_trunc_record");
}

int r6_trunc_bootstrap(float *rew, int32_t T, int64_t n, int32_t slots, const int32_t *slot_step, const float *slot_values,
                       double gamma, void *stream)
{
    if (!rew || !slot_step || !slot_values) return fail(R6_EINVAL, "null pointer%s");
    if (T < 0 || n < 0 || slots < 0) return fail(R6_EINVAL, "negative size%s");
    if (T == 0 || n == 0 || slots == 0) return R6_OK;
    trunc_bootstrap_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rew, T, n, slots, slot_step, slot_values,
                                                                                       (float)gamma);
    return check_launch("r6_trunc_bootstrap");
}

int r6_ppo_rollout_size(void) { return (int)sizeof(R6PpoRollout); }
int r6_ppo_coef_size(void) { return (int)sizeof(R6PpoCoef); }
int r6_adam_coef_size(void) { return (int)sizeof(R6AdamCoef); }

int64_t r6_ppo_work_bytes(int64_t B)
{
    return B > 0 ? ppo_ctas(B) * (int64_t)(R6_PPO_NTERMS * sizeof(double) + kPpoParamsSep * sizeof(float)) : 0;
}

}  // extern "C"

namespace {
// r6_ppo_grad / r6_ppo_grad_sde / r6_ppo_grad_sde_sep (kSde: sde_log_std != NULL; the layout follows the mlp): the
// gradient kernel, then the reduction of its CTA partials
template <bool kSde>
int ppo_grad_launch(const R6Mlp *mlp, const float *sde_log_std, const R6PpoRollout *rollout, const int64_t *idx, int64_t B,
                    const R6PpoCoef *coef, float *grad_sum, double *terms, void *work, void *stream)
{
    const bool sep = mlp_separate(*mlp);
    const int kP = kSde ? (sep ? kPpoParamsSepSde : kPpoParamsSde) : (sep ? kPpoParamsSep : kPpoParams);
    constexpr int kNT = kSde ? R6_PPO_NTERMS_SDE : R6_PPO_NTERMS;
    if (!rollout || !rollout->obs || !rollout->actions || !rollout->log_probs || !rollout->advantages || !rollout->returns)
        return fail(R6_EINVAL, "null rollout buffer%s");
    if (rollout->T < 0 || rollout->n < 0 || B < 0) return fail(R6_EINVAL, "negative size%s");
    if (!coef || !grad_sum || !terms || (B > 0 && (!idx || !work))) return fail(R6_EINVAL, "null pointer%s");
    if (!(coef->clip_range_vf >= 0.0) || !isfinite(coef->clip_range_vf))
        return fail(R6_EINVAL, "clip_range_vf must be finite and >= 0 (0 = no value clipping)%s");
    const bool vclip = coef->clip_range_vf > 0.0;
    if (vclip && B > 0 && !rollout->old_values) return fail(R6_EINVAL, "clip_range_vf > 0 needs rollout->old_values%s");
    cudaStream_t s = (cudaStream_t)stream;
    if (B == 0) {
        cudaError_t e = cudaMemsetAsync(grad_sum, 0, sizeof(float) * kP, s);
        if (e == cudaSuccess) e = cudaMemsetAsync(terms, 0, sizeof(double) * kNT, s);
        if (e != cudaSuccess) return fail(R6_ECUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
        return R6_OK;
    }
    int rc = ensure_attributes();
    if (rc) return rc;
    const int G = (int)ppo_ctas(B);
    double *pt = static_cast<double *>(work);
    float *pp = reinterpret_cast<float *>(pt + (int64_t)G * kNT);
    const float clip = (float)coef->clip_range, vf = (float)coef->vf_coef, ent = (float)coef->ent_coef;
    const float vfc = (float)coef->clip_range_vf;
    if constexpr (kSde) {
        if (sep) {
            if (vclip)
                ppo_grad_sep_sde_kernel<true><<<G, kThreads, kSmemPpoSepSde, s>>>(*mlp, sde_log_std, *rollout, idx, B, clip, vf, ent,
                                                                                 vfc, coef->adv_stats, pt, pp);
            else
                ppo_grad_sep_sde_kernel<false><<<G, kThreads, kSmemPpoSepSde, s>>>(*mlp, sde_log_std, *rollout, idx, B, clip, vf,
                                                                                  ent, vfc, coef->adv_stats, pt, pp);
            rc = check_launch("r6_ppo_grad_sde_sep");
            if (rc) return rc;
            ppo_reduce_sep_sde_kernel<<<(kP + 255) / 256, 256, 0, s>>>(pt, pp, G, grad_sum, terms);
            return check_launch("r6_ppo_grad_sde_sep (reduce)");
        }
        if (vclip)
            ppo_grad_sde_kernel<true><<<G, kThreads, kSmemPpoSde, s>>>(*mlp, sde_log_std, *rollout, idx, B, clip, vf, ent, vfc,
                                                                      coef->adv_stats, pt, pp);
        else
            ppo_grad_sde_kernel<false><<<G, kThreads, kSmemPpoSde, s>>>(*mlp, sde_log_std, *rollout, idx, B, clip, vf, ent, vfc,
                                                                       coef->adv_stats, pt, pp);
        rc = check_launch("r6_ppo_grad_sde");
        if (rc) return rc;
        ppo_reduce_sde_kernel<<<(kP + 255) / 256, 256, 0, s>>>(pt, pp, G, grad_sum, terms);
        return check_launch("r6_ppo_grad_sde (reduce)");
    } else if (sep) {
        if (vclip)
            ppo_grad_sep_kernel<true><<<G, kThreads, kSmemPpoSep, s>>>(*mlp, *rollout, idx, B, clip, vf, ent, vfc, coef->adv_stats,
                                                                      pt, pp);
        else
            ppo_grad_sep_kernel<false><<<G, kThreads, kSmemPpoSep, s>>>(*mlp, *rollout, idx, B, clip, vf, ent, vfc, coef->adv_stats,
                                                                       pt, pp);
        rc = check_launch("r6_ppo_grad (separate towers)");
        if (rc) return rc;
        ppo_reduce_sep_kernel<<<(kP + 255) / 256, 256, 0, s>>>(pt, pp, G, grad_sum, terms);
        return check_launch("r6_ppo_grad (separate towers, reduce)");
    } else {
        if (vclip)
            ppo_grad_kernel<true><<<G, kThreads, kSmemPpo, s>>>(*mlp, *rollout, idx, B, clip, vf, ent, vfc, coef->adv_stats, pt, pp);
        else
            ppo_grad_kernel<false><<<G, kThreads, kSmemPpo, s>>>(*mlp, *rollout, idx, B, clip, vf, ent, vfc, coef->adv_stats, pt, pp);
        rc = check_launch("r6_ppo_grad");
        if (rc) return rc;
        ppo_reduce_kernel<<<(kP + 255) / 256, 256, 0, s>>>(pt, pp, G, grad_sum, terms);
        return check_launch("r6_ppo_grad (reduce)");
    }
}
}  // namespace

extern "C" {

int r6_ppo_grad(const R6Mlp *mlp, const R6PpoRollout *rollout, const int64_t *idx, int64_t B, const R6PpoCoef *coef,
                float *grad_sum, double *terms, void *work, void *stream)
{
    if (int rc = check_mlp(mlp)) return rc;
    if (!mlp->wv || !mlp->bv || !mlp->log_std) return fail(R6_EINVAL, "r6_ppo_grad needs the critic head and log_std%s");
    return ppo_grad_launch<false>(mlp, nullptr, rollout, idx, B, coef, grad_sum, terms, work, stream);
}

int64_t r6_ppo_sde_work_bytes(int64_t B)
{
    // both gSDE layouts (shared trunk and separate towers): sized for the larger
    static_assert(kPpoParamsSepSde >= kPpoParamsSde, "gSDE work buffer");
    return B > 0 ? ppo_ctas(B) * (int64_t)(R6_PPO_NTERMS_SDE * sizeof(double) + kPpoParamsSepSde * sizeof(float)) : 0;
}

int r6_ppo_grad_sde(const R6Mlp *mlp, const R6Sde *sde, const R6PpoRollout *rollout, const int64_t *idx, int64_t B,
                    const R6PpoCoef *coef, float *grad_sum, double *terms, void *work, void *stream)
{
    if (int rc = check_mlp(mlp)) return rc;
    if (int rc = reject_separate(mlp, "r6_ppo_grad_sde (gSDE; r6_ppo_grad_sde_sep trains the separate towers)")) return rc;
    if (!mlp->wv || !mlp->bv || !sde || !sde->log_std) return fail(R6_EINVAL, "r6_ppo_grad_sde needs the critic head and log_std%s");
    return ppo_grad_launch<true>(mlp, sde->log_std, rollout, idx, B, coef, grad_sum, terms, work, stream);
}

int r6_ppo_grad_sde_sep(const R6Mlp *mlp, const R6Sde *sde, const R6PpoRollout *rollout, const int64_t *idx, int64_t B,
                        const R6PpoCoef *coef, float *grad_sum, double *terms, void *work, void *stream)
{
    if (int rc = check_mlp(mlp)) return rc;
    if (!mlp_separate(*mlp))
        return fail(R6_EINVAL, "r6_ppo_grad_sde_sep needs the separate towers (R6Mlp.vf_w0 set): the shared trunk's gSDE "
                               "gradient is r6_ppo_grad_sde%s");
    if (!mlp->wv || !mlp->bv || !sde || !sde->log_std)
        return fail(R6_EINVAL, "r6_ppo_grad_sde_sep needs the critic head and log_std%s");
    return ppo_grad_launch<true>(mlp, sde->log_std, rollout, idx, B, coef, grad_sum, terms, work, stream);
}

int r6_adam_step(float *params, const float *grad_sum, float *m, float *v, int64_t P, const R6AdamCoef *coef,
                 int64_t step, double *grad_norm_out, void *stream)
{
    if (!params || !grad_sum || !m || !v || !coef) return fail(R6_EINVAL, "null pointer%s");
    if (P < 0 || P > (int64_t)1 << 30) return fail(R6_EINVAL, "P out of range%s");
    if (step < 1) return fail(R6_EINVAL, "step must be >= 1%s");
    if (P == 0) return R6_OK;
    AdamArgs a;
    a.scale = (float)coef->scale;
    a.max_norm = coef->max_grad_norm;
    adam_coefs(*coef, step, a.c);
    adam_kernel<<<1, kAdamThreads, 0, (cudaStream_t)stream>>>(params, grad_sum, m, v, (int)P, a, grad_norm_out);
    return check_launch("r6_adam_step");
}

int r6_stats_reset(double *stats, void *stream)
{
    if (!stats) return fail(R6_EINVAL, "null pointer%s");
    cudaError_t e = cudaMemsetAsync(stats, 0, sizeof(double) * R6_NSTATS, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(R6_ECUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
    return R6_OK;
}

int r6_peak_fma(int32_t fp64, int64_t blocks, int32_t iters, double *sink, void *stream)
{
    if (!sink || blocks <= 0 || iters <= 0) return fail(R6_EINVAL, "bad argument%s");
    if (fp64) peak_fma_kernel<double><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    else peak_fma_kernel<float><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(iters, sink);
    return check_launch("r6_peak_fma");
}

}  // extern "C"
