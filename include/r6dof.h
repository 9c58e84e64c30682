/*
 * r6dof.h — C ABI of libr6dof.so: the B200 (sm_100a) batched 6DOF rocket-landing env step.
 *
 * The reference (Tuxliri/RL_Rocket_6DOF) is pure Python and has no FFI seam; the boundary it
 * offers is the gym API of `Rocket6DOF` (my_environment/envs/rocket_env.py:16-231) and, one level
 * up, the stable-baselines3 VecEnv protocol that SB3 wraps around it (main_6DOF.py:105-114,
 * montecarlo_script.py:54-64).  This header is what a ctypes binding of those two call sites
 * binds (see INTEGRATION.md): every entry point names the reference interface it replaces.
 *
 * Conventions
 *  - plain C: pointers + sizes, no torch / C++ types.  Every buffer pointer is DEVICE memory owned
 *    by the caller (a torch CUDA tensor's data_ptr()); the library allocates nothing and keeps
 *    no global state except a thread-local error string.  The per-step OUTPUT arrays (obs, reward,
 *    reward_f32, done, flags) and `actions` may instead point at pinned, device-mapped HOST memory
 *    (cudaHostAlloc / torch pin_memory): the kernel then streams them over PCIe itself, overlapped
 *    with the computation, and no separate copy is needed (Rocket6DOFVecEnv.step_host).
 *  - every call enqueues work on the caller's stream (`cudaStream_t` passed as void*) and returns
 *    without synchronising; results are valid after the stream is synchronised.
 *  - return value: 0 on success, negative R6_E* on error; r6_last_error() has the text.
 *  - per-env arrays are structure-of-arrays, component-major: x[c][n]  (c*n + i).
 *    Actions are the exception: [n][3] float32 row-major, exactly the array SB3 hands to
 *    VecEnv.step_async.
 *  - environments are independent; `env_offset` is the global index of local env 0 so that the
 *    counter-based RNG gives the same streams whatever the shard count (SURVEY.md §8e).
 */
#ifndef R6DOF_H
#define R6DOF_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R6_ABI_VERSION 22
#define R6_MAX_LANES 32
#define R6_NSTATE 14
#define R6_NTERMS 7
#define R6_NSTATS 8

/* error codes */
#define R6_OK 0
#define R6_EINVAL (-1) /* bad argument (null pointer, n < 0, bad mode) */
#define R6_ECUDA (-2)  /* CUDA launch / runtime error, text in r6_last_error() */

/* flags[] bits written by step / rollout (rocket_env.py:213, 226, 382-390; main_6DOF.py:47-50) */
#define R6_F_EVENT 0x01      /* solve_ivp status != 0 (ground event or solver failure) */
#define R6_F_OOB 0x02        /* _check_bounds_violation */
#define R6_F_TRUNCATED 0x04  /* TimeLimit hit and not done ("TimeLimit.truncated") */
#define R6_F_ZERO_HEIGHT 0x08
#define R6_F_VEL_LIMIT 0x10
#define R6_F_LAND_RADIUS 0x20
#define R6_F_ATT_LIMIT 0x40
#define R6_F_OMEGA_LIMIT 0x80
#define R6_F_LANDING_ALL 0xF8

/* stats[] slots (device accumulators, float64; reduced over ranks with one all_reduce(SUM)) */
enum {
    R6_S_EPISODES = 0, R6_S_RETURN_SUM, R6_S_LENGTH_SUM, R6_S_LANDED,
    R6_S_GROUND, R6_S_OOB, R6_S_TRUNCATED, R6_S_STEPS
};

/* R6Params.precision: arithmetic and storage type of the dynamics */
#define R6_PREC_F64 0  /* parity path: state / terminal_state are float64 [14][n]; <= 1e-9 vs the reference */
#define R6_PREC_F32 1  /* throughput path: state / terminal_state are float32 [14][n] (pass the float* through the
                          double* members); integrator in float32 with its own stated bound, reward / flags
                          evaluated by the float64 code on the widened state */

/* R6Params.reward_mode bits: the optional reward wrappers of my_environment/wrappers/wrappers.py */
#define R6_RW_ANNEALED 1  /* RewardAnnealing (:39-61; make_annealed_env, main_6DOF.py:55-69): reward = attitude_constraint +
                             goal_conditions + final_position + final_velocity - xi*(a[2]+1); no out-of-bounds penalty */
#define R6_RW_VERTICAL 2  /* VerticalAttitudeReward (:128-155): at touchdown with a positive final_velocity term add
                             clip(2*deg(acos(q0))*weight, -10, 10) */

/* action sources of r6_rollout */
#define R6_ACT_PHILOX 0  /* uniform(-1,1) float32 from Philox4x32-10 (synthetic random policy) */
#define R6_ACT_MLP 1     /* deterministic SB3 MlpPolicy forward, fused (montecarlo_script.py:57-64) */
#define R6_ACT_BUFFER 2  /* actions read from a [k][n][3] device buffer */
#define R6_ACT_MLP_TC 3  /* the same network as R6_ACT_MLP on the tensor cores: one warp = 32 envs, register-chained
                            mma.sync TF32 tiles with 3xTF32 error compensation (|d action| <= 2e-6 vs R6_ACT_MLP) */

/*
 * Derived constants of Rocket6DOF.__init__ (rocket_env.py:71-134, 159-168), the wrappers of
 * make_env() (main_6DOF.py:33-53) and the simulator (simulator.py:9-67).  The host computes them
 * with the reference's own numpy expressions (rl_rocket_6dof_b200/params.py) so that NumPy-version
 * promotion rules never enter the kernel.  Layout is checked at load time with r6_params_size().
 */
typedef struct R6Params {
    double dt;                 /* timestep */
    double max_gimbal;         /* np.deg2rad(20) */
    double normalizer[R6_NSTATE];
    double alfa, eta, gamma, kappa;
    double att_traj_limit[3];  /* rad */
    double land_att_limit[3];  /* rad */
    double omega_lim[3];
    double waypoint;
    double clip_lo, clip_hi;   /* ClipReward bounds (used when clip_reward != 0) */
    double oob_penalty;        /* -50, rocket_env.py:228-229 */
    float max_thrust;
    float beta, w_v_f, w_r_f, max_r_f, max_v_f;
    float maximum_v, target_r, zero_height_tol;
    float bounds_low[3], bounds_high[3];
    float ic_low[R6_NSTATE], ic_high[R6_NSTATE];
    int32_t shaping_velocity;   /* 0 'acceleration', 1 'velocity' */
    int32_t max_episode_steps;  /* TimeLimit; 0 = none */
    int32_t clip_reward;        /* apply ClipReward(clip_lo, clip_hi) to reward[] */
    int32_t auto_reset;         /* != 0: VecEnv semantics, finished envs are reset inside the step; 0: one-episode semantics
                                   (evaluate_policy / montecarlo_script.py): an env that finishes keeps done = 1, its terminal
                                   observation / state / ep_info recorded, and is skipped by every later r6_step* / r6_rollout
                                   call until r6_reset clears it */
    int32_t n_t;                /* entries in R6Buffers.t_table */
    int32_t obs_rows;           /* rows of obs[] / terminal_obs[] the kernels write: 0 or 14 = all, 13 = RemoveMassFromObs
                                   (saves the mass row when obs[] is mapped host memory) */
    int32_t precision;          /* R6_PREC_F64 / R6_PREC_F32 */
    int32_t reward_mode;        /* R6_RW_* bits, 0 = the plain env reward */
    double va_threshold;        /* VerticalAttitudeReward threshold_height (1e-3) */
    double va_weight;           /* VerticalAttitudeReward weight (-0.5) */
    float xi;                   /* RewardAnnealing thrust penalty (reward_coeff["xi"], default 0.01) */
    int32_t obs_row_major;      /* r6_step (fused kernel) only: write obs[] as [n][obs_rows] row-major — the array a VecEnv
                                   returns — instead of component-major; each warp stages its 32 x obs_rows block through
                                   shared memory and stores it as one contiguous run (meant for obs[] in mapped host memory) */
} R6Params;

/* Device pointers. n = number of local envs. Nullable members are marked. */
typedef struct R6Buffers {
    /* persistent env state */
    double *state;          /* [14][n] float64 (Simulator6DOF.state); float32 [14][n] when precision = R6_PREC_F32 */
    float *m0;              /* [n] initial mass of the episode (simulator.py:42) */
    float *v0;              /* [n] ||IC[3:6]|| (rocket_env.py:651) */
    int32_t *step_count;    /* [n] steps taken in the episode (time = t_table[step_count]) */
    uint32_t *episode_id;   /* [n] episodes started by this env (RNG counter) */
    double *ep_return;      /* [n] running sum of reward[] over the episode (Monitor "r") */
    /* per-step outputs */
    float *obs;             /* [14][n] (row 13 = mass/normalizer; RemoveMassFromObs = rows 0..12) */
    double *reward;         /* [n] nullable when reward_f32 is given */
    uint8_t *done;          /* [n] done OR truncated (what a VecEnv reports) */
    uint8_t *flags;         /* [n] R6_F_* */
    float *terminal_obs;    /* [14][n] obs of the last step of a finished episode ("terminal_observation") */
    double *terminal_state; /* [14][n] SIM.states[-1] of a finished episode (montecarlo_script.py:35); dtype as state */
    double *reward_terms;   /* [7][n] nullable: rewards_dict values in insertion order */
    uint8_t *nattempts;     /* [n] nullable: RK attempts of the step (nfev = 2 + 6*nattempts) */
    int8_t *status;         /* [n] nullable: solve_ivp status of the step (0, 1, -1) */
    double *ep_info;        /* [2][n] nullable: (return, length) of the episode that just finished — float64 like the
                               running sum Monitor reports (stable_baselines3 Monitor: info["episode"]["r"], ["l"]) */
    float *reward_f32;      /* [n] nullable: reward[] rounded to float32 (what a VecEnv hands to SB3) */
    /* tables */
    const double *t_table;  /* [n_t] t_k = round(t_{k-1}+dt, 3) (simulator.py:92) */
    const float *ic_table;  /* [ic_table_len][14] nullable: initial conditions to replay instead of
                               sampling; row = (global_env + n_global*episode) % ic_table_len */
    int64_t ic_table_len;
    int64_t n_global;       /* total envs over all shards (ic_table indexing) */
    double *stats;          /* [8] nullable: R6_S_* accumulators */
    uint8_t *scratch;       /* [2][n] nullable DEVICE bytes: when given, r6_step runs as two kernels (integrator | reward,
                               flags, reset, observation) that hand the solver status / attempt count through it */
    uint8_t *work;          /* nullable, needs scratch: r6_work_bytes(n) DEVICE bytes, zero-filled once by the caller.
                               When given, the integrator runs as three passes cut at RK-attempt boundaries, the
                               unfinished envs of a pass compacted into work lists for the next (a warp then never
                               idles through attempts only some of its envs need) */
    float *tgo;             /* [n] nullable: t_go root of the env's previous step (0 = none; r6_reset and the auto-reset
                               write 0), the warm start of the next step's root iteration (rocket_env.py:528-546).
                               Results do not depend on it beyond round-off: a warm result is used only when certified
                               to be the largest root, otherwise the cold start runs */
} R6Buffers;

/*
 * Weights of the SB3 MlpPolicy actor (net_arch [128, 64], tanh), float32 row-major [out][in].
 * With the value tower set (vf_w0 != NULL) the network is instead SB3 1.6's default separate towers,
 * net_arch [dict(pi=[64, 64], vf=[64, 64])]: w0 [64][13], b0 [64], w1 [64][64], b1 [64] are the policy tower
 * (mlp_extractor.policy_net), vf_* the value tower (mlp_extractor.value_net); w2, b2 read the policy latent and
 * wv, bv the value latent.  Entry points without a separate-tower kernel return R6_EINVAL for such a network:
 * r6_policy* with tensor_cores = 1, r6_rollout with R6_ACT_MLP / R6_ACT_MLP_TC, r6_policy_sde_range and r6_ppo_grad_sde
 * (gSDE on the separate towers has its own entry points, r6_policy_sde_sep_range and r6_ppo_grad_sde_sep).
 */
typedef struct R6Mlp {
    const float *w0, *b0;   /* [128][13], [128]   (separate towers: [64][13], [64]) */
    const float *w1, *b1;   /* [64][128], [64]    (separate towers: [64][64], [64]) */
    const float *w2, *b2;   /* [3][64],  [3]    action_net */
    const float *wv, *bv;   /* [64], [1] nullable: value_net on the same latent (the critic of the shared-trunk policy) */
    const float *log_std;   /* [3] nullable: state-independent log standard deviation of the Gaussian policy */
    const float *vf_w0, *vf_b0;   /* [64][13], [64] nullable: value tower layer 0 (all four set, or none) */
    const float *vf_w1, *vf_b1;   /* [64][64], [64] nullable: value tower layer 1 */
} R6Mlp;

int r6_abi_version(void);
const char *r6_last_error(void);
int r6_params_size(void);
int r6_buffers_size(void);

/*
 * Rocket6DOF.reset (rocket_env.py:180-199) + Simulator6DOF.__init__ (simulator.py:9-67) for every
 * env whose mask byte is non-zero (mask == NULL: all).  Initial conditions are drawn uniformly in
 * [ic_low, ic_high] in float64 and cast to float32 like gym's Box.sample, then the quaternion is
 * normalised in float32 (rocket_env.py:190).  RNG: Philox4x32-10, key = seed,
 * counter = (global env id, episode id).  Writes state, m0, v0, step_count = 0, ep_return = 0, obs.
 */
int r6_reset(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset,
             const uint8_t *mask, uint64_t seed, void *stream);

/*
 * Rocket6DOF.step (rocket_env.py:201-231) through Simulator6DOF.step (simulator.py:69-104) and
 * SciPy's solve_ivp/RK45, with the make_env() wrappers (RemoveMassFromObs is a view of obs,
 * ClipReward, TimeLimit) and the DummyVecEnv auto-reset when p->auto_reset is set.
 * actions: [n][3] float32 in [-1, 1].
 */
int r6_step(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset,
            const float *actions, uint64_t seed, void *stream);

/*
 * r6_step with the synthetic random policy generated in the kernels: action = uniform(-1,1) float32 from Philox
 * (seed, global env id, step_index) — the same stream as r6_rollout(R6_ACT_PHILOX) with step_base + j = step_index.
 * Needs R6Buffers.scratch (runs as the integrator | post-step kernel pair).
 */
int r6_step_random(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset, uint64_t seed,
                   int64_t step_index, void *stream);

/*
 * r6_step / r6_step_random restricted to the env sub-range [first, first + count) of the batch; n stays the size
 * (= SoA stride) of the buffers and actions the full [n][3] array (NULL: Philox actions keyed by step_index, as
 * r6_step_random).  Envs are independent (rocket_env.py:201-231 touches one env), so a host may step disjoint
 * sub-ranges of one batch on different streams: the tail of one range's kernels then overlaps the next range's
 * work instead of idling the SMs.  Needs R6Buffers.scratch (kernel pair only).  Ordering between the streams and
 * whatever consumes the outputs is the caller's business.  lane (0 .. R6_MAX_LANES-1) names the caller's stream:
 * ranges that may run concurrently must use different lanes (each lane has its own work-list counters).
 */
int r6_step_range(const R6Params *p, const R6Buffers *b, int64_t n, int64_t first, int64_t count, int32_t lane,
                  int64_t env_offset, const float *actions, uint64_t seed, int64_t step_index, void *stream);

/* Size of R6Buffers.work for n envs. */
int64_t r6_work_bytes(int64_t n);

/*
 * k fused env-steps per launch with the state held in registers.
 * mode R6_ACT_PHILOX: action = uniform(-1,1) from (seed, global env id, step_base + j);
 * mode R6_ACT_MLP:    action = clip(actor(obs[0:13]), -1, 1), the deterministic SB3 MlpPolicy forward
 *                     (float32, weights staged in shared memory) — evaluate_policy of
 *                     montecarlo_script.py:57-64 with the policy inside the kernel;
 * mode R6_ACT_MLP_TC: as R6_ACT_MLP, evaluated warp-collectively on the tensor cores (csrc/r6_mlp_tc.cuh);
 * mode R6_ACT_BUFFER: action = act_buf[j][i][:].
 * p->auto_reset != 0: finished envs restart inside the kernel (VecEnv semantics).
 * p->auto_reset == 0: one episode per env — an env that finishes keeps done = 1, its terminal
 *                     state / observation / ep_info, and is skipped by later launches until r6_reset.
 * traj_* (nullable) record the rollout: obs [k][13][n] (observation the action was computed
 * from), act [k][n][3], rew [k][n] float32, done [k][n] uint8 (2 = padding after a frozen env's end).
 */
int r6_rollout(const R6Params *p, const R6Buffers *b, int64_t n, int64_t env_offset, int32_t k,
               int32_t mode, const R6Mlp *mlp, const float *act_buf, uint64_t seed,
               int64_t step_base, float *traj_obs, float *traj_act, float *traj_rew,
               uint8_t *traj_done, void *stream);

/*
 * Simulator6DOF.step in raw mode (python-list IC / control: everything float64),
 * the call of test_6DOF_simulator.py:3-7.  state [14][n] in/out, u [3][n], m0 [n], t [n],
 * status [n] out, nattempts [n] nullable.
 */
int r6_sim_step_raw(double *state, const double *u, const double *m0, const double *t, double dt,
                    int64_t n, int8_t *status, uint8_t *nattempts, void *stream);

/* _compute_atarg's t_go (rocket_env.py:528-546): largest positive real root of
 * c0 t^4 + c2 t^2 + c3 t + c4, one per element (NaN when there is none).  guess [n] nullable: per-element warm
 * start of the iteration (the kernels pass the previous step's root), <= 0 = cold start. */
int r6_tgo(const double *c2, const double *c3, const double *c4, double c0, int64_t n, const double *guess, double *tgo,
           void *stream);

/*
 * The policy alone: actions[i][0:3] = clip(actor(obs[0:13][i]), -1, 1) for n envs, as its own kernel
 * (model.predict(obs, deterministic=True) of montecarlo_script.py:57-64 / PPO.collect_rollouts).  A closed-loop
 * VecEnv step is then r6_policy followed by r6_step: the network runs as a uniform, high-occupancy GEMM-chain
 * kernel instead of inside the divergent integrator.  obs: float32 [>=13][n] component-major (R6Buffers.obs);
 * actions: float32 [n][3].  tensor_cores = 0: float32 FMAs (R6_ACT_MLP's code); 1: mma.sync TF32 tiles with 3xTF32
 * compensation (|d action| <= 2e-6 vs mode 0); 2: tcgen05.mma kind::tf32 with accumulators and activations in
 * tensor memory, single pass (fast mode, |d action| ~2e-3 vs mode 0); 3: the same kernel with 3xTF32 compensation
 * chained into one TMEM accumulator and a float32-accurate tanh (faithful mode, |d action| <= 3e-6 vs mode 0 and vs
 * the reference's recorded actions; the mode the closed-loop and PPO-collection paths use by default).  Modes 2 and 3
 * need mlp->w1 (and with the separate towers mlp->vf_w1) 16-byte aligned.  The separate towers run in modes 0, 2, 3.
 */
int r6_policy(const R6Mlp *mlp, const float *obs, int64_t n, int32_t tensor_cores, float *actions, void *stream);

/*
 * The full forward pass PPO.collect_rollouts needs (SB3 ActorCriticPolicy.forward): Gaussian mean from action_net,
 * value from value_net on the same latent, and — when stochastic != 0 — an action sampled as
 * mean + exp(log_std) * eps with eps ~ N(0, 1) from Philox (seed, global env id, step_index) and its log-probability
 * (sum over the 3 action dimensions, evaluated on the UNclipped sample like SB3's DiagGaussianDistribution).
 * actions [n][3]: what the env is stepped with (clipped to [-1, 1]); actions_raw [n][3], values [n], log_prob [n]
 * are nullable.  stochastic == 0: the deterministic mean (r6_policy) with the value, log_prob of the mean.
 */
int r6_policy_ex(const R6Mlp *mlp, const float *obs, int64_t n, int32_t tensor_cores, int32_t stochastic, uint64_t seed,
                 int64_t env_offset, int64_t step_index, float *actions, float *actions_raw, float *values,
                 float *log_prob, void *stream);

/*
 * r6_policy_ex for the env sub-range [first, first + count): obs stays the [14][n] array (n = its stride) and the
 * outputs the full [n]-sized arrays, of which only the rows of the sub-range are written.  Pairs with
 * r6_step_range so that a closed loop (policy, env step) can run per sub-range on its own stream.
 */
int r6_policy_range(const R6Mlp *mlp, const float *obs, int64_t n, int64_t first, int64_t count, int32_t tensor_cores,
                    int32_t stochastic, uint64_t seed, int64_t env_offset, int64_t step_index, float *actions,
                    float *actions_raw, float *values, float *log_prob, void *stream);

/*
 * Generalised state-dependent exploration (stable-baselines3 1.6.0 `PPO(..., use_sde=True)`: StateDependentNoiseDistribution
 * with full_std=True, use_expln=False, learn_features=False, epsilon=1e-6; the latent is the 64-unit trunk output h):
 *     E_i = exp(log_std) * xi_i   (xi_i ~ N(0, 1) [64][3], one matrix per env, drawn by policy.reset_noise(n_envs))
 *     raw = mean + h E_i,   std_a = sqrt(sum_k h_k^2 exp(2 log_std[k][a]) + 1e-6)
 * log_prob and entropy are those of N(mean, std), summed over the 3 actions, with h detached.
 */
#define R6_SDE_LATENT 64
#define R6_SDE_NXI 192        /* xi components per env: [64][3], component c = 3 k + a */
typedef struct R6Sde {
    const float *log_std;     /* [64][3] */
    const float *xi;          /* [192][n] component-major standard normals (r6_sde_noise); nullable for r6_ppo_grad_sde */
} R6Sde;
int r6_sde_size(void);

/*
 * StateDependentNoiseDistribution.sample_weights / policy.reset_noise(n_envs) for the envs [first, first + count) of a
 * batch of n: xi[c][i] for the 192 components, standard normals from Philox4x32-10 keyed (seed, env_offset + i,
 * step_index) through Box-Muller.  The result depends on the global env id and the draw step only, not on the shard, lane
 * or sub-range that draws it.  The exploration matrix is E = exp(log_std) * xi, formed by the policy kernel with the
 * current log_std (log_std does not change during a collection, so that is SB3's draw-time product).
 */
int r6_sde_noise(int64_t n, int64_t first, int64_t count, uint64_t seed, int64_t env_offset, int64_t step_index, float *xi,
                 void *stream);

/*
 * r6_policy_range with the gSDE head (SB3 ActorCriticPolicy.forward with use_sde=True): mean and value as
 * r6_policy_range; stochastic != 0: actions_raw = mean + h (exp(log_std) * xi) with the env's xi column; log_prob of
 * actions_raw under N(mean, std) above; stochastic == 0: the mean and its log_prob.  mlp->log_std is not read.  Deterministic
 * actions and the values are bit-identical to r6_policy_range's.  tensor_cores = 0 (float32 FMAs), 2 or 3 (tcgen05,
 * the h E and h^2 sigma^2 sums formed in the layer-1 epilogue from the TF32 hi + lo parts); 1 (mma.sync) is not
 * available for gSDE (R6_EINVAL).
 */
int r6_policy_sde_range(const R6Mlp *mlp, const R6Sde *sde, const float *obs, int64_t n, int64_t first, int64_t count,
                        int32_t tensor_cores, int32_t stochastic, float *actions, float *actions_raw, float *values,
                        float *log_prob, void *stream);

/*
 * r6_policy_sde_range for SB3 1.6's separate towers (R6Mlp with the value tower set; PPO("MlpPolicy", env, use_sde=True)
 * without policy_kwargs): h is the POLICY tower's 64-unit latent, the value comes from the value tower and plays no part
 * in the distribution.  Same arguments and outputs as r6_policy_sde_range; deterministic actions and the values are
 * bit-identical to r6_policy_range's on the same towers.  tensor_cores = 0, 2 or 3.  Returns R6_EINVAL, before any CUDA
 * call and writing nothing, for tensor_cores = 1, for a shared trunk (its gSDE policy is r6_policy_sde_range), and in
 * modes 2 / 3 for w1 or vf_w1 not 16-byte aligned.
 */
int r6_policy_sde_sep_range(const R6Mlp *mlp, const R6Sde *sde, const float *obs, int64_t n, int64_t first, int64_t count,
                            int32_t tensor_cores, int32_t stochastic, float *actions, float *actions_raw, float *values,
                            float *log_prob, void *stream);

/*
 * Generalised advantage estimation over a recorded rollout, on the device, so that the PPO update of
 * main_6DOF.py:136 (`model.learn`) can consume r6_rollout's trajectory buffers without a host round trip.
 * Restates stable-baselines3 1.6.0 `RolloutBuffer.compute_returns_and_advantage` (common/buffers.py; SB3 is a
 * dependency of the reference, not part of its tree) in float32 with NumPy's operation order:
 *     nnt_t   = 1 - done[t]                      (done[t] = episode ended at step t = episode_starts[t+1])
 *     delta_t = rew[t] + gamma * V[t+1] * nnt_t - V[t]          (V[T] = last_values)
 *     A_t     = delta_t + f32(gamma * lambda) * nnt_t * A_{t+1}  (A_T = 0),   returns = A + V
 * rew, values, adv, ret: float32 [T][n]; done: uint8 [T][n] (non-zero = ended); last_values: float32 [n].
 */
int r6_gae(const float *rew, const float *values, const uint8_t *done, const float *last_values, int32_t T, int64_t n,
           double gamma, double gae_lambda, float *adv, float *ret, void *stream);

/*
 * Bootstrapping of TimeLimit truncations with the critic, as stable-baselines3 1.6.0
 * `OnPolicyAlgorithm.collect_rollouts` does while collecting (SB3 issue #633):
 *     if done and infos[i]["terminal_observation"] is not None and infos[i]["TimeLimit.truncated"]:
 *         rewards[i] += gamma * predict_values(terminal_observation)
 * in three passes that need no host synchronise:
 *  1. r6_trunc_record after each env step of the rollout (step = its index in [0, T)), on the stream and env sub-range of
 *     that step: every env of [first, first + count) with R6_F_TRUNCATED in flags[i] takes the first slot s with
 *     slot_step[s][i] < 0, sets slot_step[s][i] = step and copies rows 0..12 of terminal_obs[:, i] into slot_obs[s][:, i].
 *     A truncation that finds no free slot is dropped (nothing is written past slot slots - 1); one env truncates at most
 *     ceil(T / max_episode_steps) times in T steps, so that many slots always suffice.  Launched as a programmatic
 *     dependent like the env-step kernels.  slot_step: int32 [slots][n], all -1 before the first step of the rollout;
 *     slot_obs: float32 [slots][13][n] (component-major, the observation layout r6_policy_range reads).
 *  2. r6_policy_range over each slot layer slot_obs[s] (all n columns; columns of free slots hold anything and their
 *     values are not read), with the collection's tensor_cores mode, writing V into slot_values[s].
 *  3. r6_trunc_bootstrap: rew[t][i] = f32(rew[t][i] + f32(f32(gamma) * slot_values[s][i])) for every slot with
 *     t = slot_step[s][i] in [0, T) — SB3's float32 arithmetic, two roundings, no FMA.  rew: float32 [T][n] (the rewards
 *     of the rollout, before r6_gae); slot_values: float32 [slots][n].
 */
int r6_trunc_record(const uint8_t *flags, const float *terminal_obs, int64_t n, int64_t first, int64_t count, int32_t step,
                    int32_t slots, int32_t *slot_step, float *slot_obs, void *stream);
int r6_trunc_bootstrap(float *rew, int32_t T, int64_t n, int32_t slots, const int32_t *slot_step, const float *slot_values,
                       double gamma, void *stream);

/*
 * PPO update (stable-baselines3 1.6.0 `PPO.train`, the optimiser of main_6DOF.py:136).
 *
 * Flat parameter vector of the actor-critic, R6_PPO_NPARAMS float32 in SB3 [out][in] order:
 *     w0 [128][13] @0, b0 [128] @1664, w1 [64][128] @1792, b1 [64] @9984, w2 [3][64] @10048, b2 [3] @10240,
 *     wv [64] @10243, bv [1] @10307, log_std [3] @10308
 * (w1 starts at float 1792 so that an R6Mlp pointing into a 16-byte aligned buffer keeps w1 16-byte aligned, as
 * r6_policy tensor_cores = 2 / 3 need).
 *
 * The separate-tower layout (R6Mlp with the value tower), R6_PPO_NPARAMS_SEP float32:
 *     w0 [64][13] @0, vf_w0 [64][13] @832, b0 [64] @1664, vf_b0 [64] @1728, w1 [64][64] @1792, b1 [64] @5888,
 *     vf_w1 [64][64] @5952, vf_b1 [64] @10048, w2 [3][64] @10112, b2 [3] @10304, wv [64] @10307, bv [1] @10371,
 *     log_std [3] @10372
 * (the two layer-0 blocks stacked are the shared layout's [128][13] + [128]; w1 and vf_w1 are 16-byte aligned).
 * r6_ppo_grad takes the layout of its mlp: grad_sum has R6_PPO_NPARAMS_SEP elements when the value tower is set.
 */
#define R6_PPO_NPARAMS 10311
#define R6_PPO_NPARAMS_SEP 10375
#define R6_PPO_NTERMS 5
/* terms[] slots of r6_ppo_grad (float64 sums over the minibatch) */
enum { R6_PPO_T_PG = 0, R6_PPO_T_VLOSS, R6_PPO_T_CLIPPED, R6_PPO_T_APPROX_KL, R6_PPO_T_BAD_INDEX };

/* The [T][n] trajectory of a collected rollout; sample s = t * n + i. */
typedef struct R6PpoRollout {
    const float *obs;        /* observation component c of (t, i) at obs[t * obs_stride_step + c * obs_stride_comp +
                                i * obs_stride_env] (element strides): the strided [T, n, 13] view of the in-place
                                [T + 1][14][n] collection buffer and a dense [T][n][13] array are both accepted */
    int64_t obs_stride_step, obs_stride_comp, obs_stride_env;
    const float *actions;    /* [T][n][3] raw (unclipped) Gaussian samples */
    const float *log_probs;  /* [T][n] log-probabilities at collection */
    const float *advantages; /* [T][n] */
    const float *returns;    /* [T][n] */
    int64_t T, n;
    const float *old_values; /* [T][n] the critic's values at collection (collect_rollout's `values`, before any
                                truncation bootstrap); read only when R6PpoCoef.clip_range_vf > 0, nullable otherwise */
} R6PpoRollout;

typedef struct R6PpoCoef {
    double clip_range, vf_coef, ent_coef;
    const double *adv_stats; /* DEVICE [2] = (mean, 1 / (std + 1e-8)) of the minibatch's advantages, or NULL = no
                                normalisation.  A device pointer, so that no minibatch has to synchronise */
    double clip_range_vf;    /* SB3's clip_range_vf: > 0 clips the value prediction to old_values +- clip_range_vf
                                (rollout->old_values required); 0 = off.  Negative or non-finite: R6_EINVAL */
} R6PpoCoef;

typedef struct R6AdamCoef {
    double lr, beta1, beta2, eps;
    double max_grad_norm;    /* clip_grad_norm_(max_grad_norm) on the scaled gradient; <= 0: no clipping */
    double scale;            /* g = scale * grad_sum (1 / minibatch size turns r6_ppo_grad's sum into the mean) */
} R6AdamCoef;

int r6_ppo_rollout_size(void);
int r6_ppo_coef_size(void);
int r6_adam_coef_size(void);

/* Size of r6_ppo_grad's work buffer for a minibatch of B samples, either layout (DEVICE bytes, no initialisation needed). */
int64_t r6_ppo_work_bytes(int64_t B);

/*
 * Sum over the minibatch idx[0..B) (int64 sample indices s = t * n + i, any order, duplicates allowed) of the
 * per-sample gradient of SB3 1.6's PPO loss
 *     -min(A' ratio, A' clip(ratio, 1 - clip_range, 1 + clip_range)) + vf_coef (R - V)^2 - ent_coef entropy,
 * ratio = exp(logp(actions) - log_probs), A' the (optionally normalised) advantage, into grad_sum [R6_PPO_NPARAMS]
 * (flat layout above), and the loss-term sums into terms [R6_PPO_NTERMS] float64: policy-gradient loss, value loss
 * (R - V)^2, the number of samples with |ratio - 1| > clip_range, (ratio - 1) - log ratio, and the number of indices
 * outside [0, T n) (those samples are skipped).  mlp must carry wv, bv and log_std.  Sums, not means: the caller scales.
 * The launch shape depends on B only, so the result is bit-reproducible on any device.
 *
 * Value clipping (coef->clip_range_vf = c > 0, SB3's clip_range_vf): per sample, in float32 and torch's order,
 *     d = V - V_old,  vp = V_old + clamp(d, -fl32(c), fl32(c)),  value loss (R - vp)^2,
 * V_old = rollout->old_values; d loss / d V = 2 vf_coef (vp - R) for -c <= d <= c, else 0 (the sample adds nothing to
 * the value head or, with separate towers, to the value tower).  terms[R6_PPO_T_VLOSS] is then the sum of the clipped
 * (R - vp)^2.  Returns R6_EINVAL, before any CUDA call and writing nothing, for c < 0 or not finite, and for c > 0 with
 * old_values NULL and B > 0.  c = 0 is the unclipped loss above, bit for bit.
 */
int r6_ppo_grad(const R6Mlp *mlp, const R6PpoRollout *rollout, const int64_t *idx, int64_t B, const R6PpoCoef *coef,
                float *grad_sum, double *terms, void *work, void *stream);

/*
 * r6_ppo_grad for a gSDE policy (PPO(use_sde=True).train; SB3 1.6 also calls reset_noise(batch_size) per minibatch, which
 * does not enter the loss).  Flat layout R6_PPO_NPARAMS_SDE: the prefix of R6_PPO_NPARAMS through bv, then
 * log_std [64][3] @10308.  Per sample, std_a, log_prob and entropy of N(mean, std) as r6_policy_sde_range; the entropy
 * bonus uses that per-sample entropy, and
 *     d loss / d log_std[k][a] = exp(2 log_std[k][a]) sum_s h_{s,k}^2 (w_s (z_{s,a}^2 - 1) - ent_coef) / std_a(s)^2,
 * w = d pg / d logp, z = (a - mean) / std.  terms [R6_PPO_NTERMS_SDE]: those of r6_ppo_grad plus the sum of the per-sample
 * entropies (R6_PPO_T_ENTROPY).  sde->log_std is the [64][3] matrix (sde->xi is not read; mlp->log_std is not read).
 * Value clipping (coef->clip_range_vf) and its R6_EINVAL cases as r6_ppo_grad.
 */
#define R6_PPO_NPARAMS_SDE 10500
#define R6_PPO_NTERMS_SDE 6
#define R6_PPO_T_ENTROPY 5
/* Size of the work buffer of r6_ppo_grad_sde and r6_ppo_grad_sde_sep for a minibatch of B samples (either layout). */
int64_t r6_ppo_sde_work_bytes(int64_t B);
int r6_ppo_grad_sde(const R6Mlp *mlp, const R6Sde *sde, const R6PpoRollout *rollout, const int64_t *idx, int64_t B,
                    const R6PpoCoef *coef, float *grad_sum, double *terms, void *work, void *stream);

/*
 * r6_ppo_grad_sde for SB3 1.6's separate towers with gSDE (mlp with the value tower set; a shared trunk is R6_EINVAL).
 * Flat layout R6_PPO_NPARAMS_SEP_SDE: the prefix of R6_PPO_NPARAMS_SEP through bv (10372 floats), then
 * log_std [64][3] @10372 (16-byte aligned).  h above is the policy tower's latent, detached: no gradient flows through
 * std into either tower, whose deltas are those of r6_ppo_grad on the separate towers.  grad_sum [R6_PPO_NPARAMS_SEP_SDE],
 * terms [R6_PPO_NTERMS_SDE]; value clipping and its R6_EINVAL cases as r6_ppo_grad.
 */
#define R6_PPO_NPARAMS_SEP_SDE 10564
int r6_ppo_grad_sde_sep(const R6Mlp *mlp, const R6Sde *sde, const R6PpoRollout *rollout, const int64_t *idx, int64_t B,
                        const R6PpoCoef *coef, float *grad_sum, double *terms, void *work, void *stream);

/*
 * One torch.optim.Adam step (no weight decay, no amsgrad) on the flat parameters, after clip_grad_norm_:
 *     g = scale * grad_sum;  norm = ||g||_2 (accumulated in float64);  g *= min(1, max_grad_norm / (norm + 1e-6));
 *     m = lerp(m, g, 1 - beta1);  v = beta2 v + (1 - beta2) g^2;
 *     p -= lr / (1 - beta1^step) * m / (sqrt(v) / sqrt(1 - beta2^step) + eps)
 * params, grad_sum, m, v: float32 [P] DEVICE (any P: R6_PPO_NPARAMS, R6_PPO_NPARAMS_SDE, ...); step >= 1 counts the updates including this one; grad_norm_out
 * (nullable DEVICE double) receives the norm before clipping.
 */
int r6_adam_step(float *params, const float *grad_sum, float *m, float *v, int64_t P, const R6AdamCoef *coef,
                 int64_t step, double *grad_norm_out, void *stream);

/* Zeroes stats[8] (asynchronously, on the stream). */
int r6_stats_reset(double *stats, void *stream);

/* Micro-benchmarks for the roofline denominators (SURVEY.md §8d): a dependent-free DFMA / FFMA
 * loop; returns nothing, the caller times it.  flops = 2 * threads * iters * 8 chains. */
int r6_peak_fma(int32_t fp64, int64_t blocks, int32_t iters, double *sink, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* R6DOF_H */
