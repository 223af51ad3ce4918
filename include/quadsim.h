/*
 * quadsim.h -- C ABI of libquadsim.so, the B200 (sm_100a) batched WaypointQuadEnv simulator.
 *
 * The reference (LahiruCooray/rl-aerial-manipulator) has no FFI: its hot path sits behind two
 * Python protocols, gymnasium.Env (the reference class) and Stable-Baselines3 VecEnv (what drives
 * it).  The entry points below are what a binding for that path needs; each one names the reference
 * interface it replaces (paths relative to the reference root).  INTEGRATION.md shows the ctypes
 * stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every buffer is CALLER-OWNED DEVICE memory (e.g. torch CUDA tensors' data_ptr()), except where a
 *     parameter is documented as host memory; the handle owns only the per-env hidden state pool;
 *   - `stream` is a cudaStream_t passed as void*; calls are stream-ordered and return immediately;
 *   - every function returns 0 on success or a negative QS_E* code; the text of the last error of a
 *     handle (or of the library, for a NULL handle) is returned by qs_last_error();
 *   - no C++ exceptions cross this boundary; one handle must not be used from two threads at once.
 */
#ifndef QUADSIM_H
#define QUADSIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QS_ABI_VERSION 3

/* error codes */
#define QS_OK 0
#define QS_EINVAL (-1)  /* bad argument / unsupported configuration */
#define QS_ECUDA (-2)   /* a CUDA runtime call failed; see qs_last_error() */
#define QS_ENOMEM (-3)

/* qs_config.precision */
#define QS_F32 0
#define QS_F64 1
/* qs_config.integrator */
#define QS_RK4 0    /* fixed-step classical RK4, `substeps` sub-intervals per 5 ms env step (throughput mode) */
#define QS_LSODA 1  /* per-env port of ODEPACK LSODA's Adams path == scipy.integrate.odeint defaults (parity mode, f64) */

/* bits of the per-env flags byte written by qs_step / qs_rollout_step */
#define QS_FLAG_TERMINATED 0x01
#define QS_FLAG_TRUNCATED 0x02   /* the reference's `truncated` return value (may be set together with TERMINATED) */
#define QS_FLAG_SUCCESS 0x04     /* info['success'] is True  */
#define QS_FLAG_STOPPED 0x08     /* info['stopped'] is True  */
#define QS_FLAG_CRASHED 0x10     /* info['crashed']          */
#define QS_FLAG_OOB 0x20         /* info['out_of_bounds']    */
#define QS_FLAG_LSODA_FAIL 0x80  /* LSODA mode only: the integrator hit a condition the port does not cover */

#define QS_ACT_DIM 4
#define QS_STATE_DIM 13
#define QS_MAX_WAYPOINTS 3
#define QS_TRIG_TAB 6
#define QS_RESET_UNIFORMS 18  /* unit uniforms one reset may consume (qs_reset_uniforms) */

typedef struct qs_handle qs_handle;

/*
 * Environment batch configuration.
 * Replaces: WaypointQuadEnv.__init__ (initial-implementation-v2/rl_env_scaledObs.py:10-38,
 * initial-implementation-v1/rl_env_scaledObs.py:9-30) x n_envs, as built by
 * make_vec_env(WaypointQuadEnv, n_envs=8) (initial-implementation-v1/rl_train_vecN.py:10).
 */
typedef struct qs_config {
    int32_t abi_version;       /* QS_ABI_VERSION */
    int32_t env_version;       /* 1: initial-implementation-v1, 2: initial-implementation-v2 */
    int32_t obs_scaled;        /* 1: rl_env_scaledObs.py, 0: rl_env.py (raw 17-D obs; v1 only) */
    int32_t precision;         /* QS_F32 | QS_F64 */
    int32_t integrator;        /* QS_RK4 | QS_LSODA (LSODA requires QS_F64) */
    int32_t substeps;          /* RK4 sub-intervals (>= 1) */
    int32_t action_scale_f32;  /* 1: scale actions in float32 like NumPy>=2 does for float32 actions (default) */
    int32_t auto_reset;        /* 1: DummyVecEnv semantics, done envs are reset inside the step kernel */
    int32_t device;            /* CUDA device ordinal */
    int32_t v2_random_waypoints; /* env_version 2 only.  0: num_waypoints = 1, as shipped (rl_env_scaledObs.py:47).
                                    1: num_waypoints = np.random.randint(2, 4), the alternative the reference keeps commented
                                    out at :46 (drawn at that position), trajectories of 2-3 waypoints */
    int64_t n_envs;            /* envs owned by this handle (this rank's shard) */
    int64_t env_id_offset;     /* global id of local env 0; Philox is keyed on the global id, so a batch sharded
                                  over G ranks draws the same episodes as the unsharded batch */
    uint64_t seed;
    /* model constants, computed on the host with the same NumPy calls the reference uses
       (simul_files/model/params.py:10-36) so that invA / invI are bit-identical */
    double mass, g, dt;
    double inertia[9], inv_inertia[9];
    double mix[16], inv_mix[16];
    double max_prop_thrust, min_prop_thrust; /* maxF/4, minF/4 */
    double sin_tab[QS_TRIG_TAB], cos_tab[QS_TRIG_TAB]; /* np.sin / np.cos of 2*pi*j/K for K = 1..3, j = 1..K at index
                                                          K*(K-1)/2 + j-1 (utils2/utils.py:41,84-85) */
    double lsoda_rtol, lsoda_atol;           /* odeint defaults: 1.49012e-8 */
} qs_config;

/*
 * Canonical float64 struct-of-arrays view of the hidden env state, for parity injection/extraction.
 * All pointers are device pointers with n_envs rows; any pointer may be NULL (field skipped).
 * Replaces: direct attribute access on the reference env (env.quadcopter.state, env.waypoint_list, ...,
 * as read by initial-implementation-v2/simul_files/quadPlot.py:299-326 and runsim_scaledObs.py:29,65-66).
 */
typedef struct qs_state_view {
    double* y;              /* [n,13] pos, vel, quat(wxyz), omega */
    double* wp_list;        /* [n,QS_MAX_WAYPOINTS,3] */
    int32_t* n_wp;          /* [n] */
    int32_t* wp_index;      /* [n] */
    double* last_distance;  /* [n], NaN == None */
    int32_t* current_step;  /* [n] */
    int32_t* counter;       /* [n] (v2) */
    uint8_t* final_reached; /* [n] (v2; == counter_activated) */
    double* final_yaw;      /* [n] (v2) */
    double* ep_return;      /* [n] Monitor-style running episode return */
    int32_t* episode;       /* [n] resets so far (Philox counter word) */
} qs_state_view;

/* Library / lifecycle ---------------------------------------------------------------------------- */
int qs_abi_version(void);
const char* qs_last_error(const qs_handle* h);
int qs_create(const qs_config* cfg, qs_handle** out);
int qs_destroy(qs_handle* h);
int qs_obs_dim(const qs_handle* h);               /* 20 (v2) or 17 (v1) */
int64_t qs_state_bytes_per_env(const qs_handle* h); /* bytes of hidden state per env held in HBM */

/*
 * Reset.  Replaces WaypointQuadEnv.reset (v2 rl_env_scaledObs.py:40-79, v1 :32-51) / VecEnv.reset().
 * env_mask: NULL = all envs, else u8[n] (non-zero = reset).  obs_out: f32[n,obs_dim] (only reset rows written).
 */
int qs_reset(qs_handle* h, const uint8_t* env_mask, float* obs_out, void* stream);

/*
 * One env step for the whole batch: physics + reward + termination + observation (+ auto-reset).
 * Replaces WaypointQuadEnv.step (v2 rl_env_scaledObs.py:123-231, v1 :85-168) over Quadcopter.update
 * (simul_files/model/quadcopter.py:105-114), looped by DummyVecEnv.step_wait.
 *   actions          f32[n,4]   (not clipped here: SB3 clips before env.step)
 *   obs_out          f32[n,obs_dim]  post-step obs, or the reset obs for envs that were auto-reset
 *   reward_out       f32[n] (QS_F32) or f64[n] (QS_F64)
 *   flags_out        u8[n]  QS_FLAG_* bits
 *   terminal_obs_out f32[n,obs_dim] or NULL; written only for done envs (info['terminal_observation'])
 *   ep_return_out    same dtype as reward_out, or NULL; written only for done envs (Monitor 'r')
 *   ep_len_out       i32[n] or NULL; written only for done envs (Monitor 'l')
 */
int qs_step(qs_handle* h, const float* actions, float* obs_out, void* reward_out, uint8_t* flags_out,
            float* terminal_obs_out, void* ep_return_out, int32_t* ep_len_out, void* stream);

/*
 * qs_step on the env sub-range [first_env, first_env + count) only; every buffer pointer refers to the sub-range's first env.
 * first_env must be a multiple of 32 (the pool is tiled per warp).  Sub-ranges are independent, so a host-facing caller can
 * pipeline chunks on several streams: actions of chunk c+1 go up while chunk c steps and its observations come down
 * (vec_env.QuadVecEnv(pipeline_chunks=...)).  RK4 only; not available while qs_step_moments is armed.
 */
int qs_step_range(qs_handle* h, int64_t first_env, int64_t count, const float* actions, float* obs_out, void* reward_out,
                  uint8_t* flags_out, float* terminal_obs_out, void* ep_return_out, int32_t* ep_len_out, void* stream);

/*
 * T env steps in ONE launch: an env's hidden state stays in registers across the steps (throughput mode for small batches such
 * as BASELINE.json configs[2], 65,536 envs, where a launch and a state round trip per step are the floor).  Same arithmetic as
 * T calls of qs_step (the same device functions); RK4 handles only; not while qs_step_moments is armed.
 *   T                steps per launch (>= 1)
 *   actions          f32[T,n,4] time-major, or NULL: actions are drawn in the kernel, uniform over [action_lo, action_hi) --
 *                    Philox4x32-10 keyed on action_seed, counter = (global env id, *action_step + t); the last CTA to finish adds
 *                    T to *action_step (device u64), so consecutive launches and CUDA-graph replays draw fresh actions
 *   actions_out      f32[T,n,4] or NULL: the actions each step used (what a rollout buffer stores)
 *   obs_out          f32[T,n,obs_dim] time-major (n * obs_dim must be a multiple of 4), or f32[n,obs_dim] = the observations after
 *                    the last step when obs_last_only != 0
 *   reward_out       [T,n] f32/f64; flags_out u8[T,n]; terminal_obs_out f32[T,n,obs_dim] / ep_return_out [T,n] / ep_len_out i32[T,n]
 *                    or NULL, rows written where the env finished in that step
 */
typedef struct qs_step_many_args {
    int32_t T, obs_last_only;
    const float* actions;
    uint64_t action_seed;
    uint64_t* action_step;
    float action_lo[4], action_hi[4];
    float* actions_out;
    float* obs_out;
    void* reward_out;
    uint8_t* flags_out;
    float* terminal_obs_out;
    void* ep_return_out;
    int32_t* ep_len_out;
} qs_step_many_args;
int qs_step_many(qs_handle* h, const qs_step_many_args* a, void* stream);

/*
 * Fused VecNormalize moments: after this call every qs_step also leaves (n, mean[D], M2[D]) of the observations it
 * returned (f64[1+2D], device, caller-owned) in `moments_out` -- what RunningMeanStd.update(obs) needs -- computed inside the
 * step kernel from the obs tile it already holds.  shift_stats: VecNormalize stats f64[1+2D] whose mean is used as the
 * summation offset (conditioning), or NULL.  moments_out == NULL switches the feature off.
 */
int qs_step_moments(qs_handle* h, double* moments_out, const double* shift_stats);
/* merge_stats != NULL: every qs_step additionally Chan-merges that batch triplet into the running statistics merge_stats
 * (f64[1+2D]: count, mean, var), i.e. performs RunningMeanStd.update(obs) itself, in the kernel that finishes the moments --
 * for a single-GPU rollout, where no exchange step sits between the two.  NULL (default) leaves the merge to the caller. */
int qs_step_moments_merge(qs_handle* h, double* merge_stats);

int qs_get_state(qs_handle* h, const qs_state_view* out, void* stream);
int qs_set_state(qs_handle* h, const qs_state_view* in, void* stream);

/* The unit uniforms the reset of (global env id, episode) may consume: f64[n,QS_RESET_UNIFORMS]. Test hook. */
int qs_reset_uniforms(qs_handle* h, const int64_t* env_ids, const int32_t* episodes, int64_t n, double* out,
                      void* stream);

/*
 * Dynamics randomisation (opt-in): per env and per episode, the true mass m*k_m, inertia k_I*I (inverse I^-1/k_I), per-prop
 * thrust factors eta[4] (prop i delivers eta_i * clamp((invA [Fcmd; Mcmd])_i, tmin, tmax), F and M re-mixed from that) and a
 * constant world-frame wind force f_wind[3] in N (dv/dt += f_wind / (m*k_m)).  The action scaling keeps the nominal mass: the
 * controller commands thrust in units of the nominal m*g.  Observations, reward, termination and the reset draws are unchanged.
 * Drawn at every reset (qs_reset, and the auto-reset of qs_step / qs_step_range / qs_step_many) for the episode number that
 * reset uses:  u[0..9] = u53 pairs of Philox4x32-10, key = seed, counter = (global env id lo, hi, episode, 0x100 + b), b = 0..4;
 *   k_m = 1 + mass_rel*(2u0-1),  k_I = 1 + inertia_rel*(2u1-1),  eta_i = 1 + thrust_rel*(2u_{2+i}-1),  f_wind_j = wind*(2u_{6+j}-1)
 * in float64 with round-to-nearest products and sums (stored rounded to float on a QS_F32 handle).
 * Valid: 0 <= mass_rel < 1, 0 <= inertia_rel < 1, 0 <= thrust_rel <= 1 (eta = 0 is a dead motor), wind >= 0, all finite.
 * RK4 handles only; while armed, qs_rollout_step and the QS_STEP_F32_TMA opt-in kernel refuse (QS_EINVAL).
 * qs_dynamics_randomization: cfg NULL disarms.  May be called before or after the first qs_reset; on a reset handle it draws every
 *   env's parameters for its current episode.
 * qs_get_dynamics / qs_set_dynamics: f64[n, QS_DYN_PARAMS] device rows (k_m, k_I, eta[4], f_wind[3]); set values hold until that
 *   env's next reset.  Both need an armed handle.
 */
#define QS_DYN_PARAMS 9   /* k_m, k_I, eta[4], f_wind[3] */
typedef struct qs_dynamics_rand {
    uint64_t seed;
    double mass_rel, inertia_rel, thrust_rel, wind;
} qs_dynamics_rand;
int qs_dynamics_randomization(qs_handle* h, const qs_dynamics_rand* cfg, void* stream);
int qs_get_dynamics(qs_handle* h, double* out, void* stream);
int qs_set_dynamics(qs_handle* h, const double* in, void* stream);

/*
 * LSODA diagnostics of the most recent qs_step in QS_LSODA mode: i32[n,4] = nst, nfe, nqu, status and
 * f64[n,2] = hu, tcur -- the counters scipy's odeint(full_output=True) reports.  Either may be NULL.
 */
int qs_lsoda_stats(qs_handle* h, int32_t* counters_out, double* steps_out, void* stream);

/* VecNormalize --------------------------------------------------------------------------------------
 * Replaces stable_baselines3 VecNormalize(norm_obs=True, norm_reward=False) / RunningMeanStd.update
 * (call sites initial-implementation-v1/rl_train_vecN.py:11, rl_checkpoint_train_vecN.py:23-28, runsim_vecN.py:24-26;
 * field layout pinned by initial-implementation-v1/vec_normalize.pkl).
 * stats layout (device, f64): [0]=count, [1..d]=mean, [1+d..2d]=var  -- RunningMeanStd(mean, var, count).
 */
/* batch moments of x f32[n,d] -> moments f64[1+2d] = (n, mean[d], M2[d]); scratch: f64[qs_moments_scratch_len(d)].
 * The triplet is what ranks all-gather (NCCL) before qs_vecnorm_merge. */
int64_t qs_moments_scratch_len(int d);
int qs_batch_moments(const float* x, int64_t n, int d, double* moments_out, double* scratch, void* stream);
/* running stats <- Chan merge of `k` moment triplets f64[k,1+2d] (RunningMeanStd.update_from_moments, k batches) */
int qs_vecnorm_merge(double* stats, const double* moments, int k, int d, void* stream);
/* out = clip((x - mean) / sqrt(var + eps), +-clip) as f32 (VecNormalize.normalize_obs); out may alias x */
int qs_vecnorm_apply(const float* x, float* out, int64_t n, int d, const double* stats, double eps, double clip,
                     void* stream);
/* returns = returns*gamma + reward; snapshot <- returns (what ret_rms.update sees); returns[done] = 0
 * (VecNormalize.step_wait).  reward is f32[n] or f64[n]; flags u8[n] are qs_step's. */
int qs_returns_update(float* returns, const void* reward, int reward_is_f64, const uint8_t* flags, float gamma,
                      int64_t n, float* snapshot, void* stream);
const char* qs_vecnorm_last_error(void);

/* MlpPolicy rollout forward -----------------------------------------------------------------------
 * Replaces stable_baselines3 ActorCriticPolicy.forward for MlpPolicy(net_arch=[128,64,64], Tanh)
 * (PPO("MlpPolicy", ...) at initial-implementation-v2/rl_train.py:27-53, v1/rl_train_vecN.py:13-33) and, with
 * noise == NULL, ActorCriticPolicy.predict(deterministic=True) (runsim_scaledObs.py:54).
 * params: one f32 device blob of qs_policy_param_count(obs_dim) floats; per net (actor, then critic), weights
 * input-major (W^T of torch's [out,in]):  W1[obs][128] b1[128] W2[128][64] b2[64] W3[64][64] b3[64] Wh[64][4] bh[4]
 * (the critic uses column 0 of Wh / bh[0]); then log_std[4].
 *   obs        f32[n,d]
 *   noise      f32[n,4] standard normal, or NULL for deterministic actions (the mean)
 *   norm_stats f64[1+2d] VecNormalize stats applied to obs on load, or NULL; obs_norm_out f32[n,d] or NULL
 *   actions    f32[n,4] unclipped (what SB3 stores)    actions_clipped f32[n,4] or NULL (clip_lo/clip_hi f32[4], host)
 *   values f32[n]    logp f32[n]
 *   impl       QS_POLICY_FP32: CUDA-core FFMA kernel, float32 throughout;
 *              QS_POLICY_TENSOR: tcgen05/TMEM kernel, split-float16 operands (hi+lo, 3 MMAs per k-step) + float32
 *                                accumulation: float32-level accuracy (values within 2e-3 of float64 on |V| <= 2800);
 *              QS_POLICY_TENSOR_FAST: tcgen05/TMEM kernel, single float16 operands + MUFU.TANH (means within 3e-2,
 *                                values within ~1e-2 |V|max);
 *              QS_POLICY_AUTO: TENSOR for n >= 16384, FP32 below
 */
#define QS_POLICY_AUTO 0
#define QS_POLICY_FP32 1
#define QS_POLICY_TENSOR 2
#define QS_POLICY_TENSOR_FAST 3
#define QS_POLICY_TENSOR_PIPELINE 4 /* QS_POLICY_TENSOR arithmetic on the warp-specialised pipeline of qs_rollout_step (policy part only) */
#define QS_POLICY_TENSOR_CHAINS 5   /* QS_POLICY_TENSOR arithmetic on the three-chain kernel (qs_policy_tc.cu) */
#ifndef QS_POLICY_TENSOR_DEFAULT_PIPELINE
#define QS_POLICY_TENSOR_DEFAULT_PIPELINE 1 /* which of the two QS_POLICY_TENSOR / AUTO run (r02: pipeline 296 us, chains 308 us per 1M envs) */
#endif
int64_t qs_policy_param_count(int obs_dim);
int qs_policy_forward(const float* params, int obs_dim, const float* obs, const float* noise, int64_t n,
                      const double* norm_stats, float norm_eps, float norm_clip, float* obs_norm_out,
                      float* actions, float* actions_clipped, const float* clip_lo, const float* clip_hi,
                      float* values, float* logp, int impl, void* stream);
/* The same forward with the sampling noise drawn INSIDE the kernel (what SB3's DiagGaussianDistribution.sample does every rollout
 * step, call site initial-implementation-v2/rl_train.py:27): Philox4x32-10 keyed on noise_seed, counter = (env_id_offset + row,
 * step) + Box-Muller, the generator of qs_rollout_step's QS_SAMPLE_PHILOX.  counter: device u64[2], 16-byte aligned, zeroed by
 * the caller once -- [0] is the step index (the last CTA to finish adds 1, so consecutive launches and CUDA-graph replays draw
 * fresh noise), [1] is scratch.  Runs on the tcgen05 pipeline kernel (QS_POLICY_TENSOR_PIPELINE arithmetic). */
int qs_policy_forward_philox(const float* params, int obs_dim, const float* obs, int64_t n, uint64_t noise_seed, uint64_t* counter,
                             int64_t env_id_offset, const double* norm_stats, float norm_eps, float norm_clip,
                             float* obs_norm_out, float* actions, float* actions_clipped, const float* clip_lo,
                             const float* clip_hi, float* values, float* logp, void* stream);
const char* qs_policy_last_error(void);

/* Fused rollout step -----------------------------------------------------------------------------------
 * ONE kernel launch per rollout step for the whole shard: VecNormalize normalisation of the current observations -> MlpPolicy
 * forward (actor + critic, tcgen05 split-float16, float32-class accuracy) -> Gaussian sampling, log-prob, clipping to the action
 * box -> env step (physics, reward, termination, observation) -> auto-reset -> VecNormalize batch moments of the returned
 * observations (when qs_step_moments is armed; finalised and, with qs_step_moments_merge, merged into the running statistics by
 * the last CTA of the same launch).
 * Replaces one iteration of stable_baselines3 OnPolicyAlgorithm.collect_rollouts -- policy(obs) -> np.clip -> VecNormalize /
 * DummyVecEnv.step_wait -> WaypointQuadEnv.step (call sites initial-implementation-v2/rl_train.py:27-56,
 * initial-implementation-v1/rl_train_vecN.py:10-36) -- i.e. qs_policy_forward + qs_step (+ the moments kernels) in one launch;
 * results are identical to that sequence run with the same noise.  float32 / RK4 handles only.
 *
 * qs_policy_prepare turns the float32 parameter blob of qs_policy_forward into the operand image the kernel loads (float16 hi/lo
 * tensor-core operands + the float32 heads, qs_policy_image_bytes() bytes, device, 16-byte aligned); call it once per
 * parameter update.
 * sample_mode: QS_SAMPLE_MEAN   deterministic actions (model.predict(deterministic=True), runsim_scaledObs.py:54)
 *              QS_SAMPLE_NOISE  a = mean + exp(log_std) * noise[n,4]   (caller-supplied standard normal draws)
 *              QS_SAMPLE_PHILOX the kernel draws the noise itself: Philox4x32-10 keyed on noise_seed, counter = (global env id,
 *                               *noise_step), Box-Muller; *noise_step (device u64) is incremented once per launch, so a captured
 *                               CUDA graph replays fresh noise and a batch sharded over ranks draws what the unsharded batch would
 */
#define QS_SAMPLE_MEAN 0
#define QS_SAMPLE_NOISE 1
#define QS_SAMPLE_PHILOX 2
typedef struct qs_rollout_args {
    const void* policy_image;     /* qs_policy_prepare output */
    const float* obs;             /* f32[n,D] raw observations of the current states (qs_reset / the previous obs_next) */
    const double* norm_stats;     /* VecNormalize stats f64[1+2D] applied to obs before the policy, or NULL */
    float norm_eps, norm_clip;
    int32_t sample_mode;          /* QS_SAMPLE_* */
    int32_t reserved;
    const float* noise;           /* f32[n,4], QS_SAMPLE_NOISE */
    uint64_t noise_seed;          /* QS_SAMPLE_PHILOX */
    uint64_t* noise_step;         /* QS_SAMPLE_PHILOX: device counter word */
    float clip_lo[4], clip_hi[4]; /* action box (SB3 clips before env.step) */
    float* obs_norm_out;          /* f32[n,D] or NULL: the normalised observations the policy saw (RolloutBuffer.observations) */
    float* actions_out;           /* f32[n,4] sampled, unclipped (RolloutBuffer.actions) */
    float* actions_clipped_out;   /* f32[n,4] or NULL: what the envs were stepped with */
    float* values_out;            /* f32[n] */
    float* logp_out;              /* f32[n] */
    float* obs_next;              /* f32[n,D] observations after the step (reset obs where done); may alias obs */
    float* reward_out;            /* f32[n] */
    uint8_t* flags_out;           /* u8[n] QS_FLAG_* */
    float* terminal_obs_out;      /* f32[n,D] or NULL, rows of done envs */
    float* ep_return_out;         /* f32[n] or NULL, rows of done envs */
    int32_t* ep_len_out;          /* i32[n] or NULL, rows of done envs */
} qs_rollout_args;
int64_t qs_policy_image_bytes(void);
int qs_policy_prepare(const float* params, int obs_dim, void* image_out, void* stream);
int qs_rollout_step(qs_handle* h, const qs_rollout_args* a, void* stream);
/* 0, or the code of the internal hand-over that timed out (every in-kernel wait is bounded; synchronises the device, clears) */
int qs_rollout_status(void);

/* Generalized advantage estimation ------------------------------------------------------------------
 * Replaces stable_baselines3 RolloutBuffer.compute_returns_and_advantage (inside model.learn(), reference call sites
 * initial-implementation-v1/rl_train_vecN.py:36, initial-implementation-v2/rl_train.py:56; gamma 0.995, gae_lambda 0.9).
 * All buffers time-major [T, n] on the device: rewards/values f32, episode_starts u8 (1 where the env was reset before step t),
 * last_values f32[n] / last_dones u8[n] for the state after the last step.  Writes advantages and returns f32[T, n].
 */
int qs_gae(const float* rewards, const float* values, const uint8_t* episode_starts, const float* last_values,
           const uint8_t* last_dones, int T, int64_t n, float gamma, float gae_lambda, float* advantages, float* returns,
           void* stream);
const char* qs_gae_last_error(void);
/* RolloutBuffer.add for one collection step of all envs, with the buffer slot t (0 <= t < T) read from DEVICE memory so that a captured
 * CUDA graph of the step can be replayed (SB3 OnPolicyAlgorithm.collect_rollouts around env.step; reference call sites
 * initial-implementation-v1/rl_train_vecN.py:36, initial-implementation-v2/rl_train.py:56).  Time-major buffers [T, n, ...].
 *   qs_rollout_record_pre:  obs_buf[t] = obs (f32[n,D], already normalised if VecNormalize is on), actions_buf[t] = the UNclipped
 *     actions (f32[n,4]), values_buf[t], logp_buf[t], episode_starts_buf[t] = last_dones (u8[n]).
 *   qs_rollout_record_post: rewards_buf[t] = reward (f32 or f64 source; if ret_var != NULL first VecNormalize.normalize_reward:
 *     clip(reward / sqrt(ret_var[0] + epsilon), +-clip_reward)), plus gamma * terminal_values for envs whose flags say truncated and
 *     not terminated (TimeLimit.truncated bootstrap); last_dones = terminated | truncated; ep_stats[0] += sum of ep_return over the
 *     finished envs, ep_stats[1] += their number (f64[2], fixed summation order); *t_dev += 1.
 *     workspace: f64[2 * QS_RECORD_MAX_BLOCKS + 1], zero before the first call. */
#define QS_RECORD_MAX_BLOCKS 1024
int qs_rollout_record_pre(const long long* t_dev, int64_t n, int obs_dim, const float* obs, const float* actions, const float* values,
                          const float* logp, const uint8_t* last_dones, float* obs_buf, float* actions_buf, float* values_buf,
                          float* logp_buf, uint8_t* episode_starts_buf, void* stream);
int qs_rollout_record_post(long long* t_dev, int64_t n, const void* reward, int reward_is_f64, const uint8_t* flags, const void* ep_return,
                           const float* terminal_values, float gamma, const double* ret_var, double epsilon, float clip_reward,
                           float* rewards_buf, uint8_t* last_dones, double* ep_stats, double* workspace, void* stream);

/* PPO minibatch update -----------------------------------------------------------------------------------
 * Replaces one minibatch of stable_baselines3 PPO.train() (inside model.learn(); reference call sites
 * initial-implementation-v1/rl_train_vecN.py:13-36 -- batch_size 128, n_epochs 10, clip_range 0.2, ent_coef 0.01, lr 2e-4 -- and
 * initial-implementation-v2/rl_train.py:38-56): advantage normalisation over the minibatch, evaluate_actions of the
 * [128, 64, 64] Tanh actor and critic, clipped surrogate + vf_coef * MSE + ent_coef * entropy loss, backward, global-norm
 * clipping, torch.optim.Adam(eps 1e-5) -- ONE kernel launch, float32, deterministic (fixed reduction order).
 *   params        device f32[qs_ppo_n_params(obs_dim)], the qs_policy_forward blob; updated in place
 *   obs/actions/old_logp/advantages/returns   flat device rollout buffers f32[total, obs_dim] / [total, 4] / [total] x 3
 *   idx           device i64[B] rows of this minibatch (a slice of the epoch's permutation), or NULL = rows 0..B-1
 *   stats_out     device f32[8] or NULL: loss, policy_gradient_loss, value_loss, entropy_loss, grad_norm (before clipping),
 *                 clip_fraction, approx_kl, B
 * The handle owns the Adam moments and step count (device resident: the call is CUDA-graph capturable).  Several ranks:
 * qs_ppo_grad (gradient of the local minibatch -> grad_out f32[n_params], or the handle's own buffer if NULL), average over
 * ranks (NCCL all-reduce), qs_ppo_apply (clipping + Adam on the averaged gradient; grad NULL = the handle's buffer).
 */
typedef struct qs_ppo qs_ppo;
typedef struct qs_ppo_hyper {
    float clip_range, ent_coef, vf_coef, max_grad_norm;
    float lr, beta1, beta2, adam_eps;
    int32_t normalize_advantage, reserved;
} qs_ppo_hyper;
void qs_ppo_default_hyper(qs_ppo_hyper* hp); /* SB3 defaults: 0.2, 0, 0.5, 0.5, 3e-4, 0.9, 0.999, 1e-5, normalise */
int qs_ppo_n_params(int obs_dim);            /* floats in the parameter blob (17 or 20 observations), -1 otherwise */
int qs_ppo_create(int device, int obs_dim, qs_ppo** out);
int qs_ppo_destroy(qs_ppo* o);
int qs_ppo_update(qs_ppo* o, float* params, const float* obs, const float* actions, const float* old_logp,
                  const float* advantages, const float* returns, const int64_t* idx, int64_t B, const qs_ppo_hyper* hp,
                  float* stats_out, void* stream);
int qs_ppo_grad(qs_ppo* o, const float* params, const float* obs, const float* actions, const float* old_logp,
                const float* advantages, const float* returns, const int64_t* idx, int64_t B, const qs_ppo_hyper* hp,
                float* grad_out, float* stats_out, void* stream);
int qs_ppo_apply(qs_ppo* o, float* params, const float* grad, const qs_ppo_hyper* hp, float* stats_out, void* stream);
/* device pointers of the optimizer state (checkpointing, tests): Adam m, v f32[n_params], step i64[1], gradient buffer */
int qs_ppo_state(qs_ppo* o, float** m, float** v, long long** step, float** grad);
const char* qs_ppo_last_error(void);

/* Peer-memory exchange of the VecNormalize moments (multi-GPU) --------------------------------------------
 * The only exchange step of the sharded env path is the 2d+1 doubles (n, mean[d], M2[d]) each rank contributes to the running
 * statistics per step.  qs_xchg_merge is that all-gather FUSED with the Chan merge in one kernel over NVLink peer memory: the
 * rank stores its triplet straight into a slot of every peer's exchange buffer (P2P stores, release flag), waits until the
 * slots of its own buffer carry this step's sequence number, and merges them in rank order into `stats` -- bit-identical on
 * all ranks, no NCCL call, one launch, safe to capture in a CUDA graph (the sequence number lives on the device).
 * Setup: every rank calls qs_xchg_create (allocates its buffer, returns a 64-byte CUDA IPC handle), the ranks exchange the
 * handles by any host channel (torch.distributed.all_gather_object), then qs_xchg_connect maps the peers' buffers.
 * All ranks must call qs_xchg_merge the same number of times; a rank that waits longer than ~10 s on a peer gives up, sets a
 * sticky error (qs_xchg_failed() != 0) and merges what has arrived, so a dead peer cannot hang the GPU.
 * The NCCL path (all_gather_into_tensor + qs_vecnorm_merge) stays available and is the one the gloo CPU tests cover.
 */
typedef struct qs_xchg qs_xchg;
int qs_xchg_create(int device, int rank, int world, int d, qs_xchg** out, unsigned char* ipc_handle_out /*[64]*/);
int qs_xchg_connect(qs_xchg* x, const unsigned char* all_handles /*[world][64], rank order*/);
int qs_xchg_merge(qs_xchg* x, double* stats, const double* local_moments, void* stream);
int qs_xchg_failed(qs_xchg* x);   /* synchronises the device; 1 if any merge timed out */
/* Sharded rollout: arm the env handle so that the kernel which finishes the fused observation moments of every qs_step
 * (qs_step_moments must be armed) ALSO runs the exchange and the merge into `stats` (f64[1+2D]) in the same launch -- what a
 * qs_xchg_merge(x, stats, moments_out) right after the step would do, one kernel boundary earlier (the step -> exchange ->
 * policy chain of SB3's collect_rollouts ends at the slowest rank, so every boundary on it is paid in full).  All ranks arm
 * it alike; it counts as one qs_xchg_merge per qs_step.  x == NULL disarms.  Replaces, with qs_step, VecNormalize.step_wait's
 * obs_rms.update over the whole sharded batch (reference call site initial-implementation-v1/rl_train_vecN.py:11). */
int qs_step_moments_exchange(qs_handle* h, qs_xchg* x, double* stats);
int qs_xchg_destroy(qs_xchg* x);
const char* qs_xchg_last_error(void);

/* Batched PID baseline controller ----------------------------------------------------------------------
 * Replaces `run(quad, des_state, dt)` of initial-implementation-v2/PID Controller/pid_controller.py:37-115 for all envs of a
 * handle at once: position PID -> commanded acceleration -> thrust F and desired roll/pitch; attitude PID -> moments M.
 * The reference keeps one module-level `integral_error` dict (:24-31); here the six integrals per env are a caller-owned
 * buffer, updated in place (clamped to +-max_integral like :65-66, :105-106).  The vehicle state (position, velocity,
 * quaternion, body rates) is read from the handle's state pool; the attitude is RotToRPY of the Rodrigues matrix like
 * Quadcopter.attitude() (PID Controller/model/quadcopter.py:58-60).  All arithmetic is float64.
 * Gains in the order x, y, z, phi, theta, psi; qs_pid_default_gains() writes the reference's (:16-22, :34).
 * Desired state: des_pos f64[n,3] or NULL = each env's current waypoint (hover target); des_vel / des_acc f64[n,3] and
 * des_yaw / des_yawdot f64[n], NULL = zeros (des_yaw NULL on a v2 handle = the env's final_yaw).
 * Outputs (each optional): wrench_out f64[n,4] = (F, M1, M2, M3) exactly as the reference returns them; actions_out f32[n,4] =
 * the env action that commands this wrench, a0 = F/(mass*g), a[1:4] = M/0.1 (inverse of rl_env_scaledObs.py:125-126), clipped
 * to the action box [0,2]x[-1,1]^3 when clip_actions != 0 -- feed it to qs_step.
 */
typedef struct qs_pid_gains {
    double kp[6], kd[6], ki[6];
    double max_integral;
} qs_pid_gains;
void qs_pid_default_gains(qs_pid_gains* out);
int qs_pid_run(qs_handle* h, const qs_pid_gains* gains, double dt, const double* des_pos, const double* des_vel,
               const double* des_acc, const double* des_yaw, const double* des_yawdot, double* integral,
               double* wrench_out, float* actions_out, int clip_actions, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* QUADSIM_H */
