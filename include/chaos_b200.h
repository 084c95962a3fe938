/* chaos_b200.h -- C ABI of the B200-native batched chaos-control environments.
 *
 * This is the drop-in boundary for the ONE hot path of erererq/gym-lorenz: the env
 * `step` (ODE integration -> reward -> termination -> auto-reset).  Each entry point
 * names the reference interface it replaces (paths relative to
 * /root/reference/code/gym-lorenz/gym_lorenz/envs/ unless stated otherwise).
 *
 * Conventions
 *   - every function returns 0 on success or a negative CL_E* code;
 *     cl_last_error(ctx) returns a message owned by the context (or a static string).
 *   - the library never allocates user-visible memory: all state / io buffers are
 *     allocated by the caller (PyTorch) and passed as raw pointers.  Device entry
 *     points only ENQUEUE on the given cudaStream_t and return; they never synchronise.
 *     The *_host entry points take HOST pointers, perform the H2D / D2H copies through
 *     context-owned pinned staging and return after the stream has drained.
 *   - a context is not thread-safe; one context per (process, GPU, env batch).
 *   - layout: structure-of-arrays planes `plane[c][n_pad]`; n_pad >= num_envs and a
 *     multiple of 128.  Actions and observations are addressed through
 *     (env_stride, comp_stride) element strides so that both SoA planes
 *     (1, n_pad) and policy-shaped [N, C] row-major tensors (C, 1) are zero-copy.
 */
#ifndef CHAOS_B200_H
#define CHAOS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CL_ABI_VERSION 1

/* ---- error codes ------------------------------------------------------------------ */
#define CL_OK 0
#define CL_EINVAL (-1)   /* bad argument / unsupported combination */
#define CL_ECUDA (-2)    /* CUDA runtime error (message in cl_last_error) */
#define CL_ENOMEM (-3)
#define CL_ENODEV (-4)   /* no sm_100 device / device ordinal out of range */

/* ---- env kinds -------------------------------------------------------------------- */
typedef enum cl_env_kind {
  /* parity kinds: the reference's own scheme, dtype rules and quirks, bit-for-bit */
  CL_ENV_LORENZ3 = 0,      /* dynamic.py:5-93    3-D Lorenz to origin, Euler dt .01, f64 */
  CL_ENV_LORENZ3_PAIR = 1, /* dynamic.py:109-233 nested class, frozen target system     */
  CL_ENV_LORENZ4_PAIR = 2, /* lorenz_env_transient.py:247-376  4-D pair, Euler dt .001  */
  CL_ENV_HR_SYNC = 3,      /* lorenz_env_try.py:7-179  Hindmarsh-Rose pair, RK4 dt .001 */
  CL_ENV_PMSM_SYNC = 4,    /* lorenz_env_try_pmsm.py:7-184  PMSM pair, f32 Euler + Adam */
  CL_ENV_PMSM_CLASSIC = 5, /* lorenz_env_transient_pmsm.py:17-137  f64 Euler dt .01     */
  CL_ENV_PMSM_SINGLE = 6,  /* lorenz_env_transient1.py  single PMSM to origin           */
  /* north-star kinds: RK4 x S substeps per control interval, zero-order-hold control in
   * the derivative, per-env parameters (BASELINE.json north_star; SURVEY.md D1-D3) */
  CL_ENV_LORENZ_RK4 = 7,     /* f64 */
  CL_ENV_LORENZ_RK4_F32 = 8, /* f32 */
  CL_ENV_PMSM_RK4 = 9,       /* f64 PMSM pair, per-env sigma/gamma */
  /* further parity kinds (SURVEY 8f rank 4) */
  CL_ENV_MEMRISTIVE4_PAIR = 10, /* lorenz_env_transient2.py  4-D memristive pair, u*100 control */
  CL_ENV_PMSM_FREE = 11,        /* lorenz_singlecontrol.py   uncontrolled noisy PMSM, fixed IC  */
  CL_ENV_KIND_COUNT = 12
} cl_env_kind;

/* ---- flags ------------------------------------------------------------------------ */
#define CL_F_ADD_NOISE 0x01  /* HRSyncEnv(add_noise) / PMSM_Sync_Env(add_noise)          */
#define CL_F_EVAL_MODE 0x02  /* HRSyncEnv(eval_mode): sigma locked to 2.0                */
#define CL_F_ADD_FILTER 0x04 /* HRSyncEnv(add_filter): action low-pass alpha=.95         */
#define CL_F_AUTORESET 0x08  /* SB3 DummyVecEnv.step_wait semantics: reset finished envs */
#define CL_F_OBS_F64 0x10    /* emit observations as f64 (classic envs return f64 obs)   */

/* ---- statistics vector (cl_stats / cl_buffers.stats), 8 doubles -------------------- */
#define CL_STAT_EPISODES 0   /* finished episodes                       */
#define CL_STAT_RET_SUM 1    /* sum of episode returns                  */
#define CL_STAT_RET_SQ 2     /* sum of squared episode returns          */
#define CL_STAT_LEN_SUM 3    /* sum of episode lengths                  */
#define CL_STAT_NONFINITE 4  /* divergence events: env-steps that turned a finite state non-finite */
#define CL_STAT_TERMINATED 5 /* episodes ended by the env's own guard   */
#define CL_STAT_TRUNCATED 6  /* episodes ended by the TimeLimit         */
#define CL_STAT_RESERVED 7
#define CL_NSTATS 8

/* done-flag bits written to cl_io.done */
#define CL_DONE_TERMINATED 0x1
#define CL_DONE_TRUNCATED 0x2

typedef struct cl_config {
  int32_t abi_version;       /* CL_ABI_VERSION */
  int32_t kind;              /* cl_env_kind */
  int32_t device;            /* CUDA device ordinal */
  int32_t flags;             /* CL_F_* */
  int64_t num_envs;          /* envs in this slab */
  int64_t n_pad;             /* plane stride, multiple of 128, >= num_envs */
  int64_t env_id_base;       /* global index of local env 0 (rank * num_envs) */
  uint64_t seed;             /* Philox key */
  int32_t max_episode_steps; /* gymnasium TimeLimit (gym_lorenz/__init__.py:12,20); 0 = none */
  int32_t substeps;          /* RK4 substeps per control interval (north-star kinds) */
  double dt;                 /* control interval (north-star kinds; parity kinds ignore) */
  double alpha;              /* PMSM_Sync_Env(alpha) reward exponent */
  double act_limit;          /* north-star: |u| clip */
  double act_gain;           /* north-star: u = clip(a) * gain */
  double param_jitter;       /* north-star: per-env params ~ nominal * U(1-j, 1+j) on cl_reset */
} cl_config;

/* Per-kind buffer geometry (what the caller must allocate). */
typedef struct cl_layout {
  int32_t real_bytes;   /* 8 (f64 kinds) or 4 (f32 kinds): dtype of state and reward */
  int32_t n_state;      /* number of real-typed state planes */
  int32_t n_int;        /* number of int32 aux planes (PMSM_SYNC: adam_step) */
  int32_t obs_dim;
  int32_t act_dim;
  int32_t noise_dim;    /* standard-normal draws consumed per env-step (0 if none) */
  double act_low, act_high;     /* action_space bounds of the reference env */
  double obs_low, obs_high;     /* observation_space bounds (+-inf -> +-HUGE_VAL) */
  int32_t default_max_episode_steps;
  int32_t reserved;
} cl_layout;

/* Persistent per-env device buffers (caller-allocated, library never frees). */
typedef struct cl_buffers {
  void* state;        /* real [n_state][n_pad] */
  int32_t* aux_int;   /* int32 [n_int][n_pad] (may be NULL when n_int == 0) */
  int32_t* ep_len;    /* int32 [n_pad]: steps since reset (TimeLimit counter) */
  double* ep_return;  /* f64 [n_pad]: return accumulated since reset (SB3 Monitor) */
  double* stats;      /* f64 [CL_NSTATS], accumulated with atomics */
} cl_buffers;

/* Per-call io (device pointers for cl_step/cl_reset/cl_rollout). */
typedef struct cl_io {
  const float* action;   /* f32, element (env i, comp c) at action[i*act_es + c*act_cs] */
  int64_t act_es, act_cs;
  const double* noise;   /* optional f64 [noise_dim][n_pad] standard-normal override
                            (parity tests inject the oracle's draws); NULL -> Philox */
  void* obs;             /* f32 (f64 with CL_F_OBS_F64): obs[i*obs_es + c*obs_cs] */
  int64_t obs_es, obs_cs;
  void* reward;          /* real [n_pad] */
  uint8_t* done;         /* u8 [n_pad], CL_DONE_* bits */
  void* term_obs;        /* optional, same addressing as obs; written only where done
                            (SB3 infos[i]["terminal_observation"]) */
  double* last_ep_ret;   /* optional f64 [n_pad]; written only where done (Monitor "r") */
  int32_t* last_ep_len;  /* optional i32 [n_pad]; written only where done (Monitor "l") */
  const uint8_t* mask;   /* cl_reset only: optional u8 [n_pad], reset where != 0 */
} cl_io;

/* Fused multi-step rollout geometry: T control intervals per launch.  Time-major
 * buffers; element strides between consecutive steps.  Any output pointer in `io` may be
 * NULL to skip that stream.  If io.action is NULL, actions are drawn in-kernel from
 * Philox: a ~ U(-synth_amp, synth_amp) per component. */
typedef struct cl_rollout_desc {
  int32_t T;
  int32_t reserved;
  int64_t act_ts;     /* elements between action[t] and action[t+1] */
  int64_t obs_ts;     /* elements between obs[t] and obs[t+1] */
  int64_t rew_ts;     /* elements between reward[t] and reward[t+1] */
  int64_t done_ts;    /* bytes between done[t] and done[t+1] */
  double synth_amp;
} cl_rollout_desc;

typedef struct cl_ctx cl_ctx;

/* -- lifecycle.  Replaces: env construction (`gymnasium.make(id, **kw)` ->
 *    HRSyncEnv.__init__ lorenz_env_try.py:19-43, PMSM_Sync_Env.__init__
 *    lorenz_env_try_pmsm.py:9-50, lorenzEnv_transient.__init__ dynamic.py:8-33). */
int cl_abi_version(void);
int cl_env_layout(int32_t kind, cl_layout* out);
int cl_create(const cl_config* cfg, cl_ctx** out);
int cl_destroy(cl_ctx* ctx);
const char* cl_last_error(const cl_ctx* ctx);

/* -- reset.  Replaces `env.reset()` (dynamic.py:35-47,142-158;
 *    lorenz_env_transient.py:275-297; lorenz_env_try.py:49-78;
 *    lorenz_env_try_pmsm.py:59-75; lorenz_env_transient_pmsm.py:43-62).
 *    Draws initial conditions from Philox (subsequence = global env id), zeroes the
 *    per-episode counters and writes the reset observation.  io.mask selects envs
 *    (NULL = all).  Persistent cross-episode state (PMSM_SYNC lambda/m_t/v_t/adam_step)
 *    is NOT touched, exactly as in lorenz_env_try_pmsm.py:59-75. */
int cl_reset(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io);

/* -- initialise persistent state that survives reset (PMSM_SYNC Adam-dual state := 0,
 *    north-star per-env parameters := nominal * jitter).  Replaces the constructor
 *    bodies cited at cl_create. */
int cl_init_persistent(cl_ctx* ctx, void* stream, const cl_buffers* buf);

/* -- one control interval for every env.  Replaces `env.step(a)`
 *    (dynamic.py:61-90,174-230; lorenz_env_transient.py:314-373;
 *    lorenz_env_try.py:80-179; lorenz_env_try_pmsm.py:76-184;
 *    lorenz_env_transient_pmsm.py:76-133; lorenz_env_transient1.py:69-104) plus the
 *    TimeLimit / auto-reset / Monitor bookkeeping of SB3 DummyVecEnv.step_wait
 *    (call sites code/train.py:100, code/lorenz_pmsm/train.py:115-118). */
int cl_step(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io);

/* -- T fused control intervals, state held in registers across all of them.  Replaces
 *    the SB3 collect_rollouts env loop (code/train.py:120 -> OnPolicyAlgorithm
 *    .collect_rollouts) for synthetic / pre-computed action sequences. */
int cl_rollout(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
               const cl_rollout_desc* desc);

/* -- policy evaluation on the device.  Replaces the predict loop of the reference's evaluation
 *    scripts (code/test_evaluate.py, code/lorenz_pmsm/test_evaluate.py: frozen VecNormalize,
 *    model.predict(obs, deterministic=True) every step, then the metrics of cl_eval_metrics):
 *    a stable-baselines3 MlpPolicy (pi = [64, 64], Tanh, linear action_net; float32) runs inside
 *    the fused rollout of CL_ENV_HR_SYNC / CL_ENV_PMSM_SYNC, one launch for T control intervals.
 *    Per interval: z = clip((obs - mean) / sqrt(var + epsilon), +-clip_obs) as f32 (skipped when
 *    obs_mean is NULL) -> a = W3 tanh(W2 tanh(W1 z + b1) + b2) + b3 -> clip to the action box ->
 *    the env step cl_rollout runs with the same Philox step index.  io / desc carry the optional
 *    obs / reward / done streams exactly as in cl_rollout; io.action must be NULL.  The metrics use
 *    err_t = obs components 0..2 after interval t (as the f32 the policy sees next), ctrl_t = the
 *    clipped action; state, episode counters and the step index advance as in cl_rollout. */
#define CL_POLICY_HIDDEN 64   /* two hidden layers of this width (SB3 MlpPolicy default) */
typedef struct cl_policy {
  const float* params;      /* device f32, torch Linear layout: W1[64][obs_dim] b1[64] W2[64][64] b2[64]
                               W3[act_dim][64] b3[act_dim] */
  const double* obs_mean;   /* device f64 [obs_dim]; NULL = no normalisation */
  const double* obs_var;    /* device f64 [obs_dim] */
  double epsilon, clip_obs;
  const float* obs0;        /* device f32: observation interval 0 acts on, obs0[i*obs0_es + c*obs0_cs] */
  int64_t obs0_es, obs0_cs;
  float* obs_last;          /* optional device f32, same addressing: observation after the last interval
                               (may alias obs0) */
  float* act_out;           /* optional device f32 [T][n][act_dim]: the clipped actions applied */
  double* metrics;          /* optional device f64 [n][4]: mae, rmse, settling_time, energy */
  int32_t steady_start;
  double dt, error_band;
} cl_policy;
int cl_policy_rollout(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
                      const cl_rollout_desc* desc, const cl_policy* pol);

/* -- rollout collection for PPO / A2C on the device.  Replaces stable-baselines3's
 *    OnPolicyAlgorithm.collect_rollouts (code/train.py: PPO, n_steps 2048; code/lorenz_pmsm/train.py: A2C)
 *    for an ActorCriticPolicy (pi = vf = [64, 64], Tanh, Gaussian actions with state-independent
 *    log_std; float32) on CL_ENV_HR_SYNC / CL_ENV_PMSM_SYNC, one launch for T control intervals.
 *    pol.params is the actor-critic block: the actor block of cl_policy_rollout first, then
 *    V1[64][obs_dim] c1[64] V2[64][64] c2[64] Wv[1][64] bv[1], then log_std[act_dim].  pol.act_out and
 *    pol.metrics must be NULL.  Per interval t, env i (all f32 unless stated):
 *      1. z = obs, or clip((obs - mean) / sqrt(var + epsilon), +-clip_obs) in f64 rounded to f32 with
 *         obs_mean set (the frozen VecNormalize of cl_policy_rollout);
 *      2. mu = W3 tanh(W2 tanh(W1 z + b1) + b2) + b3   (cl_policy_rollout's MLP, explicit fmaf);
 *      3. V  = Wv tanh(V2 tanh(V1 z + c1) + c2) + bv   (same code, same fmaf order);
 *      4. eps_c = (float) the f64 Box-Muller normal of Philox block (env id, step index, TAG_POLICY),
 *         std = expf(log_std), a = fmaf(std, eps, mu);
 *      5. log_prob = sum_c -(a - mu)^2 / (2 std^2) - log(std) - log(sqrt(2 pi))   (torch Normal.log_prob);
 *      6. the env step of cl_rollout with clip(a, act_low, act_high) and the same Philox step index;
 *      7. reward = (float)r; where the step truncated without terminating,
 *         reward += (float)gamma * V(z_term), z_term the pre-reset observation normalised as in 1;
 *      8. obs[t][i] = z, actions[t][i] = a (unclipped), rewards[t][i], values[t][i] = V,
 *         log_probs[t][i], episode_starts[t][i] = starts[i]; then starts[i] = (done flags != 0).
 *    After the last interval: last_values[i] = V(z of the last observation), starts[i] as carried,
 *    pol.obs_last (if set) = the last raw observation; state, episode counters, statistics and the
 *    step index advance as in cl_rollout.  io / desc carry optional obs / reward / done streams as in
 *    cl_rollout; io.action and io.noise must be NULL.  Buffers are row-major with n = num_envs rows. */
typedef struct cl_collect {
  double gamma;
  float* starts;            /* device f32 [n], in/out: episode starts carried between windows */
  float* obs;               /* device f32 [T][n][obs_dim] */
  float* actions;           /* device f32 [T][n][act_dim] */
  float* rewards;           /* device f32 [T][n] */
  float* values;            /* device f32 [T][n] */
  float* log_probs;         /* device f32 [T][n] */
  float* episode_starts;    /* device f32 [T][n] */
  float* last_values;       /* device f32 [n] */
} cl_collect;
int cl_policy_collect(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
                      const cl_rollout_desc* desc, const cl_policy* pol, const cl_collect* col);

/* -- cl_policy_collect behind a VecNormalize in training mode (code/lorenz_pmsm/train.py: A2C through
 *    VecNormalize(norm_obs=True, norm_reward=False, clip_obs=10), training=True): the running statistics
 *    are updated inside the launch, as SB3's VecNormalize.step_wait does every step.  One cooperative
 *    launch; every interval ends with a grid-wide barrier, so the batch statistics of interval t are
 *    reduced over all n envs before any env normalises its next observation.  The reduction sums the
 *    per-block partial sums in block order in every block: the result is bit-reproducible run to run.
 *    Refused, besides what cl_policy_collect refuses: pol.obs_mean set (the statistics come from vn
 *    alone), pol.obs_last NULL (the raw observation is carried there between intervals), missing
 *    statistics (obs_* only with norm_obs) or returns, scratch smaller than
 *    cl_policy_collect_norm_scratch_bytes.  Per interval t, env i, after steps 2-6 of cl_policy_collect
 *    (actor, critic, sample, log-prob, env step) on z_t:
 *      1. o = the raw next observation (f32), r = the raw reward, the done flags, o_term = the pre-reset
 *         observation;
 *      2. norm_obs: obs_rms.update(o over all n envs) with cl_obs_moments + cl_rms_update's arithmetic:
 *         f64 sums of (o - mean_old) and (o - mean_old)^2, then the merge of cl_rms_update statement for
 *         statement; obs_count += n (one f64 addition per interval);
 *      3. returns[i] = returns[i] * gamma + (double)r (two roundings), then ret_rms.update(returns over
 *         all n envs) with cl_moments_f64's arithmetic and the same merge -- also with norm_reward = 0;
 *      4. reward = (float)r, or with norm_reward (float)clip((double)r / sqrt(ret_var + epsilon),
 *         +-clip_reward), ret_var the updated one; where the step truncated without terminating,
 *         reward += (float)col.gamma * V(z_term);
 *      5. z_{t+1} = clip((o - mean) / sqrt(var + epsilon), +-clip_obs) in f64 rounded to f32 with the
 *         updated obs_rms (z = o without norm_obs); z_term the same of o_term;
 *      6. returns[i] = 0 where done.
 *    z_0 is the observation in pol.obs0 normalised with the statistics passed in.  After the last
 *    interval the statistics and returns hold their updated values, pol.obs_last the last raw
 *    observation, last_values V(z_T).  io.obs / reward / done, when set, stream the raw env outputs. */
typedef struct cl_vecnorm_update {
  double* obs_mean;         /* device f64 [obs_dim], in/out (norm_obs only) */
  double* obs_var;          /* device f64 [obs_dim], in/out (norm_obs only) */
  double* obs_count;        /* device f64 [1], in/out (norm_obs only) */
  double* ret_mean;         /* device f64 [1], in/out */
  double* ret_var;          /* device f64 [1], in/out */
  double* ret_count;        /* device f64 [1], in/out */
  double* returns;          /* device f64 [n], in/out: the discounted returns VecNormalize carries */
  double gamma, epsilon, clip_obs, clip_reward;
  int32_t norm_obs, norm_reward;
  void* scratch;            /* device, caller-owned (nothing is allocated during a CUDA-graph capture) */
  int64_t scratch_bytes;
} cl_vecnorm_update;
int cl_policy_collect_norm(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
                           const cl_rollout_desc* desc, const cl_policy* pol, const cl_collect* col,
                           const cl_vecnorm_update* vn);
/* scratch cl_policy_collect_norm needs for n envs of `kind` (a function of kind and n alone: it can be
 * sized without a device): two interval-parity slots of per-block partial sums plus, per env, the raw
 * reward, done flags and pre-reset observation an interval hands to the next one across the barrier */
int cl_policy_collect_norm_scratch_bytes(int32_t kind, int64_t n, int64_t* out);

/* -- derivative helper used by the reference's evaluation script
 *    (code/lorenz_pmsm/test_evaluate.py:105-108 -> PMSM_Sync_Env._get_derivatives,
 *    lorenz_env_try_pmsm.py:51-58; hr_derivatives lorenz_env_try.py:7-12).
 *    state: real [state_dim_of_one_system][n], action f32 [act_dim][n] (SoA, stride n),
 *    out: real [3 or 4][n]. */
int cl_derivatives(cl_ctx* ctx, void* stream, const void* state, const float* action,
                   void* out, int64_t n);

/* -- statistics.  Copies the CL_NSTATS vector device->device into out8 (stream
 *    ordered) and optionally clears the accumulator. */
int cl_stats(cl_ctx* ctx, void* stream, const cl_buffers* buf, double* out8, int clear);

/* -- global step index that keys the Philox streams (checkpoint / resume). */
int cl_get_step_index(const cl_ctx* ctx, uint64_t* out);
int cl_set_step_index(cl_ctx* ctx, uint64_t value);

/* -- CUDA-graph mode.  When enabled, the Philox step index lives in device memory and is advanced
 *    by a one-thread kernel enqueued right after each env kernel, so cl_step / cl_rollout / cl_reset can be
 *    captured into a CUDA graph (e.g. torch.cuda.graph) and REPLAYED: every replay sees a fresh
 *    step index.  All scratch is allocated at cl_create, nothing allocates during capture.
 *    cl_get_step_index then synchronises the device. */
int cl_set_graph_mode(cl_ctx* ctx, int enable);

/* -- HOST-buffer path (the SB3 VecEnv numpy contract: step_async / step_wait;
 *    SB3 DummyVecEnv.step_async/step_wait, call sites code/train.py:100,
 *    code/lorenz_pmsm/train.py:115-118).
 *    action_host: f32 [num_envs][act_dim] row-major (what SB3 passes to step_async), or
 *    NULL when the caller already wrote the actions into the pinned staging area returned
 *    by cl_host_action_staging.  cl_step_host_async enqueues H2D, the step kernel and the
 *    D2H copies on `stream` ((void*)-1 = the context's own non-blocking stream);
 *    cl_step_host_wait synchronises that stream and copies obs f32 [num_envs][obs_dim],
 *    reward f32 [num_envs], done u8 [num_envs] (CL_DONE_* bits) out of pinned memory
 *    (any destination may be NULL).  term_obs / last_ep_* are filled only when n_done > 0.
 *    cl_step_host_wait_view is the zero-copy variant: it returns pointers into a ring of
 *    3 pinned result slots; a slot stays valid for the next 2 steps (SB3's
 *    collect_rollouts reads the previous obs after the following step). */
typedef struct cl_host_view {
  float* obs;            /* [num_envs][obs_dim] */
  float* reward;         /* [num_envs] */
  uint8_t* done;         /* [num_envs] */
  float* term_obs;       /* [num_envs][obs_dim], valid where done (only if n_done > 0) */
  double* last_ep_ret;   /* [num_envs], valid where done */
  int32_t* last_ep_len;  /* [num_envs], valid where done */
  int64_t n_done;
} cl_host_view;
int cl_host_action_staging(cl_ctx* ctx, float** action_pinned);
/* zero-copy variant of the host path: the step kernel reads actions from / writes results to the
 * pinned (UVA-mapped) host buffers directly instead of DMA copies around it */
int cl_host_set_zero_copy(cl_ctx* ctx, int enable);
/* how cl_step_host_async moves the data (default: STREAMED with one slice per 2,048 envs from 96 KB of
 * actions per step, ZEROCOPY below; chosen by host_mode_default() in csrc/chaos_b200.cu from the measured
 * tables profiles/r02f4_e2e_small_ab.jsonl, r02f3_e2e_host_modes.jsonl; CHAOS_B200_HOST_MODE=dma|zerocopy|pipelined|streamed overrides):
 *   CL_HOST_DMA        H2D copy of the actions -> step kernel -> one D2H copy of obs|reward|done
 *   CL_HOST_ZEROCOPY   one launch; the kernel reads / writes the pinned host buffers itself
 *   CL_HOST_PIPELINED  `slices` env slices alternate over two streams: per slice a DMA copy of its
 *                      actions, then its step kernel writing the results to pinned host memory, so
 *                      upstream and downstream PCIe traffic of neighbouring slices overlap.
 *   CL_HOST_STREAMED   ZEROCOPY whose single launch is issued BEFORE the caller's action array is staged
 *                      into pinned memory: up to four staging lanes (copy threads, CHAOS_B200_COPY_THREADS)
 *                      publish the buffer slice by slice (generation words in pinned memory, one per
 *                      lane), block 0 of the kernel mirrors those words into device memory and each
 *                      other block waits for the slice it reads, so the host memcpy, the launch latency
 *                      and the PCIe traffic of the slices already published overlap.  Falls back to ZEROCOPY when the caller
 *                      passes the pinned staging buffer itself or the context is in graph mode.
 * Results are identical in all modes (same kernel, same per-env Philox streams). */
enum { CL_HOST_DMA = 0, CL_HOST_ZEROCOPY = 1, CL_HOST_PIPELINED = 2, CL_HOST_STREAMED = 3 };
int cl_host_set_mode(cl_ctx* ctx, int mode, int slices);
/* streamed steps that were called off and redone as zero-copy steps because the CPU could not stage while
 * the kernel ran (synchronous launches: profilers, CUDA_LAUNCH_BLOCKING); after the first one the context
 * stays in zero-copy mode */
int64_t cl_host_streamed_fallbacks(const cl_ctx* ctx);
int cl_step_host_async(cl_ctx* ctx, void* stream, const cl_buffers* buf, const float* action_host);
int cl_step_host_wait(cl_ctx* ctx, void* stream, float* obs_host, float* reward_host,
                      uint8_t* done_host, float* term_obs_host, double* last_ep_ret_host,
                      int32_t* last_ep_len_host, int64_t* n_done);
int cl_step_host_wait_view(cl_ctx* ctx, void* stream, cl_host_view* view);
int cl_reset_host(cl_ctx* ctx, void* stream, const cl_buffers* buf, float* obs_host);
int64_t cl_host_h2d_bytes(const cl_ctx* ctx); /* bytes copied H2D per cl_step_host */
int64_t cl_host_d2h_bytes(const cl_ctx* ctx); /* bytes copied D2H per cl_step_host */

/* -- measurement utilities (used by bench.py for the roofline denominators that
 *    MEASURED_PEAKS.json does not carry).  dtype_bytes = 8 -> DFMA, 4 -> FFMA.
 *    Runs a register-resident FMA-chain kernel on `stream`, times it with CUDA events
 *    and returns TFLOP/s (2 flop per FMA). */
int cl_measure_fma_peak(int32_t device, int32_t dtype_bytes, double seconds, double* tflops);
/* launches issued by this context so far (bench.py's gpu_launches) */
int64_t cl_launch_count(const cl_ctx* ctx);
/* threads per block the context chose for its env kernels (wave-quantisation aware) */
int cl_block_size(const cl_ctx* ctx);
/* cl_rollout calls served by a dynamically scheduled kernel (k_rollout_sm or k_rollout_dyn: env-warp x
 * interval-chunk tasks) instead of the static one-thread-per-env mapping */
int64_t cl_dyn_launch_count(const cl_ctx* ctx);
/* rollouts that ran on the plain-I/O instantiation of the rollout kernels (FP64-bound kinds:
 * float32 SoA observation planes, real-typed reward, done flags, auto-reset, no term_obs) */
int64_t cl_plain_launch_count(const cl_ctx* ctx);
/* rollouts that ran on the SM-local kernel (k_rollout_sm: per-SM task queue, env state in shared
 * memory across the launch) -- the instantiation the bench workload selects at 65,536 envs */
int64_t cl_sm_launch_count(const cl_ctx* ctx);

/* -- device-side SB3 plumbing that directly follows the env step (SURVEY 8f ranks 1-3); all
 *    pointers are DEVICE pointers, calls only enqueue on `stream` of the current device. */

/* GAE(lambda): stable_baselines3 2.7.1 RolloutBuffer.compute_returns_and_advantage (un-vendored;
 * driven by code/train.py:112-120).  Time-major float32 planes [T][stride], n <= stride envs;
 * episode_starts[t] = 1 where env i started a new episode at step t; last_dones f32 [n]. */
int cl_gae(void* stream, const float* rewards, const float* values, const float* episode_starts,
           const float* last_values, const float* last_dones, double gamma, double gae_lambda,
           int32_t T, int64_t n, int64_t stride, float* advantages, float* returns);

/* VecNormalize (code/lorenz_pmsm/train.py:118,170; SB3 RunningMeanStd + normalize_obs):
 * cl_obs_moments: out2d[0..dim) = sum_i (x_ic - shift_c), out2d[dim..2dim) = sum_i (x_ic - shift_c)^2
 * over the n envs (f64); cl_obs_normalize: out = clip((x - mean)/sqrt(var + eps), +-clip) as f32.
 * obs addressed obs[i*es + c*cs] like cl_io. */
int cl_obs_moments(void* stream, const float* obs, int64_t es, int64_t cs, int64_t n, int32_t dim,
                   const double* shift, double* out2d);
/* RunningMeanStd.update_from_moments on the device (SB3 2.7.1 common/running_mean_std.py; used by
 * VecNormalize, code/lorenz_pmsm/train.py:118): merges the shifted sums cl_obs_moments wrote into
 * acc2d[2][dim] for a batch of n rows into mean[dim], var[dim] and the device scalar *count. */
int cl_rms_update(void* stream, const double* acc2d, int64_t n, int32_t dim, double* mean, double* var,
                  double* count);
/* cl_obs_moments for float64 input: VecNormalize feeds its float64 discounted returns to
 * ret_rms.update (SB3 2.7.1 common/vec_env/vec_normalize.py::VecNormalize._update_reward). */
int cl_moments_f64(void* stream, const double* x, int64_t es, int64_t cs, int64_t n, int32_t dim,
                   const double* shift, double* out2d);
int cl_obs_normalize(void* stream, const float* in, int64_t ies, int64_t ics, float* out, int64_t oes,
                     int64_t ocs, int64_t n, int32_t dim, const double* mean, const double* var,
                     double epsilon, double clip);

/* VecFrameStack (code/lorenz_filter/train.py:115; SB3 StackedObservations for 1-D observations):
 * stacked f32 [n][dim*n_stack] row-major is rolled by one frame, zeroed where done, then the new
 * observation is written into the last frame. */
int cl_frame_stack(void* stream, float* stacked, const float* obs, int64_t es, int64_t cs,
                   const uint8_t* done, int64_t n, int32_t dim, int32_t n_stack);
/* The same update that also produces, for envs with done[i] != 0, the stacked terminal observation
 * SB3 puts into infos[i]["terminal_observation"] (StackedObservations.update: the previous stack
 * rolled by one frame with the env's terminal observation as its last frame): term_obs f32 addressed
 * t[i*tes + c*tcs], term_stacked f32 [n][dim*n_stack] row-major (rows of unfinished envs: undefined). */
int cl_frame_stack_term(void* stream, float* stacked, const float* obs, int64_t es, int64_t cs,
                        const uint8_t* done, const float* term_obs, int64_t tes, int64_t tcs,
                        float* term_stacked, int64_t n, int32_t dim, int32_t n_stack);

/* Evaluation metrics of code/lorenz_pmsm/test_evaluate.py:25-59,239-250 for n trajectories at once:
 * err f64 [T][n_err][stride], ctrl f64 [T][n_ctrl][stride] -> out4 f64 [n][4] =
 * (MAE, RMSE over steps >= steady_start averaged over components; settling time = the largest
 * per-component settling time, np.nanmax as in the reference: a component's is (last step with
 * |e_c| > error_band) + 1) * dt, 0 if it never leaves the band and NaN if it is outside the band at
 * the last step; the result is NaN only when every component is; see calculate_advanced_metrics;
 * control energy sum(u^2) * dt). */
int cl_eval_metrics(void* stream, const double* err, const double* ctrl, int32_t T, int32_t n_err,
                    int32_t n_ctrl, int64_t n, int64_t stride, int32_t steady_start, double dt,
                    double error_band, double* out4);

/* -- host-side test hooks (no GPU needed): the exact Philox block and uniform mapping
 *    the kernels use, compiled from the same source. */
void cl_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
double cl_uniform53(uint32_t a, uint32_t b, double lo, double hi);

#ifdef __cplusplus
}
#endif
#endif /* CHAOS_B200_H */
