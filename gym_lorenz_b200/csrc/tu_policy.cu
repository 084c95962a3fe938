// Translation unit of cl_policy_rollout, cl_policy_collect and cl_policy_collect_norm: a trained SB3
// MlpPolicy (deterministic actions) fused into the hr_sync / pmsm_sync rollout, with the evaluation metrics
// of cl_eval_metrics accumulated on the fly; SB3's collect_rollouts (actor-critic, sampled actions, buffer
// rows) fused into the same rollout; and the latter behind a VecNormalize in training mode.
// Built with -fmad=false (see build.py), like tu_parity.cu, so the env arithmetic is bit-identical to
// cl_rollout's; every fused operation of the policy is an explicit fmaf.
#include <cooperative_groups.h>

#include "envs_parity.cuh"
#include "rms_merge.cuh"

using namespace cl;

namespace {

constexpr int H = CL_POLICY_HIDDEN;

// cl_policy.params, torch Linear layout: W1[H][OBS] b1[H] W2[H][H] b2[H] W3[ACT][H] b3[ACT]
template <int OBS, int ACT>
struct PolicyLayout {
  enum {
    W1 = 0, B1 = W1 + H * OBS, W2 = B1 + H, B2 = W2 + H * H, W3 = B2 + H, B3 = W3 + ACT * H,
    TOTAL = B3 + ACT, PADDED = (TOTAL + 3) & ~3
  };
  static_assert(W2 % 4 == 0, "W2 rows are read as float4");
};

// One thread per env for the whole launch (the MLP costs the same for every env: no task queue).
// Per control interval: frozen VecNormalize -> MLP (float32, fixed fmaf order) -> clip to the action box
// -> the same env_interval<E, ROLL> cl_rollout runs, with the same Philox step index -> metrics in f64.
// z = the observation, or with a frozen normaliser k_normalize's expression: the division stays a division
// by sqrt(var + eps) (s_sd), computed in f64 and rounded to f32 once
template <int OBS>
__device__ __forceinline__ void normalize_obs(const float* ob, float* z, const bool norm, const double* s_mean,
                                              const double* s_sd, const double clip) {
#pragma unroll
  for (int c = 0; c < OBS; ++c) {
    if (norm) {
      double v = ((double)ob[c] - s_mean[c]) / s_sd[c];
      v = v < -clip ? -clip : (v > clip ? clip : v);
      z[c] = (float)v;
    } else {
      z[c] = ob[c];
    }
  }
}

// out = W3 tanh(W2 tanh(W1 z + b1) + b2) + b3 with W in PolicyLayout<OBS, NOUT>: the actor (NOUT = ACT) and
// the critic (NOUT = 1) of SB3's ActorCriticPolicy.  float32, explicit fmaf in a fixed order.  h1 stays in
// registers; h2 is produced four units at a time (four independent FMA chains) and folded straight into the
// output accumulators, so it is never stored.
template <int OBS, int NOUT>
__device__ __forceinline__ void mlp_forward(const float* W, const float* z, float* out) {
  typedef PolicyLayout<OBS, NOUT> LW;
  const float4* W2v = reinterpret_cast<const float4*>(W + LW::W2);
  float h1[H];
#pragma unroll
  for (int j = 0; j < H; ++j) {
    float acc = W[LW::B1 + j];
#pragma unroll
    for (int c = 0; c < OBS; ++c) acc = fmaf(W[LW::W1 + j * OBS + c], z[c], acc);
    h1[j] = tanhf(acc);
  }
#pragma unroll
  for (int c = 0; c < NOUT; ++c) out[c] = W[LW::B3 + c];
#pragma unroll 1
  for (int j = 0; j < H; j += 4) {
    float acc[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = W[LW::B2 + j + u];
#pragma unroll
    for (int k4 = 0; k4 < H / 4; ++k4) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float4 w = W2v[(j + u) * (H / 4) + k4];
        acc[u] = fmaf(w.x, h1[4 * k4 + 0], acc[u]);
        acc[u] = fmaf(w.y, h1[4 * k4 + 1], acc[u]);
        acc[u] = fmaf(w.z, h1[4 * k4 + 2], acc[u]);
        acc[u] = fmaf(w.w, h1[4 * k4 + 3], acc[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float h2 = tanhf(acc[u]);
#pragma unroll
      for (int c = 0; c < NOUT; ++c) out[c] = fmaf(W[LW::W3 + c * H + j + u], h2, out[c]);
    }
  }
}

// The frozen normaliser of normalize_obs, set up by threads 0 .. OBS - 1 (k_normalize's expression: the
// division stays a division by sqrt(var + eps)); s_var, if given, receives var as it is.
template <int OBS>
__device__ __forceinline__ void stage_norm(const double* mean, const double* var, const double eps, double* s_mean,
                                           double* s_sd, double* s_var = nullptr) {
  if (threadIdx.x < OBS) {
    s_mean[threadIdx.x] = mean[threadIdx.x];
    const double v = var[threadIdx.x];
    if (s_var != nullptr) s_var[threadIdx.x] = v;
    s_sd[threadIdx.x] = sqrt(v + eps);
  }
}

// An actor-critic block (pack_actor_critic) in shared memory: the actor at 0, the critic at LA::PADDED (a
// 16-byte boundary: its V2 rows are read as float4), log_std after the critic at LA::PADDED + LC::PADDED.
template <int OBS, int ACT>
__device__ __forceinline__ void stage_actor_critic(const float* params, float* s_w) {
  typedef PolicyLayout<OBS, ACT> LA;
  typedef PolicyLayout<OBS, 1> LC;
  for (int k = threadIdx.x; k < LA::TOTAL; k += blockDim.x) s_w[k] = params[k];
  for (int k = threadIdx.x; k < LC::TOTAL; k += blockDim.x) s_w[LA::PADDED + k] = params[LA::TOTAL + k];
  if (threadIdx.x < ACT) s_w[LA::PADDED + LC::PADDED + threadIdx.x] = params[LA::TOTAL + LC::TOTAL + threadIdx.x];
}

// SB3's Gaussian action head, torch Normal(mu, std).log_prob with std = exp(log_std), log_scale = log(std),
// var = std^2.  sample(): a = mu + std * eps (one fmaf), lp = its log-prob summed over the components, ac =
// a clipped to the action box (the env sees ac, the buffer keeps a).
template <int ACT>
struct GaussianHead {
  float sd[ACT], lsd[ACT], var2[ACT];

  __device__ __forceinline__ explicit GaussianHead(const float* log_std) {
#pragma unroll
    for (int c = 0; c < ACT; ++c) {
      sd[c] = expf(log_std[c]);
      lsd[c] = logf(sd[c]);
      var2[c] = 2.0f * (sd[c] * sd[c]);
    }
  }

  __device__ __forceinline__ float sample(const float* mu, const double* eps, const float lo, const float hi,
                                          float* a, float* ac) const {
    const float kLogSqrt2Pi = 0.91893853320467274178f;   // (float)log(sqrt(2 pi))
    float lp = 0.0f;
#pragma unroll
    for (int c = 0; c < ACT; ++c) {
      a[c] = fmaf(sd[c], (float)eps[c], mu[c]);
      const float d = a[c] - mu[c];
      lp += -(d * d) / var2[c] - lsd[c] - kLogSqrt2Pi;
      ac[c] = clipf(a[c], lo, hi);
    }
    return lp;
  }
};

// An env's carried state -- env state, Monitor counters and, if ob is given, the observation it acts on next
// (cl_policy's obs0 layout) -- loaded from the planes and stored back; store_obs says whether q.obs_last is set.
template <class E>
__device__ __forceinline__ void load_env(typename E::S& s, int32_t& ep_len, double& ep_ret, float* ob,
                                         const KParams& p, const cl_policy& q, const int64_t i) {
  E::load(s, p, i);
  ep_len = p.ep_len[i];
  ep_ret = p.ep_return[i];
  if (ob != nullptr) {
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) ob[c] = q.obs0[i * q.obs0_es + c * q.obs0_cs];
  }
}

template <class E>
__device__ __forceinline__ void store_env(const typename E::S& s, const int32_t ep_len, const double ep_ret,
                                          const float* ob, const bool store_obs, const KParams& p,
                                          const cl_policy& q, const int64_t i) {
  E::store(s, p, i);
  p.ep_len[i] = ep_len;
  p.ep_return[i] = ep_ret;
  if (store_obs) {
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) q.obs_last[i * q.obs0_es + c * q.obs0_cs] = ob[c];
  }
}

// One row of SB3's RolloutBuffer; the reward r only with_reward (k_policy_collect_norm writes it a pass later).
template <int OBS, int ACT>
__device__ __forceinline__ void write_row(const cl_collect& col, const int64_t row, const float* z, const float* a,
                                          const bool with_reward, const float r, const float v, const float lp,
                                          const float start) {
#pragma unroll
  for (int c = 0; c < OBS; ++c) col.obs[row * OBS + c] = z[c];
#pragma unroll
  for (int c = 0; c < ACT; ++c) col.actions[row * ACT + c] = a[c];
  if (with_reward) col.rewards[row] = r;
  col.values[row] = v;
  col.log_probs[row] = lp;
  col.episode_starts[row] = start;
}

template <class E>
__global__ void __launch_bounds__(128, 4) k_policy_rollout(const KParams p, const cl_policy q, const float lo,
                                                           const float hi) {
  typedef typename E::real real;
  constexpr int OBS = E::OBS, ACT = E::ACT, NERR = 3;
  typedef PolicyLayout<OBS, ACT> LW;
  __shared__ __align__(16) float s_w[LW::PADDED];
  __shared__ double s_mean[OBS], s_sd[OBS];
  for (int k = threadIdx.x; k < LW::TOTAL; k += blockDim.x) s_w[k] = q.params[k];
  const float* W = s_w;
  const bool norm = q.obs_mean != nullptr;
  if (norm) stage_norm<OBS>(q.obs_mean, q.obs_var, q.epsilon, s_mean, s_sd);
  __syncthreads();

  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < p.n;
  const unsigned lane = threadIdx.x & 31u;
  typename E::S s = {};
  int32_t ep_len = 0;
  double ep_ret = 0.0;
  float ob[OBS];
#pragma unroll
  for (int c = 0; c < OBS; ++c) ob[c] = 0.0f;
  if (live) load_env<E>(s, ep_len, ep_ret, ob, p, q, i);
  E::prepare(s, p, live);
  const bool autoreset = (p.flags & CL_F_AUTORESET) != 0;
  const bool want_noise = E::NOISE > 0 && E::uses_noise(p);

  // metrics (cl_eval_metrics): sum |e_c| and e_c^2 over t >= steady_start, last t with |e_c| > band, sum |u|^2
  double sa[NERR], sq[NERR], en = 0.0;
  int last_ex[NERR];
#pragma unroll
  for (int c = 0; c < NERR; ++c) { sa[c] = 0.0; sq[c] = 0.0; last_ex[c] = -1; }

  unsigned bad_acc = 0u;
  bool fin = E::finite(s);
  const uint64_t step0 = step_base(p);
  for (int t = 0; t < p.T; ++t) {
    float z[OBS];
    normalize_obs<OBS>(ob, z, norm, s_mean, s_sd, q.clip_obs);
    float a[ACT];
    mlp_forward<OBS, ACT>(W, z, a);
#pragma unroll
    for (int c = 0; c < ACT; ++c) a[c] = clipf(a[c], lo, hi);   // SB3 predict: np.clip to the Box
    if (q.act_out != nullptr && live) {
#pragma unroll
      for (int c = 0; c < ACT; ++c) q.act_out[((int64_t)t * p.n + i) * ACT + c] = a[c];
    }
    real nob[OBS];
    env_interval<E, true>(s, ep_len, ep_ret, p, i, live, lane, t, step0 + (uint64_t)t, a, want_noise, false,
                          autoreset, bad_acc, nullptr, fin, nullptr, nullptr, nob);
#pragma unroll
    for (int c = 0; c < OBS; ++c) ob[c] = (float)nob[c];
#pragma unroll
    for (int c = 0; c < NERR; ++c) {
      const double e = (double)ob[c];
      if (fabs(e) > q.error_band) last_ex[c] = t;
      if (t >= q.steady_start) { sa[c] += fabs(e); sq[c] += e * e; }
    }
    double u2 = 0.0;
#pragma unroll
    for (int c = 0; c < ACT; ++c) u2 += (double)a[c] * (double)a[c];
    en += u2;
  }
  if (bad_acc && lane == 0) atomicAdd(&p.stats[CL_STAT_NONFINITE], (double)bad_acc);
  if (!live) return;
  store_env<E>(s, ep_len, ep_ret, ob, q.obs_last != nullptr, p, q, i);
  if (q.metrics != nullptr) {
    // k_eval_final's combination: averages over components, settling time as np.nanmax over components
    const double m = (double)(p.T - q.steady_start);
    double mae = 0.0, rmse = 0.0, ts = -1.0;
    bool never = false;
#pragma unroll
    for (int c = 0; c < NERR; ++c) {
      mae += sa[c] / m;
      rmse += sqrt(sq[c] / m);
      if (last_ex[c] + 1 >= p.T) never = true;
      const double tc = (last_ex[c] < 0) ? 0.0 : (double)(last_ex[c] + 1) * q.dt;
      if (last_ex[c] + 1 < p.T && tc > ts) ts = tc;
    }
    double* o = q.metrics + i * 4;
    o[0] = mae / NERR;
    o[1] = rmse / NERR;
    o[2] = (ts < 0.0 && never) ? nan("") : (ts < 0.0 ? 0.0 : ts);
    o[3] = en * q.dt;
  }
}

// SB3 OnPolicyAlgorithm.collect_rollouts for an ActorCriticPolicy, one thread per env for the whole launch
// (arithmetic: include/chaos_b200.h, cl_policy_collect).  Per control interval: frozen VecNormalize ->
// actor and critic -> Gaussian sample from the TAG_POLICY Philox block of (env, step index) -> log-prob
// -> the env step of k_policy_rollout -> TimeLimit bootstrap with the critic on the pre-reset
// observation -> one buffer row.  Shared memory holds the actor block, the critic block (moved to a
// 16-byte boundary: its V2 rows are read as float4) and log_std.
template <class E>
__global__ void __launch_bounds__(128, 4) k_policy_collect(const KParams p, const cl_policy q, const cl_collect col,
                                                           const float lo, const float hi) {
  typedef typename E::real real;
  constexpr int OBS = E::OBS, ACT = E::ACT;
  typedef PolicyLayout<OBS, ACT> LA;
  typedef PolicyLayout<OBS, 1> LC;
  __shared__ __align__(16) float s_w[LA::PADDED + LC::PADDED + ACT];
  __shared__ double s_mean[OBS], s_sd[OBS];
  stage_actor_critic<OBS, ACT>(q.params, s_w);
  const float* WA = s_w;
  const float* WC = s_w + LA::PADDED;
  const bool norm = q.obs_mean != nullptr;
  if (norm) stage_norm<OBS>(q.obs_mean, q.obs_var, q.epsilon, s_mean, s_sd);
  __syncthreads();

  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = i < p.n;
  const unsigned lane = threadIdx.x & 31u;
  typename E::S s = {};
  int32_t ep_len = 0;
  double ep_ret = 0.0;
  float ob[OBS];
#pragma unroll
  for (int c = 0; c < OBS; ++c) ob[c] = 0.0f;
  float start = 0.0f;
  if (live) {
    load_env<E>(s, ep_len, ep_ret, ob, p, q, i);
    start = col.starts[i];
  }
  E::prepare(s, p, live);
  const bool autoreset = (p.flags & CL_F_AUTORESET) != 0;
  const bool want_noise = E::NOISE > 0 && E::uses_noise(p);
  const GaussianHead<ACT> head(s_w + LA::PADDED + LC::PADDED);
  const float gamma = (float)col.gamma;

  unsigned bad_acc = 0u;
  bool fin = E::finite(s);
  const uint64_t step0 = step_base(p);
  const int64_t n = p.n;
  for (int t = 0; t < p.T; ++t) {
    const uint64_t step = step0 + (uint64_t)t;
    float z[OBS];
    normalize_obs<OBS>(ob, z, norm, s_mean, s_sd, q.clip_obs);
    float mu[ACT], v;
    mlp_forward<OBS, ACT>(WA, z, mu);
    mlp_forward<OBS, 1>(WC, z, &v);
    double eps[ACT];
    draw_normal<ACT>(make_stream(p, i, step), TAG_POLICY, eps);
    float a[ACT], ac[ACT];
    const float lp = head.sample(mu, eps, lo, hi, a, ac);
    real nob[OBS];
    TermOut<E> tr;
    env_interval<E, true>(s, ep_len, ep_ret, p, i, live, lane, t, step, ac, want_noise, false, autoreset, bad_acc,
                          nullptr, fin, nullptr, nullptr, nob, &tr);
    float r = (float)tr.rew;
    const bool boot = live && (tr.dflags & CL_DONE_TRUNCATED) && !(tr.dflags & CL_DONE_TERMINATED);
    if (__any_sync(0xffffffffu, boot)) {   // a TimeLimit truncates whole warps together
      float ot[OBS], zt[OBS], vt;
#pragma unroll
      for (int c = 0; c < OBS; ++c) ot[c] = (float)tr.obs[c];
      normalize_obs<OBS>(ot, zt, norm, s_mean, s_sd, q.clip_obs);
      mlp_forward<OBS, 1>(WC, zt, &vt);
      if (boot) r = r + gamma * vt;
    }
    if (live) write_row<OBS, ACT>(col, (int64_t)t * n + i, z, a, true, r, v, lp, start);
    start = tr.dflags != 0u ? 1.0f : 0.0f;
#pragma unroll
    for (int c = 0; c < OBS; ++c) ob[c] = (float)nob[c];
  }
  float z[OBS], v;
  normalize_obs<OBS>(ob, z, norm, s_mean, s_sd, q.clip_obs);
  mlp_forward<OBS, 1>(WC, z, &v);
  if (bad_acc && lane == 0) atomicAdd(&p.stats[CL_STAT_NONFINITE], (double)bad_acc);
  if (!live) return;
  col.last_values[i] = v;
  col.starts[i] = start;
  store_env<E>(s, ep_len, ep_ret, ob, q.obs_last != nullptr, p, q, i);
}

// Caller-owned scratch of k_policy_collect_norm, each part on a 256-byte boundary:
//   slots  f64 [2][2 OBS + 2][blocks]: per-block partial sums, double-buffered by interval parity
//   rew    f64 [n], flags u32 [n], term f32 [OBS][n]: the raw reward, done flags and pre-reset
//          observation an interval hands across the barrier to the next pass, which finishes its reward
struct NormScratch {
  double* slots;
  double* rew;
  uint32_t* flags;
  float* term;
};

int64_t norm_scratch(int obs_dim, int64_t n, char* base, NormScratch* sc) {
  const auto up = [](int64_t b) { return (b + 255) & ~(int64_t)255; };
  const int64_t max_blocks = (n + 31) / 32;   // policy_block never picks fewer than 32 threads
  const int64_t o_rew = up(2 * max_blocks * (2 * obs_dim + 2) * (int64_t)sizeof(double));
  const int64_t o_flags = o_rew + up(n * (int64_t)sizeof(double));
  const int64_t o_term = o_flags + up(n * (int64_t)sizeof(uint32_t));
  if (sc != nullptr) {
    sc->slots = (double*)base;
    sc->rew = (double*)(base + o_rew);
    sc->flags = (uint32_t*)(base + o_flags);
    sc->term = (float*)(base + o_term);
  }
  return o_term + up(obs_dim * n * (int64_t)sizeof(float));
}

// k_policy_collect with SB3's VecNormalize in training mode (arithmetic: include/chaos_b200.h,
// cl_policy_collect_norm).  One cooperative launch: thread g owns envs g, g + G, g + 2G, ... (G grid threads)
// and loads / stores their state, counters, raw observation, start and return through the planes every
// interval, so any n runs on a co-resident grid.  Pass t (0 <= t <= T) of every env first finishes interval
// t - 1 -- its reward needs the ret_rms that interval updated, its bootstrap the updated obs_rms -- and then
// runs interval t on z_t, adding the env's centred moments to its warp's row of s_acc.  After the pass each
// block writes its sums to its slot of interval parity t & 1, one grid.sync() follows, and EVERY block sums
// all slots in block order and applies cl_rms_update's merge itself: all blocks hold bit-identical statistics
// without a second barrier.  Two parities make one barrier per interval enough: a block writes the slots of
// interval t + 2 only after barrier t + 1, which no block passes before it has read the slots of t.
template <class E>
__global__ void __launch_bounds__(128, 4) k_policy_collect_norm(const KParams p, const cl_policy q,
                                                                const cl_collect col, const cl_vecnorm_update u,
                                                                const NormScratch sc, const float lo, const float hi) {
  typedef typename E::real real;
  constexpr int OBS = E::OBS, ACT = E::ACT, NS = 2 * OBS + 2;   // sums: obs (x - m), obs (x - m)^2, ret, ret^2
  typedef PolicyLayout<OBS, ACT> LA;
  typedef PolicyLayout<OBS, 1> LC;
  __shared__ __align__(16) float s_w[LA::PADDED + LC::PADDED + ACT];
  __shared__ double s_mean[OBS], s_var[OBS], s_sd[OBS];
  __shared__ double s_ret[3], s_cnt[2];   // ret mean, var, sqrt(var + eps); obs count, ret count
  __shared__ double s_acc[4][NS];         // per-warp sums of the current interval (blockDim <= 128)
  __shared__ double s_part[4][NS];        // per-warp partial sums of all blocks' slots
  __shared__ double s_tot[NS];
  stage_actor_critic<OBS, ACT>(q.params, s_w);
  const float* WA = s_w;
  const float* WC = s_w + LA::PADDED;
  const bool norm = u.norm_obs != 0, nrew = u.norm_reward != 0;
  if (norm) stage_norm<OBS>(u.obs_mean, u.obs_var, u.epsilon, s_mean, s_sd, s_var);
  if (threadIdx.x == 0) {
    s_ret[0] = *u.ret_mean;
    s_ret[1] = *u.ret_var;
    s_ret[2] = sqrt(s_ret[1] + u.epsilon);
    s_cnt[0] = norm ? *u.obs_count : 0.0;
    s_cnt[1] = *u.ret_count;
  }
  for (int k = threadIdx.x; k < 4 * NS; k += blockDim.x) (&s_acc[0][0])[k] = 0.0;
  __syncthreads();

  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  const int64_t n = p.n;
  const int64_t G = (int64_t)gridDim.x * blockDim.x;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int K = (int)((n + G - 1) / G);   // envs per thread (the last ones of some threads are past n)
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const bool autoreset = (p.flags & CL_F_AUTORESET) != 0;
  const bool want_noise = E::NOISE > 0 && E::uses_noise(p);
  const GaussianHead<ACT> head(s_w + LA::PADDED + LC::PADDED);
  const float gamma = (float)col.gamma;
  const double bn = (double)n;   // batch count of every update: live envs only

  unsigned bad_acc = 0u;
  const uint64_t step0 = step_base(p);
  for (int t = 0; t <= p.T; ++t) {
    const float* obs_in = t == 0 ? q.obs0 : q.obs_last;
    for (int k = 0; k < K; ++k) {
      const int64_t i = g + (int64_t)k * G;
      if (i - (int64_t)lane >= n) break;   // warp-uniform: the whole warp is past the batch, and stays so
      const bool live = i < n;
      float ob[OBS];
#pragma unroll
      for (int c = 0; c < OBS; ++c) ob[c] = live ? obs_in[i * q.obs0_es + c * q.obs0_cs] : 0.0f;

      if (t > 0) {   // finish interval t - 1 with the statistics it updated
        const double r0 = live ? sc.rew[i] : 0.0;
        const uint32_t f0 = live ? sc.flags[i] : 0u;
        float r;
        if (nrew) {
          double v = r0 / s_ret[2];
          v = v < -u.clip_reward ? -u.clip_reward : (v > u.clip_reward ? u.clip_reward : v);
          r = (float)v;
        } else {
          r = (float)r0;
        }
        // k_policy_collect's TimeLimit bootstrap.  It stays written out in both kernels: as a shared inline
        // function it changed the instruction schedule of both.
        const bool boot = live && (f0 & CL_DONE_TRUNCATED) && !(f0 & CL_DONE_TERMINATED);
        if (__any_sync(0xffffffffu, boot)) {
          float ot[OBS], zt[OBS], vt;
#pragma unroll
          for (int c = 0; c < OBS; ++c) ot[c] = boot ? sc.term[c * n + i] : 0.0f;
          normalize_obs<OBS>(ot, zt, norm, s_mean, s_sd, u.clip_obs);
          mlp_forward<OBS, 1>(WC, zt, &vt);
          if (boot) r = r + gamma * vt;
        }
        if (live) col.rewards[(int64_t)(t - 1) * n + i] = r;
      }
      float z[OBS];
      normalize_obs<OBS>(ob, z, norm, s_mean, s_sd, u.clip_obs);
      if (t == p.T) {
        float v;
        mlp_forward<OBS, 1>(WC, z, &v);
        if (live) col.last_values[i] = v;
        continue;
      }

      const uint64_t step = step0 + (uint64_t)t;
      typename E::S s = {};
      int32_t ep_len = 0;
      double ep_ret = 0.0, ret = 0.0;
      float start = 0.0f;
      if (live) {
        load_env<E>(s, ep_len, ep_ret, nullptr, p, q, i);
        start = col.starts[i];
        ret = u.returns[i];
      }
      bool fin = E::finite(s);   // what k_policy_collect carries in a register: finite after every reset
      float mu[ACT], v;
      mlp_forward<OBS, ACT>(WA, z, mu);
      mlp_forward<OBS, 1>(WC, z, &v);
      double eps[ACT];
      draw_normal<ACT>(make_stream(p, i, step), TAG_POLICY, eps);
      float a[ACT], ac[ACT];
      const float lp = head.sample(mu, eps, lo, hi, a, ac);
      real nob[OBS];
      TermOut<E> tr;
      env_interval<E, true>(s, ep_len, ep_ret, p, i, live, lane, t, step, ac, want_noise, false, autoreset, bad_acc,
                            nullptr, fin, nullptr, nullptr, nob, &tr);
      // VecNormalize: obs_rms.update(o) around mean_old, returns = returns * gamma + r, ret_rms.update(returns)
      double m[NS];
      ret = ret * u.gamma + (double)tr.rew;
#pragma unroll
      for (int c = 0; c < OBS; ++c) {
        ob[c] = (float)nob[c];
        const double d = live && norm ? (double)ob[c] - s_mean[c] : 0.0;
        m[c] = d;
        m[OBS + c] = d * d;
      }
      {
        const double d = live ? ret - s_ret[0] : 0.0;
        m[2 * OBS] = d;
        m[2 * OBS + 1] = d * d;
      }
#pragma unroll
      for (int c = 0; c < NS; ++c) {
        if (c < 2 * OBS && !norm) continue;
        const double w = warp_sum(m[c]);
        if (lane == 0) s_acc[warp][c] += w;
      }
      if (live) {
        write_row<OBS, ACT>(col, (int64_t)t * n + i, z, a, false, 0.0f, v, lp, start);
        sc.rew[i] = (double)tr.rew;
        sc.flags[i] = tr.dflags;
        if ((tr.dflags & CL_DONE_TRUNCATED) && !(tr.dflags & CL_DONE_TERMINATED)) {
#pragma unroll
          for (int c = 0; c < OBS; ++c) sc.term[c * n + i] = (float)tr.obs[c];
        }
        store_env<E>(s, ep_len, ep_ret, ob, true, p, q, i);   // obs_last is required here
        col.starts[i] = tr.dflags != 0u ? 1.0f : 0.0f;
        u.returns[i] = tr.dflags != 0u ? 0.0 : ret;
      }
    }
    if (t == p.T) break;

    // interval t's batch statistics: block sums -> slot, barrier, every block sums all slots in one fixed order
    __syncthreads();
    const unsigned nb = gridDim.x;
    double* slot = sc.slots + (size_t)(t & 1) * NS * nb;   // [NS][blocks]: component-major
    const int nwarp = blockDim.x >> 5;
    if (threadIdx.x < NS) {
      double a = 0.0;
      for (int w = 0; w < nwarp; ++w) { a += s_acc[w][threadIdx.x]; s_acc[w][threadIdx.x] = 0.0; }
      slot[(size_t)threadIdx.x * nb + blockIdx.x] = a;
    }
    grid.sync();
    {
      // thread j sums blocks j, j + blockDim, ... (NS independent loads in flight), then warp shuffles and the
      // warps in order: the same tree in every block, so every block gets the same bits
      double a[NS];
#pragma unroll
      for (int c = 0; c < NS; ++c) a[c] = 0.0;
      for (unsigned b = threadIdx.x; b < nb; b += blockDim.x) {
#pragma unroll
        for (int c = 0; c < NS; ++c) a[c] += __ldcg(slot + (size_t)c * nb + b);
      }
#pragma unroll
      for (int c = 0; c < NS; ++c) {
        const double w = warp_sum(a[c]);
        if (lane == 0) s_part[warp][c] = w;
      }
      __syncthreads();
      if (threadIdx.x < NS) {
        double v = 0.0;
        for (int w = 0; w < nwarp; ++w) v += s_part[w][threadIdx.x];
        s_tot[threadIdx.x] = v;
      }
    }
    __syncthreads();
    // cl_rms_update's merge (rms_merge.cuh): thread c < OBS feature c, thread OBS ret
    const int c = threadIdx.x;
    const bool mo = norm && c < OBS, mr = c == OBS;
    if (mo || mr) {
      const double acc1 = mo ? s_tot[c] : s_tot[2 * OBS], acc2 = mo ? s_tot[OBS + c] : s_tot[2 * OBS + 1];
      double* mean = mo ? &s_mean[c] : &s_ret[0];
      double* var = mo ? &s_var[c] : &s_ret[1];
      rms_merge(*mean, *var, mo ? s_cnt[0] : s_cnt[1], bn, acc1, acc2);
      if (mo) s_sd[c] = sqrt(*var + u.epsilon);
      else s_ret[2] = sqrt(*var + u.epsilon);
    }
    __syncthreads();   // every merging thread has read the counts
    if (threadIdx.x == 0) { s_cnt[0] += norm ? bn : 0.0; s_cnt[1] += bn; }
    __syncthreads();
  }
  if (bad_acc && lane == 0) atomicAdd(&p.stats[CL_STAT_NONFINITE], (double)bad_acc);
  if (blockIdx.x == 0) {   // every block holds the same statistics
    if (norm && threadIdx.x < OBS) { u.obs_mean[threadIdx.x] = s_mean[threadIdx.x]; u.obs_var[threadIdx.x] = s_var[threadIdx.x]; }
    if (threadIdx.x == 0) {
      *u.ret_mean = s_ret[0];
      *u.ret_var = s_ret[1];
      *u.ret_count = s_cnt[1];
      if (norm) *u.obs_count = s_cnt[0];
    }
  }
}

// Threads of the fullest SM decide the launch: ceil(blocks / SMs) * block, ties -> the larger block (a
// smaller one stages the weights into shared memory more often: 14 blocks of 32 would not fit one SM).
int policy_block(int64_t n, int sms) {
  int best = 128;
  int64_t best_cost = -1;
  for (int b = 128; b >= 32; b /= 2) {
    const int64_t cost = (((n + b - 1) / b + sms - 1) / sms) * b;
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = b; }
  }
  return best;
}

int64_t grid_for(int64_t n, int block) { return (n + block - 1) / block; }

// f(EnvHRSync()) or f(EnvPMSMSync()) for the env kind: the policy kernels exist for these two only
template <class F>
cudaError_t with_policy_env(int kind, const F& f) {
  switch (kind) {
    case CL_ENV_HR_SYNC: return f(EnvHRSync());
    case CL_ENV_PMSM_SYNC: return f(EnvPMSMSync());
    default: return cudaErrorInvalidValue;
  }
}

// Cooperative: the grid is what the occupancy calculator says is co-resident (blocks per SM x SMs), capped at
// the blocks n needs.  The driver refuses a cooperative launch that could not be co-resident, so grid.sync()
// cannot wait on a block that never starts.
template <class E>
cudaError_t launch_policy_collect_norm(const KParams& p, const cl_policy& q, const cl_collect& col,
                                       const cl_vecnorm_update& u, float lo, float hi, cudaStream_t st, int sms) {
  int block = policy_block(p.n, sms), per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_policy_collect_norm<E>, block, 0);
  if (e == cudaSuccess && block != 128 && grid_for(p.n, block) > (int64_t)per_sm * sms) {
    // policy_block's grid is not co-resident: 128-thread blocks hold the most envs per SM (the weights in
    // shared memory, not the registers, limit the smaller ones), so the fewest threads own two envs
    block = 128;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_policy_collect_norm<E>, block, 0);
  }
  if (e != cudaSuccess) return e;
  if (per_sm < 1) return cudaErrorCooperativeLaunchTooLarge;
  const int64_t need = grid_for(p.n, block), fit = (int64_t)per_sm * sms;
  NormScratch sc;
  norm_scratch(E::OBS, p.n, (char*)u.scratch, &sc);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(need < fit ? need : fit));
  cfg.blockDim = dim3((unsigned)block);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_policy_collect_norm<E>, p, q, col, u, sc, lo, hi);
}

}  // namespace

int64_t cl_policy_collect_norm_bytes(int obs_dim, int64_t n) { return norm_scratch(obs_dim, n, nullptr, nullptr); }

cudaError_t cl_launch_policy(int kind, const KParams& p, const cl_policy& q, float lo, float hi, cudaStream_t st,
                             int sms) {
  return with_policy_env(kind, [&](auto env) {
    const int block = policy_block(p.n, sms);
    k_policy_rollout<decltype(env)><<<(unsigned)grid_for(p.n, block), block, 0, st>>>(p, q, lo, hi);
    return cudaGetLastError();
  });
}

cudaError_t cl_launch_policy_collect(int kind, const KParams& p, const cl_policy& q, const cl_collect& col, float lo,
                                     float hi, cudaStream_t st, int sms) {
  return with_policy_env(kind, [&](auto env) {
    const int block = policy_block(p.n, sms);
    k_policy_collect<decltype(env)><<<(unsigned)grid_for(p.n, block), block, 0, st>>>(p, q, col, lo, hi);
    return cudaGetLastError();
  });
}

cudaError_t cl_launch_policy_collect_norm(int kind, const KParams& p, const cl_policy& q, const cl_collect& col,
                                          const cl_vecnorm_update& u, float lo, float hi, cudaStream_t st, int sms) {
  return with_policy_env(kind, [&](auto env) {
    return launch_policy_collect_norm<decltype(env)>(p, q, col, u, lo, hi, st, sms);
  });
}
