// Generic one-thread-per-env kernels: step / fused rollout / reset / init.
//
// Every env kind is a small struct (`E`) giving the register-resident state `E::S`, its
// SoA load/store, `reset`, `step` and a few predicates; the kernels below add what is
// common to all kinds: action fetch (strided, or in-kernel Philox for synthetic
// rollouts), process-noise draws, TimeLimit, SB3-style auto-reset, Monitor-style episode
// accounting and warp-reduced statistics.  State stays in registers across all T control
// intervals (and all RK4 substeps) of a launch.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "../../include/chaos_b200.h"
#include "philox.cuh"

namespace cl {

struct KParams {
  int64_t n, n_pad, env_id_base;
  int64_t i_begin;        // first env of this launch (host path: env slices pipelined over streams)
  uint32_t k0, k1;
  uint64_t step_index;
  // graph mode: the Philox step index lives on the device so that CUDA-graph replays advance it
  uint64_t* step_ptr;     // nullptr -> use step_index
  int32_t max_steps, substeps, flags, reward_f32;
  double dt, alpha, act_limit, act_gain, param_jitter;
  // persistent buffers
  void* state;
  int32_t* aux_int;
  int32_t* ep_len;
  double* ep_return;
  double* stats;
  // io
  const float* action;
  int64_t act_es, act_cs;
  const double* noise;
  void* obs;
  int64_t obs_es, obs_cs;
  void* reward;
  uint8_t* done;
  void* term_obs;
  double* last_ep_ret;
  int32_t* last_ep_len;
  const uint8_t* mask;
  // host path (cl_step_host_async): per-env-warp "an episode ended here" flags in the pinned result
  // slot, Monitor numbers written as whole warp rows, and -- streamed mode -- the generation flags the
  // CPU publishes slice by slice while it stages the caller's action array into pinned memory
  uint8_t* warp_done;
  int32_t host_rows;
  const uint32_t* act_ready;
  uint32_t act_gen;
  int32_t act_slice_envs;
  int32_t act_lane_slices;   // slices per staging lane; lane k's progress word is act_ready[k]
  // in-kernel relay (block 0 of the step kernel mirrors the pinned progress words itself; nullptr: k_relay does, on a side stream)
  const uint32_t* act_host_words;
  int32_t act_lanes, act_nslices;
  uint32_t* host_err;
  // rollout
  int32_t T;
  int64_t act_ts, obs_ts, rew_ts, done_ts;
  float synth_amp;
  // PMSM_SYNC Adam bias-correction tables: tabK[n] = (float)(1 - betaK**n), see chaos_b200.cu
  const float* bc1;
  const float* bc2;
  int32_t bc1_n, bc2_n;
  // RK4 kinds: step sizes precomputed on the host so they are constant-bank operands of the
  // FMAs (a DFMA with three distinct REGISTER sources issues at 2/3 rate on sm_100, see
  // DESIGN.md "FP64 cost model"): h = dt/S, hh = h/2, h3 = h/3, h6 = h/6 (+ float copies),
  // and the nominal parameters for the warp-uniform fast path.
  double h, hh, h3, h6;
  float hf, hhf, h3f, h6f;
  double nom[3];
  float nomf[3];
  double nom_br;   // Lorenz: beta * rho, PMSM: unused -- the interval constant of the shifted integrator
  float nom_brf;
  float act_limit_f, act_gain_f;
  // dynamic rollout scheduling (k_rollout_dyn)
  uint32_t* dyn_counter;
  uint32_t* dyn_progress;
  int32_t dyn_chunk, dyn_nchunks, dyn_nwarps, dyn_tma, dyn_grid;
  // SM-local rollout scheduling (k_rollout_sm): grid, worker warps per block, control intervals per task
  int32_t sm_grid, sm_workers, sm_chunk, sm_gdiv;   // sm_gdiv: guest chunk = sm_chunk / sm_gdiv
  int32_t sm_tmap_ok;                  // *host_tmap describes the action tensor (x env, y channel, z interval)
  const CUtensorMap* host_tmap;        // host-side only: passed to k_rollout_sm as its own __grid_constant__ parameter
  // observations go out as contiguous, 16-byte aligned float32 rows -> warp-transposed vector stores
  int32_t rows_fast;
  int32_t no_plain;  // host-side only: keep the generic instantiation (tests, A/B runs)
  int32_t* host_plain_out;  // host-side only: launch_env reports which instantiation it launched (bit 0 plain, bit 1 k_rollout_sm)
};

enum LaunchMode { MODE_STEP = 0, MODE_ROLLOUT = 1, MODE_RESET = 2, MODE_INIT = 3, MODE_ROLLOUT_DYN = 4 };

// ---- small numeric helpers -----------------------------------------------------------

// np.clip semantics (NaN propagates: both comparisons are false).
__device__ __forceinline__ float clipf(float a, float lo, float hi) {
  return a < lo ? lo : (a > hi ? hi : a);
}
__device__ __forceinline__ double clipd(double a, double lo, double hi) {
  return a < lo ? lo : (a > hi ? hi : a);
}

// x**a for x >= 0 (reward terms): exp(a*log(x)) costs roughly half of the fully general double
// pow() and is accurate to ~1e-15 relative here (|a*log x| stays below ~10), far inside the
// tolerances of the quantities it feeds (1 ulp f32 after rounding / 1e-12 in f64).  The general
// pow() handles the exceptional exponents.
__device__ __forceinline__ double pow_pos(double x, double a) {
  // alpha = 1/2 is the envs' default exponent: a correctly rounded sqrt (~10 FP64 instructions
  // instead of ~150 for log + exp); warp-uniform test (a is a launch parameter).  x < 0 -> NaN, as pow.
  if (a == 0.5) return sqrt(x);
  // alpha = 1/3 (the memristive pair's reward, lorenz_env_transient2.py): cbrt is ~4x cheaper than
  // log + exp and within 1 ulp of pow(x, 0.3333333333333333) for every x the reward can reach
  // (the exponent's rounding error shifts the result by ln(x) * 1.9e-17 relative)
  if (a == 1.0 / 3) return cbrt(x);
  if (!(a > 0.0) || !(a < 64.0)) return pow(x, a);
  if (x == 0.0) return 0.0;
  return exp(a * log(x));   // log(inf)=inf -> inf, NaN propagates, x<0 -> NaN like pow for non-integer a
}

// products that must stay products: `u = a*g; ... u - y` would otherwise be contracted into
// fma(a, g, -y), a DFMA with three register sources (3 issue cycles instead of a 2-cycle DADD,
// DESIGN.md "FP64 cost model") in every RK4 stage
__device__ __forceinline__ double mul_keep(double a, double b) { return __dmul_rn(a, b); }
// FP32: a three-register FFMA issues at full rate, so the contraction is a free saving of one
// instruction per stage there (measured: 45.7 vs 42.3 TFLOP/s at 1 Mi envs) -- leave it to ptxas
__device__ __forceinline__ float mul_keep(float a, float b) { return a * b; }
// a product rounded exactly once, in either precision (never contracted)
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }

__device__ __forceinline__ Stream make_stream(const KParams& p, int64_t i, uint64_t step) {
  const uint64_t gid = (uint64_t)(p.env_id_base + i);
  Stream s;
  s.id_lo = (uint32_t)gid;
  s.id_hi = (uint32_t)(gid >> 32);
  s.step = (uint32_t)step;
  // the upper 24 bits of a 56-bit step counter are folded into the second key word
  s.k0 = p.k0;
  s.k1 = p.k1 ^ (uint32_t)((step >> 32) & 0x00FFFFFFu);
  return s;
}

// Step index of this launch: by value, or (graph mode) read from the device counter.
__device__ __forceinline__ uint64_t step_base(const KParams& p) {
  return p.step_ptr != nullptr ? *((volatile const uint64_t*)p.step_ptr) : p.step_index;
}
// Graph mode: a one-thread kernel enqueued right after each env kernel advances the device
// counter (a per-block completion ticket would put one same-address atomic per block on the
// critical path: +35 us at 16,384 blocks).
__global__ void k_advance_step(uint64_t* step, uint64_t count);
// Streamed host mode: mirrors the pinned "slices staged" word (gen << 8 | count) into device memory until
// all `nslices` of generation `gen` are published (bounded: ~2 s).
__global__ void k_relay(const uint32_t* host_words, uint32_t* dev_words, uint32_t gen, uint32_t lanes, uint32_t spl,
                        uint32_t nslices, uint32_t* host_err);

// n uniforms in [lo,hi) (NumPy construction), 2 per Philox block.
template <int N>
__device__ __forceinline__ void draw_uniform(const Stream& rng, uint32_t tag, double lo, double hi,
                                             double* out) {
#pragma unroll
  for (int b = 0; b < (N + 1) / 2; ++b) {
    const u32x4 r = rng.draw(tag + (uint32_t)b);
    out[2 * b] = uniform53(r.x, r.y, lo, hi);
    if (2 * b + 1 < N) out[2 * b + 1] = uniform53(r.z, r.w, lo, hi);
  }
}

// n standard normals (Box-Muller on 53-bit uniforms), 2 per Philox block.
template <int N>
__device__ __forceinline__ void draw_normal(const Stream& rng, uint32_t tag, double* out) {
#pragma unroll
  for (int b = 0; b < (N + 1) / 2; ++b) {
    const u32x4 r = rng.draw(tag + (uint32_t)b);
    const double u1 = 1.0 - u01_53(r.x, r.y);  // (0,1]
    const double u2 = u01_53(r.z, r.w);
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    out[2 * b] = rad * cs;
    if (2 * b + 1 < N) out[2 * b + 1] = rad * sn;
  }
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename real>
__device__ __forceinline__ void store_obs(void* base, int64_t off, int64_t es, int64_t cs, int64_t i,
                                          const real* obs, int n, bool f64) {
  if (f64) {
    double* o = (double*)base + off + i * es;
    for (int c = 0; c < n; ++c) o[c * cs] = (double)obs[c];
  } else {
    float* o = (float*)base + off + i * es;
    for (int c = 0; c < n; ++c) o[c * cs] = (float)obs[c];
  }
}

// Row-major [N][OBS] float32 observations (what a policy network and the SB3 host path want):
// a warp's 32 rows are one contiguous run of 32*OBS floats.  Writing them lane-by-lane would be
// OBS strided 4-byte stores per lane; instead the warp transposes through shared memory and
// writes whole 16-byte vectors, i.e. full 128-byte lines (this is what makes direct stores to
// pinned host memory over PCIe efficient in the zero-copy host path).
template <typename real, int OBS>
__device__ __forceinline__ void store_obs_rows_warp(float* __restrict__ sm, float* __restrict__ base,
                                                    const int64_t warp_env0, const int64_t n, const unsigned lane,
                                                    const real* obs) {
#pragma unroll
  for (int c = 0; c < OBS; ++c) sm[lane * OBS + c] = (float)obs[c];
  __syncwarp();
  const int64_t rows = n - warp_env0;
  const int nflt = (int)(rows >= 32 ? 32 : (rows > 0 ? rows : 0)) * OBS;
  float* dst = base + warp_env0 * OBS;
  for (int k = (int)lane * 4; k + 3 < nflt; k += 128)
    *reinterpret_cast<float4*>(dst + k) = *reinterpret_cast<const float4*>(sm + k);
  for (int k = (nflt & ~3) + (int)lane; k < nflt; k += 32) dst[k] = sm[k];
  __syncwarp();
}

// plane accessors
template <typename real>
__device__ __forceinline__ real ldp(const KParams& p, int c, int64_t i) {
  return __ldcg((const real*)p.state + (int64_t)c * p.n_pad + i);  // L1-bypassing: see k_rollout_dyn
}
template <typename real>
__device__ __forceinline__ void stp(const KParams& p, int c, int64_t i, real v) {
  ((real*)p.state)[(int64_t)c * p.n_pad + i] = v;
}

__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---- one control interval of one env (shared by the static and the dynamic kernels) ----

// The "plain rollout" I/O shape -- what a synthetic-action benchmark or a device-side collector
// uses: canonical time-major float32 observation planes [T][OBS][n_pad], reward [T][n_pad] in the
// env's real type, done flags, auto-reset on, no terminal-observation buffer, actions given (staged
// by bulk copies in the dynamic kernel).  For the kinds whose rollout is arithmetic / issue bound
// (PlainRollout<E>::value) the rollout kernels are instantiated a second time with these as
// compile-time facts: the generic interval executes ~245 non-FP64 instructions per warp (runtime
// layout / null-pointer tests, 64-bit stride arithmetic), the plain one under half of that, and
// with only ~3 warps per scheduler every epilogue instruction shows (-3 % launch time at 65,536 envs
// for FP64, -12...17 % for the issue-bound FP32 kind).
// launch_env() picks the instantiation from the launch parameters; results are identical.
template <class E> struct PlainRollout { enum { value = 0 }; };
// Kinds whose termination test bounds the state (e.g. |x|+|y|+|z| <= 1e6): a step that does not
// terminate leaves a finite state, so the plain rollout loop (auto-reset always on) evaluates
// E::finite only on the rare terminating step.
template <class E> struct FiniteUnlessTerm { enum { value = 0 }; };
template <int N> struct SpecTag { enum { value = N }; };

// ---- deferred outputs of the plain rollout loop -------------------------------------------
// The plain loop keeps the outputs of interval t in registers and emits them at the top of interval
// t+1 as branch-free predicated stores (inline PTX `@p st`): no divergent `if (live)` region with
// its reconvergence barrier, conversions and address arithmetic in the same basic block as the
// action fetch and the integrator.  ptxas still schedules them ahead of the DFMA stream rather
// than into it; measured neutral for FP64 and +5.4 % for the issue-bound FP32 kind at 65,536 envs.
// It also lets the dynamic kernel hand an env-warp over BEFORE its last outputs go out.
// Terminations and resets are still decided at the end of interval t.
#ifndef CL_PLAIN_DEFER
#define CL_PLAIN_DEFER 1
#endif
template <class E> struct PlainPending {
  typename E::real obs[E::OBS];
  typename E::real rew;
  uint32_t dflags, valid;
  int t;   // interval the record belongs to (addressing of the static kernel)
  // Dynamic kernel: running output pointers of this lane, bumped by one time step per emit --
  // recomputing t * stride + i with 64-bit arithmetic costs ~20 more integer instructions per
  // interval (+1.3 % FP64, +2.6 % FP32 at 65,536 envs).  The static kernel keeps the recomputation:
  // at 1 Mi envs it lives on occupancy and the six extra registers cost the FP32 kind 3 %.
  float* o;
  typename E::real* rp;
  uint8_t* dp;
  __device__ __forceinline__ void begin(const KParams& p, const int64_t i, const int t0) {
    const int64_t np = p.n_pad, row = (int64_t)t0 * np + i;   // i < n_pad always
    o = (float*)p.obs + (int64_t)t0 * (E::OBS * np) + i;
    rp = (typename E::real*)p.reward + row;
    dp = p.done + row;
    t = t0;
    valid = 0u; dflags = 0u; rew = 0;
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) obs[c] = 0;
  }
};
__device__ __forceinline__ void st_if(float* ptr, float v, uint32_t pr) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %0, 0;\n@p st.global.f32 [%1], %2;\n}" ::"r"(pr), "l"(ptr), "f"(v) : "memory");
}
__device__ __forceinline__ void st_if(double* ptr, double v, uint32_t pr) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %0, 0;\n@p st.global.f64 [%1], %2;\n}" ::"r"(pr), "l"(ptr), "d"(v) : "memory");
}
__device__ __forceinline__ void st_if(uint8_t* ptr, uint32_t v, uint32_t pr) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %0, 0;\n@p st.global.u8 [%1], %2;\n}" ::"r"(pr), "l"(ptr), "r"(v) : "memory");
}
template <class E, bool RUNPTR>
__device__ __forceinline__ void plain_emit(const KParams& p, const int64_t i, const bool live, PlainPending<E>& d) {
  typedef typename E::real real;
  const uint32_t pr = (live && d.valid) ? 1u : 0u;
  // canonical time-major planes obs[T][OBS][n_pad], reward[T][n_pad], done[T][n_pad]: every stride
  // derives from n_pad (uniform registers are scarce in this loop, see PlainRollout)
  const int64_t np = p.n_pad;
  if (RUNPTR) {
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) st_if(d.o + c * np, (float)d.obs[c], pr);
    st_if(d.rp, d.rew, pr);
    st_if(d.dp, d.dflags, pr);
    if (d.valid) {   // warp-uniform; the first emit of a task is the empty one and must not move
      d.o += E::OBS * np;
      d.rp += np;
      d.dp += np;
    }
  } else {
    const int64_t row = (int64_t)d.t * np + i;   // i < n_pad always
    float* o = (float*)p.obs + (int64_t)d.t * (E::OBS * np) + i;
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) st_if(o + c * np, (float)d.obs[c], pr);
    st_if((real*)p.reward + row, d.rew, pr);
    st_if(p.done + row, d.dflags, pr);
  }
}

// SPEC: warp-uniform specialisation of E::step chosen once per launch / task (0 = generic).  Kinds
// with PlainRollout<E>::value provide `static int spec(const S&, const KParams&)` (evaluated by all
// 32 lanes) and `template <int SPEC> step_spec(...)`; the plain rollout kernels then run one of two
// separately compiled interval loops, each a straight line of code (e.g. Lorenz: nominal parameters
// as constant-bank operands + 16 unrolled substeps) instead of branching per interval.
template <class E, int SPEC>
__device__ __forceinline__ void step_dispatch(typename E::S& s, const KParams& p, const float* a, const double* nz,
                                              typename E::real* obs, typename E::real& rew, bool& term) {
  if constexpr (SPEC != 0) E::template step_spec<SPEC>(s, p, a, nz, obs, rew, term);
  else E::step(s, p, a, nz, obs, rew, term);
}

// What the rollout collector (k_policy_collect) needs of an interval in registers besides the next
// observation: the reward, the done flags and the pre-reset (terminal) observation it bootstraps from.
template <class E>
struct TermOut {
  typename E::real obs[E::OBS];
  typename E::real rew;
  uint32_t dflags;
};

template <class E, bool ROLL, bool PLAIN = false, int SPEC = 0, bool RUNPTR = false, class TermPtr = decltype(nullptr)>
__device__ __forceinline__ unsigned env_interval(typename E::S& s, int32_t& ep_len, double& ep_ret,
                                             const KParams& p, const int64_t i, const bool live,
                                             const unsigned lane, const int t, const uint64_t step,
                                             const float* a, const bool want_noise, const bool obs64,
                                             const bool autoreset, unsigned& bad_acc, float* sm_rows, bool& fin,
                                             PlainPending<E>* pend = nullptr, double* blk_stats = nullptr,
                                             typename E::real* obs_out = nullptr, TermPtr term_out = nullptr) {
  typedef typename E::real real;
  if (PLAIN && CL_PLAIN_DEFER) plain_emit<E, RUNPTR>(p, i, live, *pend);   // outputs of the previous interval
  // The per-interval Philox stream (key / counter words).  Generic kernels build it up front: building
  // it inside the noise and reset branches instead measured -10 % on the HR single-step kernel at
  // 1 Mi envs (-5 % pmsm_classic).  The plain rollout kernels build it only when an episode ends:
  // their interval loop is short of uniform registers (see PlainRollout) and has no noise draw.
  Stream rng = {};
  if (!PLAIN) rng = make_stream(p, i, step);
  double nz[E::NOISE > 0 ? E::NOISE : 1];
  nz[0] = 0.0;
  if (want_noise) {
    if (p.noise != nullptr) {
#pragma unroll
      for (int c = 0; c < E::NOISE; ++c) nz[c] = live ? p.noise[c * p.n_pad + i] : 0.0;
    } else {
      draw_normal<(E::NOISE > 0 ? E::NOISE : 1)>(rng, TAG_NOISE, nz);
    }
  }

  real obs[E::OBS];
  real rew;
  bool term;
  const bool was_finite = fin;  // finiteness is carried from the previous interval, not recomputed
  step_dispatch<E, SPEC>(s, p, a, nz, obs, rew, term);
  ep_len += 1;
  ep_ret += (double)rew;
  const bool trunc = E::time_limit(p, ep_len);
  const bool done = term || trunc;
  bool bad;  // divergence EVENT (a diverged env that is never reset would otherwise cost an atomic every step)
  if constexpr (PLAIN && FiniteUnlessTerm<E>::value != 0) {
    fin = true;
    bad = false;
    if (term) { fin = E::finite(s); bad = was_finite && !fin; }
  } else {
    fin = E::finite(s);
    bad = was_finite && !fin;
  }

  // warp-aggregated statistics (one set of atomics per warp, only when something ended)
  const bool has_term = !PLAIN && p.term_obs != nullptr;
  const unsigned dall = __ballot_sync(0xffffffffu, live && done && (autoreset || has_term));
  const unsigned dm = autoreset ? dall : 0u;
  const unsigned bm = __ballot_sync(0xffffffffu, live && bad);
  if (dm) {
    const bool mine = (dm >> lane) & 1u;
    const double r1 = warp_sum(mine ? ep_ret : 0.0);
    const double r2 = warp_sum(mine ? ep_ret * ep_ret : 0.0);
    const int l1 = warp_sum(mine ? ep_len : 0);
    const unsigned tm = __ballot_sync(0xffffffffu, mine && term);
    const unsigned um = __ballot_sync(0xffffffffu, mine && trunc && !term);
    if (lane == 0) {
      // blk_stats: block-shared accumulator of k_step (flushed once per block).  With a global atomic per
      // warp, a batch in which most env-warps end an episode every step (memristive pair under full-range
      // forcing at 1 Mi envs: 32,768 warps x 6 atomics on 6 addresses) spends half its time queueing there.
      double* dst = blk_stats != nullptr ? blk_stats : p.stats;
      atomicAdd(&dst[CL_STAT_EPISODES], (double)__popc(dm));
      atomicAdd(&dst[CL_STAT_RET_SUM], r1);
      atomicAdd(&dst[CL_STAT_RET_SQ], r2);
      atomicAdd(&dst[CL_STAT_LEN_SUM], (double)l1);
      if (tm) atomicAdd(&dst[CL_STAT_TERMINATED], (double)__popc(tm));
      if (um) atomicAdd(&dst[CL_STAT_TRUNCATED], (double)__popc(um));
    }
  }
  bad_acc += __popc(bm);  // flushed once per launch / task (diverged envs would otherwise
                          // serialise every warp on one atomic each interval)

  const int64_t oo = ROLL ? t * p.obs_ts : 0;
  const bool rows_fast = !PLAIN && p.rows_fast != 0;  // warp-uniform
  if (has_term && rows_fast && dall) {
    // a warp with a finished episode writes all 32 of its rows (whole 128-byte lines; the host
    // path points term_obs at pinned host memory, where scattered 4-byte stores would each be
    // a PCIe transaction).  Rows of unfinished envs are not meaningful and never read.
    store_obs_rows_warp<real, E::OBS>(sm_rows, (float*)p.term_obs + oo, i - (int64_t)lane, p.n, lane, obs);
  }
  const bool host_rows = !PLAIN && p.host_rows != 0;   // warp-uniform
  if (host_rows && dall && live) {
    // host path: the Monitor numbers go to pinned host memory; a warp with a finished episode writes
    // all of its rows (256 + 128 contiguous bytes) instead of one scattered PCIe write per finished env.
    // Entries of unfinished envs are not meaningful and never read.
    p.last_ep_ret[i] = ep_ret;
    p.last_ep_len[i] = ep_len;
  }
  // before the auto-reset overwrites obs.  term_out is a TermOut<E>* or (every other caller) the default
  // nullptr: its type removes the copy before code generation (a run-time null test, although folded,
  // measurably changed the register allocation of k_policy_rollout)
  if constexpr (!std::is_same<TermPtr, decltype(nullptr)>::value) {
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) term_out->obs[c] = obs[c];
    term_out->rew = rew;
    term_out->dflags = (uint32_t)((term ? CL_DONE_TERMINATED : 0) | (trunc ? CL_DONE_TRUNCATED : 0));
  }
  if (live && done) {
    if (has_term && !rows_fast) store_obs<real>(p.term_obs, oo, p.obs_es, p.obs_cs, i, obs, E::OBS, obs64);
    if (!host_rows) {
      if (p.last_ep_ret) p.last_ep_ret[i] = ep_ret;   // tested only when an episode ends
      if (p.last_ep_len) p.last_ep_len[i] = ep_len;
    }
    if (autoreset) {
      E::reset(s, p, PLAIN ? make_stream(p, i, step) : rng, obs);
      ep_len = 0;
      ep_ret = 0.0;
      fin = true;
    }
  }
  // warp-uniform: contiguous float32 rows -> coalesced vector stores through shared memory
  if (rows_fast)
    store_obs_rows_warp<real, E::OBS>(sm_rows, (float*)p.obs + oo, i - (int64_t)lane, p.n, lane, obs);
  if (live) {
    const uint8_t dflags = (uint8_t)((term ? CL_DONE_TERMINATED : 0) | (trunc ? CL_DONE_TRUNCATED : 0));
    if (PLAIN && CL_PLAIN_DEFER) {
      // emitted at the top of the next interval (or by the caller after the last one)
    } else if (PLAIN) {
      const int64_t np = p.n_pad, row = (int64_t)t * np + i;
      float* o = (float*)p.obs + (int64_t)t * (E::OBS * np) + i;
#pragma unroll
      for (int c = 0; c < E::OBS; ++c) o[c * np] = (float)obs[c];
      ((real*)p.reward)[row] = rew;
      p.done[row] = dflags;
    } else {
      if (p.obs && !rows_fast) store_obs<real>(p.obs, oo, p.obs_es, p.obs_cs, i, obs, E::OBS, obs64);
      if (p.reward) {
        const int64_t ro = (ROLL ? t * p.rew_ts : 0) + i;
        if (p.reward_f32) ((float*)p.reward)[ro] = (float)rew;
        else ((real*)p.reward)[ro] = rew;
      }
      if (p.done) p.done[(ROLL ? t * p.done_ts : 0) + i] = dflags;
    }
  }
  if (PLAIN && CL_PLAIN_DEFER) {
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) pend->obs[c] = obs[c];
    pend->rew = rew;
    pend->dflags = (uint32_t)((term ? CL_DONE_TERMINATED : 0) | (trunc ? CL_DONE_TRUNCATED : 0));
    pend->t = t;
    pend->valid = 1u;
  }
  // the observation the env is in now (the reset observation where it auto-reset): the policy rollout's
  // next input.  Every other caller leaves obs_out null and the copy compiles away.
  if (obs_out != nullptr) {
#pragma unroll
    for (int c = 0; c < E::OBS; ++c) obs_out[c] = obs[c];
  }
  return dall;
}

template <class E>
__device__ __forceinline__ void synth_action(const KParams& p, const Stream& rng, float* a) {
  const u32x4 r = rng.draw(TAG_ACTION);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int c = 0; c < E::ACT; ++c) a[c] = p.synth_amp * (2.0f * u01_24(w[c & 3]) - 1.0f);
}

// ---- streamed host mode: the relay ----------------------------------------------------------
// Mirrors the pinned progress words of the staging lanes ((gen << 8) | slices of that lane staged so far;
// host_copy.h) into device memory until every lane is complete: relay thread k reads lane k's word (the
// system-scope reads of the lanes are in flight together) and is the only writer of its device copy.  The
// warp is also the judge of whether streaming works at all: if NO lane has published anything within 20 ms of
// its start, the CPU is evidently not running concurrently with the GPU work (a profiler or
// CUDA_LAUNCH_BLOCKING made the launches synchronous, so the staging loop only starts after the kernels have
// finished).  It then writes count 255 = "called off" to every lane: every block of the step kernel exits
// before storing anything (no block can have passed its wait: nothing was mirrored), *host_err = 2 tells
// cl_step_host_wait to redo the step from the (by then complete) staging buffer without streaming and to
// keep this context out of streamed mode.  The decision is a warp vote taken in the same loop iteration by
// all lanes, so "called off" and "a lane was mirrored" exclude each other.
// *host_err = 1: published partially and then nothing for 2 s -- unrecoverable, reported as an error.
// Runs either as block 0 of the step kernel itself (KParams::act_host_words, one launch per step) or as the
// one-warp kernel k_relay on a side stream.
static __device__ __noinline__ void relay_lanes(const uint32_t* host_words, uint32_t* dev_words, uint32_t gen, uint32_t lanes,
                                         uint32_t spl, uint32_t nslices, uint32_t* host_err) {
  const uint32_t k = threadIdx.x;
  if (k >= lanes) return;
  const unsigned mask = lanes >= 32u ? 0xffffffffu : ((1u << lanes) - 1u);
  const uint32_t first = k * spl;
  const uint32_t want = first >= nslices ? 0u : (nslices - first < spl ? nslices - first : spl);
  const uint32_t* host_word = host_words + (size_t)k * 16u;   // CL_STAGE_WORD_STRIDE
  uint32_t last = 0, polls = 0;
  uint64_t t0 = 0, t1 = 0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
    if (last < want) {
      const uint32_t v = ld_acquire_sys_u32(host_word);   // one system-scope read per lane per ~4 us: the only ones on the GPU
      if ((v >> 8) == gen && (v & 255u) > last && (v & 255u) <= want) {
        last = v & 255u;
        *(volatile uint32_t*)(dev_words + k) = v;
        __threadfence();
      }
    }
    if (__all_sync(mask, last >= want)) return;
    if ((++polls & 7u) == 0u) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      const uint64_t waited = __shfl_sync(mask, t1 - t0, 0);
      const bool none = !__any_sync(mask, last > 0u);
      if ((none && waited > 20000000ull) || waited > 2000000000ull) {
        if (last < want) {
          *(volatile uint32_t*)(dev_words + k) = (gen << 8) | 255u;
          __threadfence();
        }
        __syncwarp(mask);
        if (k == 0) *host_err = none ? 2u : 1u;
        return;
      }
    }
  }
}

// ---- the static step / rollout kernel: thread i owns env i for the whole launch ----------

// Resident 256-thread blocks per SM the SINGLE-STEP kernel is compiled for (0 = leave it to ptxas).
// The parity kinds' single steps are HBM-bound: what counts is bytes in flight, i.e. occupancy, so
// their register budget is capped at 64 (4 blocks) or 48 (5 blocks) -- measured at 1 Mi envs:
// hr_sync 0.72 -> 0.76 of the copy bandwidth, pmsm_sync 0.61 -> 0.75, pmsm_classic 0.67 -> 0.68,
// lorenz3 0.87 -> 0.88; 5 blocks cost lorenz3_pair / lorenz4_pair 2 % (spills), so they stay at 4.
template <class E> struct StepMinBlocks { enum { value = 0 }; };
// Kinds whose episodes end in a large share of the env-warps every step (memristive pair under full-range
// forcing): k_step accumulates the episode statistics per block in shared memory and flushes once -- 65 -> 49 us
// at 1 Mi envs.  Everywhere else the two block barriers and the flush cost 3-5 % of a 25-40 us step for
// nothing (measured, profiles/r02_sweep_block_stats.jsonl), so it is a per-kind choice.
template <class E> struct StepBlockStats { enum { value = 0 }; };

template <class E, bool ROLL, bool PLAIN = false>
__global__ void __launch_bounds__(256, ROLL ? 0 : StepMinBlocks<E>::value) k_step(const KParams p) {
  extern __shared__ __align__(16) float sm_rows_all[];  // [warps per block][32 * OBS], row-store staging
  constexpr bool BLKSTATS = StepBlockStats<E>::value != 0;
  __shared__ double s_stats[BLKSTATS ? CL_NSTATS : 1];   // episode statistics of this block
  if (BLKSTATS) {
    if (threadIdx.x < CL_NSTATS) s_stats[threadIdx.x] = 0.0;
    __syncthreads();
  }
  // streamed host mode with the relay inside this launch: block 0 is the relay (dispatched first, so it is
  // resident whatever the grid size), env blocks follow
  const bool relay_inside = !ROLL && p.act_host_words != nullptr;   // block-uniform
  if (relay_inside && blockIdx.x == 0) {
    if (threadIdx.x < 32)
      relay_lanes(p.act_host_words, const_cast<uint32_t*>(p.act_ready), p.act_gen, (uint32_t)p.act_lanes,
                  (uint32_t)p.act_lane_slices, (uint32_t)p.act_nslices, p.host_err);
    return;
  }
  const int64_t i = p.i_begin + (int64_t)(blockIdx.x - (relay_inside ? 1u : 0u)) * blockDim.x + threadIdx.x;
  const bool live = i < p.n;
  const unsigned lane = threadIdx.x & 31u;
  float* sm_rows = sm_rows_all + (threadIdx.x >> 5) * (32 * E::OBS);

  typename E::S s = {};
  int32_t ep_len = 0;
  double ep_ret = 0.0;
  if (live) {
    E::load(s, p, i);
    ep_len = p.ep_len[i];
    ep_ret = p.ep_return[i];
  }
  E::prepare(s, p, live);  // executed by all 32 lanes (may vote)
  const bool obs64 = !PLAIN && (p.flags & CL_F_OBS_F64) != 0;
  const bool autoreset = PLAIN || (p.flags & CL_F_AUTORESET) != 0;
  const bool want_noise = !PLAIN && E::NOISE > 0 && E::uses_noise(p);
  const int T = ROLL ? p.T : 1;
  const bool streamed = !ROLL && p.act_ready != nullptr;   // block-uniform
  if (streamed) {
    // Streamed host mode: this kernel was launched BEFORE the CPU finished staging the caller's action
    // array into the pinned buffer.  The slices (act_slice_envs envs each, a whole number of blocks) are dealt
    // out to staging lanes of act_lane_slices slices, one CPU thread each; every lane publishes the number of
    // its slices staged so far in a pinned word of its own; k_relay (one warp, side stream) mirrors those
    // words into device memory, and every block polls the DEVICE copy of its lane: uncached reads of host memory
    // cost ~4 us each and are served one at a time (measured: 1 ms per step when all 256 blocks polled
    // the host word themselves), a device word is an L2 hit.  The state loads above are already in
    // flight meanwhile.  If the relay reports that the CPU is not publishing at all (launches made
    // synchronous by a profiler or CUDA_LAUNCH_BLOCKING: the CPU cannot stage while the kernel runs) every
    // block leaves before it has stored anything and cl_step_host_wait redoes the step without streaming.
    __shared__ int s_abort;
    if (threadIdx.x == 0) {
      const uint32_t slice = (uint32_t)((i - p.i_begin) / p.act_slice_envs);
      const uint32_t spl = p.act_lane_slices > 0 ? (uint32_t)p.act_lane_slices : 0xffffffffu;
      const uint32_t need = slice % spl + 1u;
      const volatile uint32_t* word = p.act_ready + slice / spl;
      uint64_t t0 = 0, t1 = 0;
      uint32_t polls = 0;
      int ab = 0;
      for (;;) {
        const uint32_t v = *word;
        if ((v >> 8) == p.act_gen) {
          const uint32_t cnt = v & 255u;
          if (cnt == 255u) { ab = 1; break; }   // the relay called the step off (see k_relay): leave without a trace
          if (cnt >= need) break;
        }
        __nanosleep(200);
        if ((++polls & 63u) == 0u) {
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
          if (t0 == 0) t0 = t1;
          if (t1 - t0 > 3000000000ull) { if (p.host_err) *p.host_err = 1u; ab = 1; break; }
        }
      }
      __threadfence();   // the relay's device store is ordered after its (system-scope) read of the host word
      s_abort = ab;
    }
    __syncthreads();
    if (s_abort) return;   // nothing has been stored yet
  }

  // actions are fetched one control interval ahead; this only hides their latency while
  // scoreboard slots are free (ptxas drains the loads before long bodies, DESIGN.md section 5) --
  // the dynamic kernel below stages them through shared memory instead
  float a_next[E::ACT];
#pragma unroll
  // Streamed mode: ordinary (L1-allocating) loads on purpose.  The rows of this block are whole 128-byte
  // lines nobody touched before the flag above was seen (L1 is invalidated at launch), so they are fetched
  // fresh; volatile loads instead re-fetch every 32-byte sector over PCIe for each of the ACT strided
  // loads of a row -- measured 1 ms per step at 65,536 envs (request-rate bound).
  for (int c = 0; c < E::ACT; ++c)
    a_next[c] = (live && (PLAIN || p.action != nullptr)) ? p.action[i * p.act_es + c * p.act_cs] : 0.0f;

  unsigned bad_acc = 0u;
  bool fin = E::finite(s);
  const uint64_t step0 = step_base(p);
  PlainPending<E> pend;
  pend.begin(p, i, 0);
  auto intervals = [&](auto spec_tag) {
    constexpr int SPEC = decltype(spec_tag)::value;
    for (int t = 0; t < T; ++t) {
      const uint64_t step = step0 + (uint64_t)t;
      float a[E::ACT];
      if (ROLL && !PLAIN && p.action == nullptr) {
        synth_action<E>(p, make_stream(p, i, step), a);
      } else {
#pragma unroll
        for (int c = 0; c < E::ACT; ++c) a[c] = a_next[c];
        if (ROLL && live && t + 1 < T) {
#pragma unroll
          for (int c = 0; c < E::ACT; ++c)
            a_next[c] = p.action[(int64_t)(t + 1) * p.act_ts + i * p.act_es + c * p.act_cs];
        }
      }
      const unsigned dall = env_interval<E, ROLL, PLAIN, SPEC>(s, ep_len, ep_ret, p, i, live, lane, t, step, a, want_noise, obs64, autoreset, bad_acc, sm_rows, fin, &pend, BLKSTATS ? s_stats : nullptr);
      if (!ROLL && !PLAIN && p.warp_done != nullptr && dall && lane == 0) p.warp_done[i >> 5] = 1;
    }
  };
  if constexpr (PLAIN) {
    if (E::spec(s, p) == 1) intervals(SpecTag<1>{});
    else intervals(SpecTag<0>{});
    if (CL_PLAIN_DEFER) plain_emit<E, false>(p, i, live, pend);   // the last interval's outputs
  } else {
    intervals(SpecTag<0>{});
  }
  if (bad_acc && lane == 0) atomicAdd(BLKSTATS ? &s_stats[CL_STAT_NONFINITE] : &p.stats[CL_STAT_NONFINITE], (double)bad_acc);
  if (live) {
    E::store(s, p, i);
    p.ep_len[i] = ep_len;
    p.ep_return[i] = ep_ret;
  }
  if (BLKSTATS) {
    __syncthreads();
    if (threadIdx.x < CL_NSTATS && s_stats[threadIdx.x] != 0.0) atomicAdd(&p.stats[threadIdx.x], s_stats[threadIdx.x]);
  }
}

// ---- the dynamic rollout kernel ---------------------------------------------------------
// At 65,536 envs there are 2048 env-warps for 148 x 4 = 592 warp schedulers: 3.46 each, so a
// static thread<->env mapping leaves every scheduler waiting for the ones that hold 4 (86.5 %
// balance; partial warps cost a full FP64 issue, tools/dfma_probe.cu).  Here the launch is cut
// into tasks (env-warp e, chunk c of `dyn_chunk` control intervals); persistent worker warps
// (3 per scheduler at 65,536 envs: fewer workers than env-warps) pull tasks from an atomic counter in c-major order.  Chunk c of an env-warp
// may only start after chunk c-1 finished (possibly on another SM): the finishing warp publishes
// progress[e] with a release store, the next one reads it with an acquire load and
// reads the state planes with L1-bypassing loads.  A waiting warp only ever waits for a task
// with a smaller index, which some running (or finished) warp already owns, so the scheme cannot
// deadlock whatever the residency.
// The chunk's actions are staged in shared memory by bulk async copies (cp.async.bulk ->
// UBLKCP, completion on an mbarrier) issued one task ahead: no register scoreboard is involved,
// which removes the loop-head stall ptxas attaches to prefetching LDGs
// (profiles/r01_rollout_ncu_source_stalls.txt).

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra WAIT_LOOP;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// Every wait loop of the scheduling kernels is bounded: a protocol bug must end in a launch failure
// (trap -> cudaErrorLaunchFailure at the next synchronisation), never in a kernel that spins forever.
__device__ __forceinline__ void spin_guard(uint32_t& spins) {
  if (++spins > (1u << 24)) __trap();
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n.reg .pred P1;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
      "selp.u32 %0, 1, 0, P1;\n}\n"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

template <class E, bool PLAIN = false>
__global__ void __launch_bounds__(128) k_rollout_dyn(const KParams p) {
  extern __shared__ __align__(128) unsigned char dyn_smem[];
  __shared__ __align__(16) float sm_rows_all[4][32 * E::OBS];
  const unsigned lane = threadIdx.x & 31u;
  const int wib = threadIdx.x >> 5;
  float* sm_rows = sm_rows_all[wib];
  const int wpb = blockDim.x >> 5;
  const int Tc = p.dyn_chunk;
  const int per_buf = Tc * E::ACT * 32;  // floats
  float* abuf = (float*)dyn_smem + (size_t)wib * per_buf;
  uint64_t* mbar = (uint64_t*)(dyn_smem + (size_t)wpb * per_buf * sizeof(float)) + wib;
  const bool tma = PLAIN || p.dyn_tma != 0;
  if (tma) {
    if (lane == 0) {
      mbar_init(&mbar[0], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
  }
  const bool obs64 = !PLAIN && (p.flags & CL_F_OBS_F64) != 0;
  const bool autoreset = PLAIN || (p.flags & CL_F_AUTORESET) != 0;
  const bool want_noise = !PLAIN && E::NOISE > 0 && E::uses_noise(p);
  const uint32_t W = (uint32_t)p.dyn_nwarps, total = W * (uint32_t)p.dyn_nchunks;

  auto grab = [&]() -> uint32_t {
    uint32_t q = 0;
    if (lane == 0) q = atomicAdd(p.dyn_counter, 1u);
    return __shfl_sync(0xffffffffu, q, 0);
  };
  // stage the actions of task q into buffer b: lanes 0..len*ACT-1 issue one 128 B copy each
  auto stage = [&](uint32_t q, int b) {
    const uint32_t e = q % W, c = q / W;
    const int t0 = (int)c * Tc;
    const int len = min(Tc, p.T - t0);
    if (lane == 0) mbar_expect_tx(&mbar[b], (uint32_t)(len * E::ACT * 128));
    __syncwarp();
    for (int k = (int)lane; k < len * E::ACT; k += 32) {  // every expected byte must be issued
      const int tl = k / E::ACT, cc = k % E::ACT;
      const float* src = p.action + (int64_t)(t0 + tl) * p.act_ts + (int64_t)cc * p.act_cs + (int64_t)e * 32;
      bulk_g2s(abuf + (size_t)b * per_buf + ((size_t)tl * E::ACT + cc) * 32, src, 128u, &mbar[b]);
    }
  };

  // No task is reserved ahead of time: with W env-warps in c-major order and fewer than W
  // workers, the predecessor (same env-warp, previous chunk) of a freshly grabbed task was
  // grabbed W grabs -- i.e. W task completions -- earlier, so it has finished and the dependency
  // wait below practically never spins (a reserve-ahead scheme doubled the in-flight window and
  // spent 20 % of its samples spinning: profiles/r01_dyn_ncu_source_stalls.txt).
  uint32_t phase = 0u;
  const uint64_t step0 = step_base(p);
  uint32_t q = grab();
  while (q < total) {
    const uint32_t e = q % W, c = q / W;
    const int t0 = (int)c * Tc;
    const int len = min(Tc, p.T - t0);
    const int64_t i = (int64_t)e * 32 + lane;
    const bool live = i < p.n;
    if (tma) {
      // the staging buffer was last read (generic proxy) by this warp in the previous task
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      stage(q, 0);
    }
    if (c > 0) {
      // acquire load: pairs with the writer's release store and orders the state loads below after
      // it, without waiting for this warp's own outstanding output stores (a fence.acq_rel would).
      // The warp barrier extends the ordering from lane 0 to the other lanes; all per-env loads
      // additionally bypass L1.
      if (lane == 0) {
        uint32_t spins = 0;
        while (ld_acquire_u32(p.dyn_progress + e) < c) { __nanosleep(32); spin_guard(spins); }
      }
      __syncwarp();
    }
    typename E::S s = {};
    int32_t ep_len = 0;
    double ep_ret = 0.0;
    if (live) {
      E::load(s, p, i);
      ep_len = __ldcg(p.ep_len + i);
      ep_ret = __ldcg(p.ep_return + i);
    }
    E::prepare(s, p, live);
    if (tma) {
      mbar_wait(&mbar[0], phase);
      phase ^= 1u;
    }
    const float* ab = abuf;
    unsigned bad_acc = 0u;
    bool fin = E::finite(s);
    PlainPending<E> pend;
    pend.begin(p, i, t0);
    auto intervals = [&](auto spec_tag) {
      constexpr int SPEC = decltype(spec_tag)::value;
      for (int tl = 0; tl < len; ++tl) {
        const int t = t0 + tl;
        const uint64_t step = step0 + (uint64_t)t;
        float a[E::ACT];
        if (!PLAIN && p.action == nullptr) {
          synth_action<E>(p, make_stream(p, i, step), a);
        } else if (tma) {
#pragma unroll
          for (int cc = 0; cc < E::ACT; ++cc) a[cc] = ab[(tl * E::ACT + cc) * 32 + lane];
        } else {
#pragma unroll
          for (int cc = 0; cc < E::ACT; ++cc)
            a[cc] = live ? p.action[(int64_t)t * p.act_ts + i * p.act_es + cc * p.act_cs] : 0.0f;
        }
        env_interval<E, true, PLAIN, SPEC, true>(s, ep_len, ep_ret, p, i, live, lane, t, step, a, want_noise, obs64, autoreset, bad_acc, sm_rows, fin, &pend);
      }
    };
    if constexpr (PLAIN) {
      if (E::spec(s, p) == 1) intervals(SpecTag<1>{});
      else intervals(SpecTag<0>{});
    } else {
      intervals(SpecTag<0>{});
    }
    if (bad_acc && lane == 0) atomicAdd(&p.stats[CL_STAT_NONFINITE], (double)bad_acc);
    bad_acc = 0u;
    if (live) {
      E::store(s, p, i);
      p.ep_len[i] = ep_len;
      p.ep_return[i] = ep_ret;
    }
    // publish: the warp barrier orders every lane's stores before lane 0's release store
    __syncwarp();
    if (lane == 0) st_release_u32(p.dyn_progress + e, c + 1u);
    if constexpr (PLAIN) {
      // the last interval's output streams go out AFTER the hand-off: the release only has to wait
      // for the state planes (nobody reads the output streams through `progress`)
      if (CL_PLAIN_DEFER) plain_emit<E, true>(p, i, live, pend);
    }
    q = grab();
  }
}


// ---- the SM-local rollout kernel ----------------------------------------------------------
// Same goal as k_rollout_dyn -- 2048 env-warps spread evenly over 592 schedulers -- but nothing crosses
// an SM.  Block b (one per SM: >= 120 KB of shared memory each keeps two blocks off one SM) owns a
// contiguous range of 13-14 env-warps for the whole launch:
//  * RESIDENTS: worker warp w integrates env-warp w from the first to the last control interval with
//    its state in registers -- no task switch, no hand-off; 12 workers = 3 per scheduler.
//  * GUESTS: the 1-2 env-warps an SM owns beyond its workers are cut into chunks of Tc intervals; their
//    state, episode counters and hand-off words live in shared memory.  After every nres / g of its own
//    chunks (Bresenham, phase-shifted per worker) a worker parks its resident in shared memory, runs ONE
//    guest chunk and resumes -- so every worker does (1 + g / nres) x T intervals and all finish
//    together, with ~7x fewer task switches than a queue holding every env-warp (that version spent
//    ~9 % of its stall samples in per-task code: queue atomic, index arithmetic, hand-off wait, state and
//    pointer set-up, a 23-iteration uniform loop issuing the chunk's bulk copies).
//  * A guest hand-off is shared-memory only: chunk counter + mbarrier (arrive = release, try_wait =
//    acquire, CTA scope) -- no GPU-scope release/acquire through L2 as in k_rollout_dyn (CCTL.IVALL,
//    ERRBAR and cold state loads: ~11 % of its stall samples), and no MEMBAR at all.
//  * ACTIONS: per env-warp double buffer in shared memory; a chunk [Tc][ACT][32] f32 arrives by ONE
//    3-D tensor copy (cp.async.bulk.tensor, completion on the buffer's mbarrier) issued by one lane a
//    whole chunk ahead; rows past T are zero-filled by the copy engine.  Without a tensor map (driver
//    entry point missing) the chunk is fetched by one 128 B bulk copy per row.
// Cost: SMs owning 14 env-warps run 1.2 % longer than the 13.84 average.
// Plain rollout I/O shape only (PlainRollout<E>): launch_env falls back to k_rollout_dyn otherwise.

template <class E>
struct SmLayout {
  typedef typename E::real real;
  size_t act, state, ep_ret, ep_len, mbar, prog, total;
  __host__ __device__ SmLayout(int cnt, int chunk) {
    size_t o = 0;
    act = o;    o += (size_t)cnt * 2 * chunk * E::ACT * 32 * sizeof(float);   // 128 B multiples
    state = o;  o += (size_t)cnt * E::NSTATE * 32 * sizeof(real);
    ep_ret = o; o += (size_t)cnt * 32 * sizeof(double);
    ep_len = o; o += (size_t)cnt * 32 * sizeof(int32_t);
    mbar = o;   o += (size_t)cnt * 3 * sizeof(uint64_t);                      // 2 action buffers + hand-off
    prog = o;   o += ((size_t)cnt + 1) * sizeof(uint32_t);                    // chunks finished per env-warp, guest queue
    total = (o + 127) & ~(size_t)127;
  }
};

__device__ __forceinline__ void tma_load_3d(void* dst, const void* tmap, int x, int y, int z, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(smem_u32(dst)), "l"(tmap), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
      : "memory");
}

#ifndef CL_SM_THREADS
#define CL_SM_THREADS 576
#endif
#ifndef CL_SM_MINB
#define CL_SM_MINB 0
#endif
// Launch bound (576, no minimum-blocks hint; blocks have at most 16 warps): a ptxas scheduling lottery.
// With this bound (92 registers) the two x-multiplied DFMAs of every RHS evaluation end up adjacent, so
// 106 of the 128 three-register DFMAs of an interval find one source in the operand reuse cache (2.2
// instead of 3 issue cycles, tools/dfma_probe.cu); (512, 0) gives 1 of 128, (384, 0) 76 of 128 --
// checked on the built library by tests/test_sass.py with tools/sass_mix.py
template <class E>
// The tensor map is its own __grid_constant__ parameter (the descriptor must be addressable in param
// space); KParams stays an ordinary by-value parameter -- as a __grid_constant__ it faulted on sm_100a.
__global__ void __launch_bounds__(CL_SM_THREADS, CL_SM_MINB) k_rollout_sm(const KParams p,
                                                                         const __grid_constant__ CUtensorMap tmap) {
  typedef typename E::real real;
  extern __shared__ __align__(128) unsigned char sm_raw[];
  const unsigned lane = threadIdx.x & 31u;
  const int wib = threadIdx.x >> 5, nres = blockDim.x >> 5;     // one resident env-warp per worker warp
  const int W = p.dyn_nwarps, G = (int)gridDim.x, b = (int)blockIdx.x;
  const int qn = W / G, rn = W % G;
  const int e0 = b * qn + (b < rn ? b : rn);
  const int cnt = qn + (b < rn ? 1 : 0);                       // >= nres by construction (host)
  const int cmax = qn + (rn ? 1 : 0);
  const int ng = cnt - nres;                                   // guests of this block
  // Chunk schedule of local env-warp le: a first chunk of f(le) = 1 + le * Tc / cnt control intervals,
  // then chunks of Tc: chunk boundaries (action-buffer swaps, guest slots) of the warps sharing a
  // scheduler do not coincide, and the guests' last chunks have mixed lengths.  Every env-warp has the
  // same number of chunks; trailing chunks past T are empty.
  // Guests use chunks of Tg = Tc / sm_gdiv intervals: every guest chunk a worker takes or does not take is
  // that worker's imbalance at the end of the launch (all workers wait for the last one at the final barrier).
  const int Tc = p.sm_chunk, Tg = max(1, Tc / max(1, p.sm_gdiv));
  const int nchunks = 1 + (p.T - 1 + Tc - 1) / Tc;          // residents
  const int nchunks_g = 1 + (p.T - 1 + Tg - 1) / Tg;        // guests
  auto chunk_t0 = [&](int f, int c, int tc) { return c == 0 ? 0 : min(p.T, f + (c - 1) * tc); };
  auto chunk_len = [&](int f, int c, int tc) { return min(c == 0 ? f : tc, p.T - chunk_t0(f, c, tc)); };
  const SmLayout<E> L(cmax, Tc);
  float* const act = (float*)(sm_raw + L.act);
  real* const st = (real*)(sm_raw + L.state);
  double* const s_ret = (double*)(sm_raw + L.ep_ret);
  int32_t* const s_len = (int32_t*)(sm_raw + L.ep_len);
  uint64_t* const mbar = (uint64_t*)(sm_raw + L.mbar);     // [le][0..1]: action buffers, [le][2]: hand-off
  volatile uint32_t* const prog = (volatile uint32_t*)(sm_raw + L.prog);
  uint32_t* const counter = (uint32_t*)(sm_raw + L.prog) + cmax;
  const int per_buf = Tc * E::ACT * 32;  // floats

  // ---- prologue: barriers, queue words, the block's state planes -> shared memory
  for (int k = threadIdx.x; k < cnt * 3; k += blockDim.x) mbar_init(&mbar[k], 1);
  for (int k = threadIdx.x; k <= cmax; k += blockDim.x) ((uint32_t*)(sm_raw + L.prog))[k] = 0u;
  for (int k = threadIdx.x; k < cnt * 32; k += blockDim.x) {
    const int le = k >> 5, ln = k & 31;
    const int64_t i = (int64_t)(e0 + le) * 32 + ln;   // < n_pad: the planes are padded
#pragma unroll
    for (int c = 0; c < E::NSTATE; ++c) st[(le * E::NSTATE + c) * 32 + ln] = ldp<real>(p, c, i);
    s_ret[k] = __ldcg(p.ep_return + i);
    s_len[k] = __ldcg(p.ep_len + i);
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();

  // stage the actions of chunk c of local env-warp le into its buffer (c & 1)
  auto stage = [&](int le, int f, int c, int tc) {
    const int t0 = chunk_t0(f, c, tc);
    uint64_t* bar = &mbar[le * 3 + (c & 1)];
    float* dst = act + (size_t)(le * 2 + (c & 1)) * per_buf;
    if (p.sm_tmap_ok) {
      // one tensor copy: box (32 envs, ACT channels, Tc intervals); the whole box counts towards the
      // barrier's transaction bytes, rows past T arrive as zeros
      if (lane == 0) {
        mbar_expect_tx(bar, (uint32_t)(per_buf * sizeof(float)));
        tma_load_3d(dst, &tmap, (e0 + le) * 32, 0, t0, bar);
      }
    } else {
      const int len = chunk_len(f, c, tc);
      if (lane == 0) mbar_expect_tx(bar, (uint32_t)(len * E::ACT * 128));
      __syncwarp();
      for (int k = (int)lane; k < len * E::ACT; k += 32) {  // every expected byte must be issued
        const int tl = k / E::ACT, cc = k % E::ACT;
        const float* src = p.action + (int64_t)(t0 + tl) * p.act_ts + (int64_t)cc * p.act_cs + (int64_t)(e0 + le) * 32;
        bulk_g2s(dst + (tl * E::ACT + cc) * 32, src, 128u, bar);
      }
    }
  };
  auto wait_actions = [&](int le, int c) {
    uint64_t* bar = &mbar[le * 3 + (c & 1)];
    const uint32_t parity = (uint32_t)(c >> 1) & 1u;
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) spin_guard(spins);
  };
  for (int le = wib; le < cnt; le += nres) { const int tc = le < nres ? Tc : Tg; stage(le, 1 + le * tc / cnt, 0, tc); }

  const uint64_t step0 = step_base(p);
  unsigned bad_acc = 0u;

  // the control intervals of one chunk of one env-warp; state, episode counters and the pending output
  // record stay in the caller's registers
  auto run_chunk = [&](typename E::S& s, int32_t& ep_len, double& ep_ret, bool& fin, PlainPending<E>& pend,
                       const int le, const int c, const int t0, const int len, const int64_t i, const bool live) {
    const float* ab = act + (size_t)(le * 2 + (c & 1)) * per_buf;
    auto intervals = [&](auto spec_tag) {
      constexpr int SPEC = decltype(spec_tag)::value;
      for (int tl = 0; tl < len; ++tl) {
        const int t = t0 + tl;
        const uint64_t step = step0 + (uint64_t)t;
        float a[E::ACT];
#pragma unroll
        for (int cc = 0; cc < E::ACT; ++cc) a[cc] = ab[(tl * E::ACT + cc) * 32 + lane];
        env_interval<E, true, true, SPEC, true>(s, ep_len, ep_ret, p, i, live, lane, t, step, a, false, false, true,
                                                bad_acc, nullptr, fin, &pend);
      }
    };
    if (E::spec(s, p) == 1) intervals(SpecTag<1>{});
    else intervals(SpecTag<0>{});
  };

  // ---- worker loop: own chunks in order, a guest chunk whenever the Bresenham credit says so.
  // ONE call site of run_chunk (the unrolled interval body is ~13 KB of code per specialisation; a second
  // inlined copy would double the instruction-cache footprint of the hot loop).
  const uint32_t g_total = (uint32_t)ng * (uint32_t)nchunks_g;
  const int g_credit = ng * (Tc / Tg);     // guest chunks owed per round of own chunks, times nres
  typename E::S s = {};
  int32_t ep_len = 0;
  double ep_ret = 0.0;
  bool fin = true;
  PlainPending<E> pend;
  pend.valid = 0u;
  int in_regs = -1;                     // local env-warp whose state is in this warp's registers
  int c_own = 0;
  int credit = (wib * g_credit) % nres; // phase shift: the workers' guest slots interleave evenly in time
  bool guests_left = ng > 0, want_guest = false;
  for (;;) {
    int le, c;
    bool guest;
    if (want_guest) {
      uint32_t q = 0;
      if (lane == 0) q = atomicAdd(counter, 1u);
      q = __shfl_sync(0xffffffffu, q, 0);
      if (q >= g_total) { guests_left = false; want_guest = false; continue; }
      guest = true; le = nres + (int)(q % (uint32_t)ng); c = (int)(q / (uint32_t)ng);
    } else if (c_own < nchunks) {
      guest = false; le = wib; c = c_own;
    } else if (guests_left) {
      want_guest = true;                // own env-warp finished: drain what is left of the guests
      continue;
    } else {
      break;
    }
    const int tc = guest ? Tg : Tc, nch = guest ? nchunks_g : nchunks;
    const int f = 1 + le * tc / cnt;
    const int t0 = chunk_t0(f, c, tc), len = chunk_len(f, c, tc);
    const int64_t i = (int64_t)(e0 + le) * 32 + lane;
    const bool live = i < p.n;
    if (guest && c > 0) {
      // Hand-off from the warp that ran chunk c-1 of this guest.  Two steps:
      //  1. wait until exactly c chunks are counted in prog[le] (plain shared-memory word: a phase
      //     PARITY alone cannot tell "chunk c-1 finished" from "chunk c-3 finished" when several
      //     chunks of one env-warp are in hand);
      //  2. the completion of chunk c-1 is phase c-1 of the env-warp's hand-off mbarrier, whose arrive
      //     follows the counter store: try_wait on that phase is the acquire (arrive = release, CTA
      //     scope) that orders the state loads below.  No MEMBAR -- a __threadfence_block() here also
      //     waits for the warp's outstanding global output stores, ~0.5 us per task.
      uint32_t spins = 0;
      if (lane == 0) {
        while (prog[le] != (uint32_t)c) { __nanosleep(32); spin_guard(spins); }
      }
      __syncwarp();
      uint64_t* hb = &mbar[le * 3 + 2];
      const uint32_t parity = (uint32_t)(c - 1) & 1u;
      while (!mbar_try_wait(hb, parity)) spin_guard(spins);
    }
    // Buffer (c+1)&1 was last READ (LDS, generic proxy) during chunk c-1 -- by this warp (resident) or by
    // the warp whose hand-off we just acquired (guest); those loads had returned their values long
    // before.  No fence.proxy.async here -- it compiles to MEMBAR.ALL.CTA, which also waits for this
    // warp's outstanding global output stores; the write-after-read direction is ordered by the mbarrier
    // alone (the usual TMA pipeline pattern).
    if (c + 1 < nch) stage(le, f, c + 1, tc);
    if (in_regs != le) {
      E::load_sm(s, st + (size_t)le * E::NSTATE * 32, lane);
      ep_len = s_len[le * 32 + lane];
      ep_ret = s_ret[le * 32 + lane];
      E::prepare(s, p, live);
      fin = E::finite(s);
      pend.begin(p, i, t0);
      in_regs = le;
    }
    wait_actions(le, c);
    run_chunk(s, ep_len, ep_ret, fin, pend, le, c, t0, len, i, live);
    bool park;
    if (guest) {
      park = true;
      want_guest = false;               // one guest chunk per slot
    } else {
      c_own += 1;
      credit += g_credit;
      want_guest = guests_left && credit >= nres && c_own < nchunks;
      if (want_guest) credit -= nres;
      park = want_guest || c_own == nchunks;
    }
    if (park) {
      // state back to its shared-memory slot; a guest is then published to whichever warp runs its next
      // chunk (the warp barrier orders every lane's stores before lane 0's counter store and arrive)
      E::store_sm(s, st + (size_t)le * E::NSTATE * 32, lane);
      s_len[le * 32 + lane] = ep_len;
      s_ret[le * 32 + lane] = ep_ret;
      if (guest) {
        __syncwarp();
        if (lane == 0) {
          prog[le] = (uint32_t)c + 1u;
          mbar_arrive(&mbar[le * 3 + 2]);
        }
      }
      if (CL_PLAIN_DEFER) plain_emit<E, true>(p, i, live, pend);   // the last interval's outputs, after the hand-off
      pend.valid = 0u;
      in_regs = -1;
    }
  }
  if (bad_acc && lane == 0) atomicAdd(&p.stats[CL_STAT_NONFINITE], (double)bad_acc);

  // ---- epilogue: state planes and episode counters back to global memory
  __syncthreads();
  for (int k = threadIdx.x; k < cnt * 32; k += blockDim.x) {
    const int le = k >> 5, ln = k & 31;
    const int64_t i = (int64_t)(e0 + le) * 32 + ln;
    if (i < p.n) {
#pragma unroll
      for (int c = 0; c < E::NSTATE; ++c) stp<real>(p, c, i, st[(le * E::NSTATE + c) * 32 + ln]);
      p.ep_return[i] = s_ret[k];
      p.ep_len[i] = s_len[k];
    }
  }
}

template <class E>
__global__ void __launch_bounds__(256) k_reset(const KParams p) {
  typedef typename E::real real;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t step0 = step_base(p);
  if (i < p.n && (p.mask == nullptr || p.mask[i] != 0)) {
    typename E::S s = {};
    E::load(s, p, i);  // keeps persistent fields (Adam-dual state, per-env parameters)
    const Stream rng = make_stream(p, i, step0);
    real obs[E::OBS];
    E::reset(s, p, rng, obs);
    E::store(s, p, i);
    p.ep_len[i] = 0;
    p.ep_return[i] = 0.0;
    if (p.obs) store_obs<real>(p.obs, 0, p.obs_es, p.obs_cs, i, obs, E::OBS, (p.flags & CL_F_OBS_F64) != 0);
  }
}

template <class E>
__global__ void __launch_bounds__(256) k_init(const KParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  typename E::S s = {};
  const Stream rng = make_stream(p, i, 0);
  E::init_persistent(s, p, rng);
  E::store(s, p, i);
  p.ep_len[i] = 0;
  p.ep_return[i] = 0.0;
}

// Row-store fast path: contiguous float32 rows [N][OBS] whose every warp segment is 16-byte
// aligned (base pointer, and in rollouts the per-interval stride).  Decided once on the host.
template <class E>
inline bool rows_fast_ok(const KParams& p, bool rollout) {
  return p.obs != nullptr && !(p.flags & CL_F_OBS_F64) && p.obs_cs == 1 && p.obs_es == E::OBS &&
         ((uintptr_t)p.obs % 16) == 0 && (!rollout || (p.obs_ts % 4) == 0) &&
         ((uintptr_t)p.term_obs % 16) == 0;  // term_obs (if any) shares the obs layout
}

// Plain-rollout instantiation (see PlainRollout): decided once per launch on the host.
template <class E>
inline bool plain_rollout_ok(const KParams& p, int mode) {
  return PlainRollout<E>::value && !p.no_plain && E::NOISE == 0 && p.action != nullptr && p.obs != nullptr && p.obs_es == 1 &&
         p.obs_cs == p.n_pad && p.obs_ts == (int64_t)E::OBS * p.n_pad && p.rew_ts == p.n_pad && p.done_ts == p.n_pad &&
         !(p.flags & CL_F_OBS_F64) && !p.rows_fast && p.reward != nullptr && !p.reward_f32 && p.done != nullptr &&
         p.term_obs == nullptr &&
         (p.flags & CL_F_AUTORESET) && (mode != MODE_ROLLOUT_DYN || p.dyn_tma);
}

template <class E>
cudaError_t launch_env(const KParams& p_in, int mode, cudaStream_t st, int block) {
  KParams p = p_in;
  const bool roll = (mode == MODE_ROLLOUT || mode == MODE_ROLLOUT_DYN);
  p.rows_fast = (mode == MODE_STEP || roll) && rows_fast_ok<E>(p, roll) ? 1 : 0;
  constexpr bool HAS_PLAIN = PlainRollout<E>::value != 0;
  const bool plain = roll && plain_rollout_ok<E>(p, mode);
  if (p.host_plain_out) *p.host_plain_out = plain ? 1 : 0;
  p.host_plain_out = nullptr;
  const size_t row_smem = p.rows_fast ? (size_t)(block / 32) * 32 * E::OBS * sizeof(float) : 0;
  const unsigned grid = (unsigned)((p.n - p.i_begin + block - 1) / block);  // i_begin != 0 only for MODE_STEP
  const unsigned step_grid = grid + ((mode == MODE_STEP && p.act_host_words != nullptr) ? 1u : 0u);   // + the relay block
  switch (mode) {
    // dynamic smem only when observations go out as contiguous float32 rows (row-store staging)
    case MODE_STEP: k_step<E, false><<<step_grid, block, row_smem, st>>>(p); break;
    case MODE_ROLLOUT:
      if (plain) k_step<E, true, HAS_PLAIN><<<grid, block, row_smem, st>>>(p);
      else k_step<E, true><<<grid, block, row_smem, st>>>(p);
      break;
    case MODE_RESET: k_reset<E><<<grid, block, 0, st>>>(p); break;
    case MODE_INIT: k_init<E><<<grid, block, 0, st>>>(p); break;
    case MODE_ROLLOUT_DYN: {
      if constexpr (HAS_PLAIN) {
        if (plain && p.sm_grid > 0) {
          // SM-local scheduling: one block per SM (>= 120 KB of shared memory each keeps two blocks off one SM)
          const int cmax = (p.dyn_nwarps + p.sm_grid - 1) / p.sm_grid;
          size_t smem = SmLayout<E>(cmax, p.sm_chunk).total;
          if (smem < 120 * 1024) smem = 120 * 1024;
          if (smem <= 200 * 1024) {
            static bool attr_set = false;
            if (!attr_set) {
              cudaError_t e = cudaFuncSetAttribute(k_rollout_sm<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
              if (e != cudaSuccess) return e;
              attr_set = true;
            }
            if (p_in.host_plain_out) *p_in.host_plain_out |= 2;
            alignas(64) CUtensorMap tm;
            if (p.sm_tmap_ok && p.host_tmap) tm = *p.host_tmap;
            else { memset(&tm, 0, sizeof(tm)); p.sm_tmap_ok = 0; }
            p.host_tmap = nullptr;
            k_rollout_sm<E><<<(unsigned)p.sm_grid, (unsigned)p.sm_workers * 32, smem, st>>>(p, tm);
            break;
          }
        }
      }
      // block = 128 threads (one warp per scheduler), p.dyn_grid blocks, smem = action staging
      const size_t smem = (size_t)4 * p.dyn_chunk * E::ACT * 32 * sizeof(float) + 4 * sizeof(uint64_t);
      if (plain) k_rollout_dyn<E, HAS_PLAIN><<<(unsigned)p.dyn_grid, 128, smem, st>>>(p);
      else k_rollout_dyn<E><<<(unsigned)p.dyn_grid, 128, smem, st>>>(p);
      break;
    }
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

template <class E>
cudaError_t dyn_occupancy(int chunk, int* blocks_per_sm) {
  const size_t smem = (size_t)4 * chunk * E::ACT * 32 * sizeof(float) + 4 * sizeof(uint64_t);
  cudaError_t e = cudaFuncSetAttribute(k_rollout_dyn<E>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
  if (e != cudaSuccess) return e;
  int occ = 0, occ_plain = 1 << 30;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_rollout_dyn<E>, 128, smem);
  if (e != cudaSuccess) return e;
  if (PlainRollout<E>::value) {  // the worker grid must be resident whichever instantiation is launched
    e = cudaFuncSetAttribute(k_rollout_dyn<E, PlainRollout<E>::value != 0>, cudaFuncAttributePreferredSharedMemoryCarveout, 50);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_plain, k_rollout_dyn<E, PlainRollout<E>::value != 0>, 128, smem);
    if (e != cudaSuccess) return e;
  }
  *blocks_per_sm = occ < occ_plain ? occ : occ_plain;
  return cudaSuccess;
}

}  // namespace cl

// per-TU dispatch (implemented in tu_parity.cu / tu_northstar.cu)
cudaError_t cl_launch_parity(int kind, const cl::KParams& p, int mode, cudaStream_t st, int block);
cudaError_t cl_launch_northstar(int kind, const cl::KParams& p, int mode, cudaStream_t st, int block);
cudaError_t cl_occupancy_parity(int kind, int block, int* blocks_per_sm);
cudaError_t cl_occupancy_northstar(int kind, int block, int* blocks_per_sm);
cudaError_t cl_dyn_occupancy_parity(int kind, int chunk, int* blocks_per_sm);
cudaError_t cl_dyn_occupancy_northstar(int kind, int chunk, int* blocks_per_sm);
// tu_policy.cu
cudaError_t cl_launch_policy(int kind, const cl::KParams& p, const cl_policy& q, float act_lo, float act_hi,
                             cudaStream_t st, int sms);
cudaError_t cl_launch_policy_collect(int kind, const cl::KParams& p, const cl_policy& q, const cl_collect& col,
                                     float act_lo, float act_hi, cudaStream_t st, int sms);
cudaError_t cl_launch_policy_collect_norm(int kind, const cl::KParams& p, const cl_policy& q, const cl_collect& col,
                                          const cl_vecnorm_update& vn, float act_lo, float act_hi, cudaStream_t st,
                                          int sms);
int64_t cl_policy_collect_norm_bytes(int obs_dim, int64_t n);
cudaError_t cl_fma_peak_launch(int dtype_bytes, int grid, int block, int iters, void* sink, cudaStream_t st);
