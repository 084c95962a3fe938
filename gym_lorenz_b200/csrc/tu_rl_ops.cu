// Device-side versions of the SB3 machinery that sits directly around the env step in the
// reference's pipelines (SURVEY 8f ranks 1-3), so that observations / rewards never leave HBM:
//   * GAE(lambda)            -- stable_baselines3 2.7.1 RolloutBuffer.compute_returns_and_advantage
//                               (un-vendored; driven by code/train.py:112-120, gae_lambda=0.95)
//   * VecNormalize           -- running mean/var update + normalise + clip
//                               (code/lorenz_pmsm/train.py:118,170: norm_obs=True, clip_obs=10)
//   * VecFrameStack          -- code/lorenz_filter/train.py:115 (n_stack=4)
//   * evaluation metrics     -- code/lorenz_pmsm/test_evaluate.py:25-59,239-250,
//                               code/test_evaluate.py:136-145 (steady-state MAE/RMSE, settling
//                               time, control energy)
// All four are HBM-bound streaming kernels: one thread per env (coalesced [T][n] planes).
// Built with -fmad=false so that the float32 GAE recurrence rounds exactly like NumPy's.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <atomic>

#include "../../include/chaos_b200.h"
#include "rms_merge.cuh"

namespace {

// ---- GAE -------------------------------------------------------------------------------
// for step in reversed(range(T)):
//   nnt, nv = (1 - dones, last_values) if step == T-1 else (1 - episode_starts[step+1], values[step+1])
//   delta = rewards[step] + gamma * nv * nnt - values[step]
//   last = delta + gamma * gae_lambda * nnt * last
//   advantages[step] = last
// returns = advantages + values          (all float32; gamma, gamma*lambda weak scalars -> f32)
__global__ void __launch_bounds__(256) k_gae(const float* __restrict__ rew, const float* __restrict__ val,
                                             const float* __restrict__ starts, const float* __restrict__ last_val,
                                             const float* __restrict__ last_done, float gamma, float gl, int T,
                                             int64_t n, int64_t stride, float* __restrict__ adv,
                                             float* __restrict__ ret) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float last = 0.0f;
  float nnt = __fsub_rn(1.0f, last_done[i]);
  float nv = last_val[i];
  // The recurrence is serial in t, the loads are not: with one thread per env and only 65,536 envs the
  // kernel was latency-bound (ncu: 87 % long-scoreboard stalls, 3.1 TB/s).  The three input streams of U
  // consecutive steps are fetched first, then the U recurrence steps run out of registers.
  constexpr int U = 8;
  int t = T - 1;
  for (; t >= U - 1; t -= U) {
    float r[U], v[U], s[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t o = (int64_t)(t - k) * stride + i;
      r[k] = rew[o]; v[k] = val[o]; s[k] = starts[o];
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t o = (int64_t)(t - k) * stride + i;
      const float delta = __fsub_rn(__fadd_rn(r[k], __fmul_rn(__fmul_rn(gamma, nv), nnt)), v[k]);
      last = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nnt), last));
      adv[o] = last;
      ret[o] = __fadd_rn(last, v[k]);
      nnt = __fsub_rn(1.0f, s[k]);
      nv = v[k];
    }
  }
  for (; t >= 0; --t) {
    const int64_t o = (int64_t)t * stride + i;
    const float v = val[o];
    const float delta = __fsub_rn(__fadd_rn(rew[o], __fmul_rn(__fmul_rn(gamma, nv), nnt)), v);
    last = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nnt), last));
    adv[o] = last;
    ret[o] = __fadd_rn(last, v);
    nnt = __fsub_rn(1.0f, starts[o]);
    nv = v;
  }
}

// ---- running moments: per-feature sum(x - shift) and sum((x - shift)^2) over envs --------
template <int MAXD, typename TIN>
__global__ void __launch_bounds__(256) k_moments(const TIN* __restrict__ obs, int64_t es, int64_t cs, int64_t n,
                                                 int dim, const double* __restrict__ shift, double* __restrict__ out) {
  double s1[MAXD], s2[MAXD];
#pragma unroll
  for (int c = 0; c < MAXD; ++c) { s1[c] = 0.0; s2[c] = 0.0; }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int c = 0; c < MAXD; ++c) {
      if (c < dim) {
        const double d = (double)obs[i * es + c * cs] - shift[c];
        s1[c] += d;
        s2[c] += d * d;
      }
    }
  }
  // warp shuffle -> shared memory -> ONE atomic per block and feature: with an atomic per warp, 9,472 warps
  // queued on 12 addresses (ncu: 122 us for 25 MB, 91 % long-scoreboard) -- the same-address atomics, not
  // the reads, set the time
  __shared__ double sm_part[8][2 * MAXD];
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
#pragma unroll
  for (int c = 0; c < MAXD; ++c) {
    if (c < dim) {
      double a = s1[c], b = s2[c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
      }
      if (lane == 0) { sm_part[warp][c] = a; sm_part[warp][MAXD + c] = b; }
    }
  }
  __syncthreads();
  const int nwarp = blockDim.x >> 5;
  for (int k = threadIdx.x; k < 2 * dim; k += blockDim.x) {
    const int c = k < dim ? k : MAXD + (k - dim);
    double a = 0.0;
    for (int w = 0; w < nwarp; ++w) a += sm_part[w][c];
    atomicAdd(&out[k], a);
  }
}

// ---- normalise + clip: clip((x - mean) / sqrt(var + eps), -clip, clip).astype(float32) ----
// ROWS: the output is a contiguous, 16-byte aligned [N][dim] block (what a policy network reads): a
// warp's 32 rows are one run of 32*dim floats, written as whole float4 vectors through a shared-memory
// transpose instead of `dim` stores of 32 scattered 4-byte words each.
template <bool ROWS>
__global__ void __launch_bounds__(256) k_normalize(const float* __restrict__ in, int64_t ies, int64_t ics,
                                                   float* __restrict__ out, int64_t oes, int64_t ocs, int64_t n,
                                                   int dim, const double* __restrict__ mean,
                                                   const double* __restrict__ var, double eps, double clip) {
  extern __shared__ __align__(16) float sm_norm[];   // ROWS: [warps][32 * dim]
  // sqrt(var + eps) and the mean once per block (was: one f64 sqrt per element; ncu: FP64 + XU pipes 46 %
  // busy on a kernel that should only stream); the division stays a division, so the result keeps the
  // exact rounding of (x - mean) / sqrt(var + eps)
  __shared__ double sm_mean[48], sm_std[48];
  for (int c = threadIdx.x; c < dim && c < 48; c += blockDim.x) { sm_mean[c] = mean[c]; sm_std[c] = sqrt(var[c] + eps); }
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned lane = threadIdx.x & 31u;
  float* sm = sm_norm + (threadIdx.x >> 5) * (32 * dim);
  if (i < n) {
    for (int c = 0; c < dim; ++c) {
      const double m = c < 48 ? sm_mean[c] : mean[c], sd = c < 48 ? sm_std[c] : sqrt(var[c] + eps);
      double z = ((double)in[i * ies + c * ics] - m) / sd;
      z = z < -clip ? -clip : (z > clip ? clip : z);
      if (ROWS) sm[lane * dim + c] = (float)z;
      else out[i * oes + c * ocs] = (float)z;
    }
  }
  if (ROWS) {
    __syncwarp();
    const int64_t row0 = i - (int64_t)lane;
    const int64_t rows = n - row0;
    const int nflt = (int)(rows >= 32 ? 32 : (rows > 0 ? rows : 0)) * dim;
    float* dst = out + row0 * dim;
    for (int k = (int)lane * 4; k + 3 < nflt; k += 128)
      *reinterpret_cast<float4*>(dst + k) = *reinterpret_cast<const float4*>(sm + k);
    for (int k = (nflt & ~3) + (int)lane; k < nflt; k += 32) dst[k] = sm[k];
  }
}

// ---- frame stack (SB3 StackedObservations, 1-D observations stacked along the last axis) --
// stacked[i] = roll(stacked[i], -dim); if done[i]: stacked[i] = 0; stacked[i, -dim:] = obs[i]
// and, for envs that finished an episode (StackedObservations.update): the stacked terminal
// observation term_out[i] = concat(rolled previous stack minus its last frame, term_in[i]).
//
// One warp owns 32 consecutive rows = one contiguous run of 32 * dim * k floats.  It reads the run with
// whole float4 loads into shared memory (plus the 32 new observations and, if asked, the 32 terminal
// observations), and writes the updated run back with whole float4 stores: every global access is a
// full 128-byte line.  The previous version walked one private 96-byte row per thread (24 scalar
// loads and stores at a 96-byte lane stride).  In place is safe: a warp reads its whole run before it
// writes any of it, and runs of different warps are disjoint.
__global__ void __launch_bounds__(256) k_frame_stack_warp(float* __restrict__ stacked, const float* __restrict__ obs,
                                                          int64_t es, int64_t cs, const uint8_t* __restrict__ done,
                                                          const float* __restrict__ term_in, int64_t tes, int64_t tcs,
                                                          float* __restrict__ term_out, int64_t n, int dim, int k) {
  extern __shared__ __align__(16) float sm_fs[];   // per warp: [32 * rowlen] old rows | [32 * dim] obs | [32 * dim] term
  const unsigned lane = threadIdx.x & 31u;
  const int rowlen = dim * k, keep = rowlen - dim;
  const int per_warp = 32 * rowlen + 64 * dim;
  float* sm_old = sm_fs + (threadIdx.x >> 5) * per_warp;
  float* sm_obs = sm_old + 32 * rowlen;
  float* sm_term = sm_obs + 32 * dim;
  const int64_t row0 = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32;
  if (row0 >= n) return;
  const int rows = (int)(n - row0 >= 32 ? 32 : n - row0);
  const int nflt = rows * rowlen;
  float* run = stacked + row0 * rowlen;
  const bool vec = (((uintptr_t)run) & 15) == 0;
  if (vec) {
    for (int q = (int)lane * 4; q + 3 < nflt; q += 128)
      *reinterpret_cast<float4*>(sm_old + q) = *reinterpret_cast<const float4*>(run + q);
    for (int q = (nflt & ~3) + (int)lane; q < nflt; q += 32) sm_old[q] = run[q];
  } else {
    for (int q = (int)lane; q < nflt; q += 32) sm_old[q] = run[q];
  }
  const bool mine = (int)lane < rows;
  const bool d = mine && done != nullptr && done[row0 + lane] != 0;
  const unsigned any_done = __ballot_sync(0xffffffffu, d);
  if (mine) {
    for (int c = 0; c < dim; ++c) sm_obs[lane * dim + c] = obs[(row0 + lane) * es + c * cs];
    if (term_out != nullptr && any_done)
      for (int c = 0; c < dim; ++c) sm_term[lane * dim + c] = term_in[(row0 + lane) * tes + c * tcs];
  }
  __syncwarp();
  const unsigned done_mask = any_done;
  // (row, column) of a float of the run advance incrementally -- per 128 floats by (128 / rowlen,
  // 128 % rowlen) -- instead of two integer divisions per float (ncu on the first version: 1,443
  // instructions per warp, issue slots 70 % busy on a kernel that should only stream)
  auto val_at = [&](int q, int r, int j) -> float {
    if (j >= keep) return sm_obs[r * dim + (j - keep)];
    return ((done_mask >> r) & 1u) ? 0.0f : sm_old[q + dim];
  };
  const int dr = 128 / rowlen, dj = 128 % rowlen;
  if (vec) {
    int q = (int)lane * 4, r = q / rowlen, j = q - r * rowlen;
    for (; q + 3 < nflt; q += 128) {
      float v[4];
      int rr = r, jj = j;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        v[e] = val_at(q + e, rr, jj);
        if (++jj == rowlen) { jj = 0; ++rr; }
      }
      *reinterpret_cast<float4*>(run + q) = make_float4(v[0], v[1], v[2], v[3]);
      r += dr; j += dj;
      if (j >= rowlen) { j -= rowlen; ++r; }
    }
    for (int q2 = (nflt & ~3) + (int)lane; q2 < nflt; q2 += 32) { const int r2 = q2 / rowlen; run[q2] = val_at(q2, r2, q2 - r2 * rowlen); }
  } else {
    for (int q2 = (int)lane; q2 < nflt; q2 += 32) { const int r2 = q2 / rowlen; run[q2] = val_at(q2, r2, q2 - r2 * rowlen); }
  }
  if (term_out != nullptr && any_done) {
    // rows of envs that did not finish are not meaningful and never read (same convention as term_obs)
    float* trun = term_out + row0 * rowlen;
    for (int q = (int)lane; q < nflt; q += 32) {
      const int r = q / rowlen, j = q - r * rowlen;
      trun[q] = j >= keep ? sm_term[r * dim + (j - keep)] : sm_old[q + dim];
    }
  }
}

// fallback for very long rows (shared memory): one thread per row
__global__ void __launch_bounds__(256) k_frame_stack(float* __restrict__ stacked, const float* __restrict__ obs,
                                                     int64_t es, int64_t cs, const uint8_t* __restrict__ done,
                                                     const float* __restrict__ term_in, int64_t tes, int64_t tcs,
                                                     float* __restrict__ term_out, int64_t n, int dim, int k) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float* row = stacked + i * (int64_t)(dim * k);
  const bool d = done != nullptr && done[i] != 0;
  if (d && term_out != nullptr) {
    float* trow = term_out + i * (int64_t)(dim * k);
    for (int j = 0; j < dim * (k - 1); ++j) trow[j] = row[j + dim];
    for (int c = 0; c < dim; ++c) trow[dim * (k - 1) + c] = term_in[i * tes + c * tcs];
  }
  for (int j = 0; j < dim * (k - 1); ++j) row[j] = d ? 0.0f : row[j + dim];
  for (int c = 0; c < dim; ++c) row[dim * (k - 1) + c] = obs[i * es + c * cs];
}

// ---- evaluation metrics over stored trajectories err[T][3][stride], u[T][2][stride] (f64) ---
// out[i][4] = mae, rmse, settling_time (NaN = never settles), energy -- see the header.
// One thread per trajectory walking all T steps is latency-bound with a few thousand trajectories (ncu:
// 85 % long-scoreboard, 382 GB/s; 746 GB/s with four steps of loads in flight).  The time axis is
// therefore cut into segments (blockIdx.y): k_eval_partial accumulates per (trajectory, segment) and adds
// its sums / last-exceedance indices into a scratch row with atomics, k_eval_final turns the row into the
// four metrics.  Scratch row (f64): [0..3] sum|e_c|, [4..7] sum e_c^2, [8] energy, [9..12] last index with
// |e_c| > band as a double (-1 = never; max-merged as an integer, see atomic_max_index).
__device__ __forceinline__ void atomic_max_index(double* addr, int v) {
  // indices are >= 0 and stored as v + 1 in a 64-bit integer view of the slot (0 = never exceeded)
  atomicMax((unsigned long long*)addr, (unsigned long long)(v + 1));
}

__global__ void __launch_bounds__(128) k_eval_partial(const double* __restrict__ err, const double* __restrict__ u,
                                                      int T, int ncomp, int nctrl, int64_t n, int64_t stride,
                                                      int steady_start, double band, int seg_len,
                                                      double* __restrict__ scratch) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int t_lo = (int)blockIdx.y * seg_len, t_hi = min(T, t_lo + seg_len);
  double sa[4] = {0, 0, 0, 0}, sq[4] = {0, 0, 0, 0}, en = 0.0;
  int last_ex[4] = {-1, -1, -1, -1};
  constexpr int U = 4;
  auto step = [&](int t, const double* e, const double* a) {
    for (int c = 0; c < ncomp; ++c) {
      if (fabs(e[c]) > band) last_ex[c] = t;
      if (t >= steady_start) { sa[c] += fabs(e[c]); sq[c] += e[c] * e[c]; }
    }
    double q = 0.0;
    for (int c = 0; c < nctrl; ++c) q += a[c] * a[c];
    en += q;
  };
  int t = t_lo;
  for (; t + U <= t_hi; t += U) {
    double e[U][4], a[U][4];
#pragma unroll
    for (int k = 0; k < U; ++k) {
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        e[k][c] = c < ncomp ? err[((int64_t)(t + k) * ncomp + c) * stride + i] : 0.0;
        a[k][c] = c < nctrl ? u[((int64_t)(t + k) * nctrl + c) * stride + i] : 0.0;
      }
    }
#pragma unroll
    for (int k = 0; k < U; ++k) step(t + k, e[k], a[k]);
  }
  for (; t < t_hi; ++t) {
    double e[4], a[4];
    for (int c = 0; c < 4; ++c) {
      e[c] = c < ncomp ? err[((int64_t)t * ncomp + c) * stride + i] : 0.0;
      a[c] = c < nctrl ? u[((int64_t)t * nctrl + c) * stride + i] : 0.0;
    }
    step(t, e, a);
  }
  double* row = scratch + i * 13;
  for (int c = 0; c < ncomp; ++c) {
    if (sa[c] != 0.0) atomicAdd(&row[c], sa[c]);
    if (sq[c] != 0.0) atomicAdd(&row[4 + c], sq[c]);
    if (last_ex[c] >= 0) atomic_max_index(&row[9 + c], last_ex[c]);
  }
  if (en != 0.0) atomicAdd(&row[8], en);
}

__global__ void __launch_bounds__(128) k_eval_final(const double* __restrict__ scratch, int T, int ncomp, int64_t n,
                                                    int steady_start, double dt, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* row = scratch + i * 13;
  const double m = (double)(T - steady_start);
  double mae = 0.0, rmse = 0.0, ts = -1.0;
  bool never = false;
  for (int c = 0; c < ncomp; ++c) {
    mae += row[c] / m;
    rmse += sqrt(row[4 + c] / m);
    const int last_ex = (int)(*(const unsigned long long*)&row[9 + c]) - 1;
    if (last_ex + 1 >= T) never = true;                       // np.nan for that component
    const double tc = (last_ex < 0) ? 0.0 : (double)(last_ex + 1) * dt;
    if (last_ex + 1 < T && tc > ts) ts = tc;                   // np.nanmax ignores the NaNs
  }
  double* o = out + i * 4;
  o[0] = mae / ncomp;
  o[1] = rmse / ncomp;
  o[2] = (ts < 0.0 && never) ? nan("") : (ts < 0.0 ? 0.0 : ts);
  o[3] = row[8] * dt;
}

int fail_if(cudaError_t e) { return e == cudaSuccess ? CL_OK : CL_ECUDA; }

}  // namespace

extern "C" int cl_gae(void* stream, const float* rewards, const float* values, const float* episode_starts,
                      const float* last_values, const float* last_dones, double gamma, double gae_lambda,
                      int32_t T, int64_t n, int64_t stride, float* advantages, float* returns) {
  if (!rewards || !values || !episode_starts || !last_values || !last_dones || !advantages || !returns || T < 1 || n < 1)
    return CL_EINVAL;
  const int block = 128;
  k_gae<<<(unsigned)((n + block - 1) / block), block, 0, (cudaStream_t)stream>>>(
      rewards, values, episode_starts, last_values, last_dones, (float)gamma, (float)(gamma * gae_lambda), T, n,
      stride, advantages, returns);
  return fail_if(cudaGetLastError());
}

extern "C" int cl_obs_moments(void* stream, const float* obs, int64_t es, int64_t cs, int64_t n, int32_t dim,
                              const double* shift, double* out2d) {
  if (!obs || !shift || !out2d || dim < 1 || dim > 32 || n < 1) return CL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(out2d, 0, sizeof(double) * 2 * (size_t)dim, st);
  if (e != cudaSuccess) return CL_ECUDA;
  const int block = 256;
  int64_t blocks = (n + block - 1) / block;
  if (blocks > 148 * 4) blocks = 148 * 4;
  if (dim <= 8) k_moments<8, float><<<(unsigned)blocks, block, 0, st>>>(obs, es, cs, n, dim, shift, out2d);
  else k_moments<32, float><<<(unsigned)blocks, block, 0, st>>>(obs, es, cs, n, dim, shift, out2d);
  return fail_if(cudaGetLastError());
}

// float64 input (SB3 feeds VecNormalize's float64 discounted returns to ret_rms.update)
extern "C" int cl_moments_f64(void* stream, const double* x, int64_t es, int64_t cs, int64_t n, int32_t dim,
                              const double* shift, double* out2d) {
  if (!x || !shift || !out2d || dim < 1 || dim > 32 || n < 1) return CL_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(out2d, 0, sizeof(double) * 2 * (size_t)dim, st);
  if (e != cudaSuccess) return CL_ECUDA;
  const int block = 256;
  int64_t blocks = (n + block - 1) / block;
  if (blocks > 148 * 4) blocks = 148 * 4;
  if (dim <= 8) k_moments<8, double><<<(unsigned)blocks, block, 0, st>>>(x, es, cs, n, dim, shift, out2d);
  else k_moments<32, double><<<(unsigned)blocks, block, 0, st>>>(x, es, cs, n, dim, shift, out2d);
  return fail_if(cudaGetLastError());
}

// Chan et al. parallel update of (mean, var, count) with one batch's shifted sums (rms_merge.cuh),
// entirely on the device: the running count is a device scalar, so a VecNormalize step neither
// synchronises nor bakes host state into a captured CUDA graph.
//   acc[0][c] = sum(x - mean_old), acc[1][c] = sum((x - mean_old)^2)   (cl_obs_moments)
__global__ void k_rms_merge(const double* __restrict__ acc, double n, int dim, double* mean, double* var,
                            double* count) {
  const int c = threadIdx.x;
  const double cnt = *count, tot = cnt + n;
  if (c < dim) rms_merge(mean[c], var[c], cnt, n, acc[c], acc[dim + c]);
  __syncthreads();  // every thread has read *count
  if (c == 0) *count = tot;
}

extern "C" int cl_rms_update(void* stream, const double* acc2d, int64_t n, int32_t dim, double* mean, double* var,
                             double* count) {
  if (!acc2d || !mean || !var || !count || dim < 1 || dim > 32 || n < 1) return CL_EINVAL;
  k_rms_merge<<<1, 32, 0, (cudaStream_t)stream>>>(acc2d, (double)n, dim, mean, var, count);
  return fail_if(cudaGetLastError());
}

extern "C" int cl_obs_normalize(void* stream, const float* in, int64_t ies, int64_t ics, float* out, int64_t oes,
                                int64_t ocs, int64_t n, int32_t dim, const double* mean, const double* var,
                                double epsilon, double clip) {
  if (!in || !out || !mean || !var || dim < 1 || n < 1) return CL_EINVAL;
  const int block = 256;
  const unsigned grid = (unsigned)((n + block - 1) / block);
  // The ROWS transpose needs 32 * dim floats of dynamic shared memory per warp.  Without an opt-in a block
  // gets 48 KiB in all, and k_normalize<true>'s static sm_mean / sm_std take part of that: the dynamic
  // allowance is what remains (maxDynamicSharedSizeBytes; dim 47 fits, dim 48 takes the strided kernel).
  // Only a successful query is kept; after a failed one this call takes the strided kernel, which needs no
  // shared memory, and the next call asks again.
  static std::atomic<int64_t> rows_smem_max{-1};
  int64_t smem_max = rows_smem_max.load(std::memory_order_relaxed);
  if (smem_max < 0) {
    cudaFuncAttributes a{};
    if (cudaFuncGetAttributes(&a, k_normalize<true>) == cudaSuccess) {
      smem_max = (int64_t)a.maxDynamicSharedSizeBytes;
      rows_smem_max.store(smem_max, std::memory_order_relaxed);
    } else {
      (void)cudaGetLastError();   // a sticky error fails the launch below and is reported there
    }
  }
  const int64_t rows_smem = (int64_t)(block / 32) * 32 * dim * (int64_t)sizeof(float);
  const bool rows = oes == dim && ocs == 1 && (((uintptr_t)out) & 15) == 0 && rows_smem <= smem_max;
  if (rows)
    k_normalize<true><<<grid, block, (size_t)rows_smem, (cudaStream_t)stream>>>(in, ies, ics, out, oes, ocs, n, dim,
                                                                                mean, var, epsilon, clip);
  else
    k_normalize<false><<<grid, block, 0, (cudaStream_t)stream>>>(in, ies, ics, out, oes, ocs, n, dim, mean, var,
                                                                  epsilon, clip);
  return fail_if(cudaGetLastError());
}

static int frame_stack_launch(cudaStream_t st, float* stacked, const float* obs, int64_t es, int64_t cs,
                              const uint8_t* done, const float* term_in, int64_t tes, int64_t tcs, float* term_out,
                              int64_t n, int32_t dim, int32_t n_stack) {
  const int block = 256, wpb = block / 32;
  const size_t smem = (size_t)wpb * (32 * (size_t)dim * n_stack + 64 * (size_t)dim) * sizeof(float);
  if (smem <= 48 * 1024) {
    const int64_t warps = (n + 31) / 32;
    k_frame_stack_warp<<<(unsigned)((warps + wpb - 1) / wpb), block, smem, st>>>(stacked, obs, es, cs, done, term_in, tes,
                                                                                 tcs, term_out, n, dim, n_stack);
  } else {
    k_frame_stack<<<(unsigned)((n + block - 1) / block), block, 0, st>>>(stacked, obs, es, cs, done, term_in, tes, tcs,
                                                                          term_out, n, dim, n_stack);
  }
  return fail_if(cudaGetLastError());
}

extern "C" int cl_frame_stack(void* stream, float* stacked, const float* obs, int64_t es, int64_t cs,
                              const uint8_t* done, int64_t n, int32_t dim, int32_t n_stack) {
  if (!stacked || !obs || dim < 1 || n_stack < 1 || n < 1) return CL_EINVAL;
  return frame_stack_launch((cudaStream_t)stream, stacked, obs, es, cs, done, nullptr, 0, 0, nullptr, n, dim, n_stack);
}

extern "C" int cl_frame_stack_term(void* stream, float* stacked, const float* obs, int64_t es, int64_t cs,
                                   const uint8_t* done, const float* term_obs, int64_t tes, int64_t tcs,
                                   float* term_stacked, int64_t n, int32_t dim, int32_t n_stack) {
  if (!stacked || !obs || !done || !term_obs || !term_stacked || dim < 1 || n_stack < 1 || n < 1) return CL_EINVAL;
  return frame_stack_launch((cudaStream_t)stream, stacked, obs, es, cs, done, term_obs, tes, tcs, term_stacked, n, dim,
                            n_stack);
}

extern "C" int cl_eval_metrics(void* stream, const double* err, const double* ctrl, int32_t T, int32_t n_err,
                               int32_t n_ctrl, int64_t n, int64_t stride, int32_t steady_start, double dt,
                               double error_band, double* out4) {
  if (!err || !ctrl || !out4 || T < 1 || n_err < 1 || n_err > 4 || n_ctrl < 0 || n_ctrl > 4 || n < 1 || steady_start < 0 ||
      steady_start >= T)
    return CL_EINVAL;
  const int block = 128;
  cudaStream_t st = (cudaStream_t)stream;
  // enough (trajectory, segment) threads to cover the memory latency: ~512 K, segments of at least 64 steps
  int64_t segs = (512 * 1024 + n - 1) / n;
  if (segs > (T + 63) / 64) segs = (T + 63) / 64;
  if (segs < 1) segs = 1;
  const int seg_len = (int)((T + segs - 1) / segs);
  segs = (T + seg_len - 1) / seg_len;
  double* scratch = nullptr;
  if (cudaMallocAsync((void**)&scratch, sizeof(double) * 13 * (size_t)n, st) != cudaSuccess) return CL_ENOMEM;
  if (cudaMemsetAsync(scratch, 0, sizeof(double) * 13 * (size_t)n, st) != cudaSuccess) return CL_ECUDA;
  const dim3 grid((unsigned)((n + block - 1) / block), (unsigned)segs);
  k_eval_partial<<<grid, block, 0, st>>>(err, ctrl, T, n_err, n_ctrl, n, stride, steady_start, error_band, seg_len, scratch);
  k_eval_final<<<grid.x, block, 0, st>>>(scratch, T, n_err, n, steady_start, dt, out4);
  cudaFreeAsync(scratch, st);
  return fail_if(cudaGetLastError());
}
