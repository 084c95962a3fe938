// C-ABI implementation (include/chaos_b200.h): context, argument validation, kernel
// dispatch, pinned host staging for the SB3 numpy contract, measurement utilities.
#include <math.h>
#include <pthread.h>
#include <sched.h>
#include <stdarg.h>
#include <time.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "kernels_common.cuh"
#include "host_copy.h"

cudaError_t cl_launch_derivatives(int kind, const void* state, const float* action, void* out,
                                  int64_t n, cudaStream_t st);

using cl::KParams;

struct CopyHelper;

namespace {

const cl_layout kLayouts[CL_ENV_KIND_COUNT] = {
    // real_bytes n_state n_int obs act noise  act_lo act_hi  obs_lo obs_hi  max_steps
    /* LORENZ3       */ {8, 4, 0, 6, 3, 0, -500.0, 500.0, -HUGE_VAL, HUGE_VAL, 0, 0},
    /* LORENZ3_PAIR  */ {8, 10, 0, 6, 3, 0, -500.0, 500.0, -HUGE_VAL, HUGE_VAL, 0, 0},
    /* LORENZ4_PAIR  */ {8, 9, 0, 8, 3, 0, -2.0, 2.0, -HUGE_VAL, HUGE_VAL, 0, 0},
    /* HR_SYNC       */ {8, 9, 0, 6, 2, 3, -1.0, 1.0, -1.0, 1.0, 5000, 0},
    /* PMSM_SYNC     */ {4, 9, 1, 6, 2, 3, -1.0, 1.0, -HUGE_VAL, HUGE_VAL, 2000, 0},
    /* PMSM_CLASSIC  */ {8, 7, 0, 6, 2, 3, -2.0, 2.0, -HUGE_VAL, HUGE_VAL, 0, 0},
    /* PMSM_SINGLE   */ {8, 4, 0, 6, 2, 0, -10.0, 10.0, -HUGE_VAL, HUGE_VAL, 0, 0},
    /* LORENZ_RK4    */ {8, 6, 0, 6, 3, 0, -1.0, 1.0, -HUGE_VAL, HUGE_VAL, 1000, 0},
    /* LORENZ_RK4_F32*/ {4, 6, 0, 6, 3, 0, -1.0, 1.0, -HUGE_VAL, HUGE_VAL, 1000, 0},
    /* PMSM_RK4      */ {8, 8, 0, 6, 2, 0, -1.0, 1.0, -HUGE_VAL, HUGE_VAL, 2000, 0},
    /* MEMRISTIVE4   */ {8, 9, 0, 8, 3, 0, -2.0, 2.0, -HUGE_VAL, HUGE_VAL, 0, 0},
    /* PMSM_FREE     */ {8, 4, 0, 6, 2, 3, -100.0, 100.0, -HUGE_VAL, HUGE_VAL, 0, 0},
};

const int CL_DYN_CHUNK_DEFAULT = 8;
const int kHostRing = 3;  // pinned output slots: obs returned at step t stays valid through t+2

struct HostSlot {
  unsigned char* out;  // pinned, same layout as HostStage::d_out
  float* obs;
  float* reward;
  uint8_t* done;
  float* term_obs;
  double* last_ep_ret;
  int32_t* last_ep_len;
  uint8_t* warp_done;  // pinned [ceil(N/32)] (+ padding to 8): 1 where an env-warp ended an episode in this step
};

struct HostStage {
  bool ready;
  float* h_act;   // pinned [N][A]
  float* d_act;   // device [N][A]
  unsigned char* d_out;  // device, one block: [obs N*O f32 | reward N f32 | done N u8] -> ONE D2H copy
  float* d_obs;   // = d_out
  float* d_rew;   // = d_out + N*O*4
  uint8_t* d_done;
  size_t out_bytes;
  float* d_term;  // device [N][O]
  double* d_ler;
  int32_t* d_lel;
  HostSlot slot[kHostRing];
  int cur;        // slot being filled / last filled
  cudaStream_t stream;
  bool pending;
  // CL_HOST_DMA: H2D copy -> kernel -> one D2H copy.  CL_HOST_ZEROCOPY: the kernel reads the
  // actions from and writes the results to pinned host memory.  CL_HOST_PIPELINED: the env batch
  // is cut into slices that alternate over two streams; each slice's actions arrive by DMA
  // (SM-initiated PCIe reads top out near 20 GB/s) and its kernel writes the results straight to
  // pinned host memory, so slice j's upstream writes overlap slice j+1's downstream copy.
  int mode;
  bool extras_on_host;  // the pending step wrote term_obs / last_ep_* to the host slot itself
  int slices;        // CL_HOST_PIPELINED / CL_HOST_STREAMED: number of env slices (>= 1)
  cudaStream_t side; // second stream of the pipeline
  cudaEvent_t ev_fork, ev_join;
  // CL_HOST_STREAMED: the step kernel is launched first and waits, block by block, for the slice of
  // the pinned action buffer it reads to be published (generation number) by the staging loop
  uint32_t* h_ready;   // pinned progress words, one per staging lane (CL_STAGE_WORD_STRIDE apart): (generation << 8) | slices of the lane staged so far
  uint32_t* d_ready;   // their device mirrors (adjacent words), kept up to date by k_relay
  uint32_t* h_err;     // pinned: set by a block whose bounded wait expired
  uint32_t gen;
  uint8_t* d_warp_done;  // device copy for CL_HOST_DMA (travels with the result block)
  size_t wd_bytes;
  struct CopyHelper* helper;   // helper threads of the staging lanes (nullptr: single-threaded staging)
  int relay_kernel;            // 1: k_relay on the side stream (a second launch per step; CHAOS_B200_RELAY=kernel), 0: block 0 of the step kernel
  cl_buffers redo_buf;         // buffers of the step in flight
  int64_t streamed_fallbacks;  // streamed steps called off by k_relay and redone as zero-copy steps
};

}  // namespace

struct cl_ctx {
  cl_config cfg;
  cl_layout lay;
  char err[512];
  uint64_t step_index;
  int64_t launches;
  int block;
  int sm_count;
  float* d_bc1;
  float* d_bc2;
  int bc1_n, bc2_n;
  HostStage hs;
  uint32_t* d_dyn;      // [1 + n_envwarps]: task counter + per-env-warp progress (k_rollout_dyn)
  uint64_t* d_step;     // graph mode: device-resident Philox step index (+ ticket word behind it)
  int graph_mode;
  int dyn_bps;          // resident worker blocks per SM (0 = not yet queried)
  int no_plain;         // never pick the plain-rollout kernel instantiation
  int64_t dyn_launches;
  int64_t plain_launches;  // rollouts that ran on the plain-I/O kernel instantiation
  int64_t sm_launches;     // rollouts that ran on the SM-local kernel (k_rollout_sm)
};

static char g_err[512] = "";

static int fail(cl_ctx* ctx, int code, const char* fmt, ...) {
  char* dst = ctx ? ctx->err : g_err;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(ctx, CL_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                  __FILE__, __LINE__);                                                    \
  } while (0)

static bool is_parity(int kind) { return !(kind >= CL_ENV_LORENZ_RK4 && kind <= CL_ENV_PMSM_RK4); }

// Threads on the most loaded SM decide the duration of a single partial wave; pick the block
// size that minimises ceil(blocks / SMs) * block (ties -> larger block).  65,536 envs on 148
// SMs: 64-thread blocks give 7 x 64 = 448 threads on the fullest SM vs 512 for 128 / 256.
static int pick_block(int64_t n, int sms) {
  // ties -> the smaller block: at 1 Mi envs 64 / 128 / 256 are within 1 % of each other in balance and
  // 64-thread blocks measured 1-5 % faster on every HBM-bound kind (profiles/r02_sweep_block_stats.jsonl)
  const int cand[3] = {64, 128, 256};
  int best = 64;
  int64_t best_cost = -1;
  for (int k = 0; k < 3; ++k) {
    const int64_t blocks = (n + cand[k] - 1) / cand[k];
    const int64_t cost = ((blocks + sms - 1) / sms) * cand[k];
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = cand[k]; }
  }
  return best;
}

extern "C" int cl_abi_version(void) { return CL_ABI_VERSION; }

extern "C" int cl_env_layout(int32_t kind, cl_layout* out) {
  if (!out || kind < 0 || kind >= CL_ENV_KIND_COUNT) return fail(nullptr, CL_EINVAL, "bad kind %d", kind);
  *out = kLayouts[kind];
  return CL_OK;
}

extern "C" const char* cl_last_error(const cl_ctx* ctx) { return ctx ? ctx->err : g_err; }

extern "C" int cl_create(const cl_config* cfg, cl_ctx** out) {
  cl_ctx* ctx = nullptr;
  if (!cfg || !out) return fail(nullptr, CL_EINVAL, "null argument");
  if (cfg->abi_version != CL_ABI_VERSION) return fail(nullptr, CL_EINVAL, "abi mismatch: caller %d library %d", cfg->abi_version, CL_ABI_VERSION);
  if (cfg->kind < 0 || cfg->kind >= CL_ENV_KIND_COUNT) return fail(nullptr, CL_EINVAL, "bad kind %d", cfg->kind);
  if (cfg->num_envs <= 0) return fail(nullptr, CL_EINVAL, "num_envs must be > 0");
  if (cfg->n_pad < cfg->num_envs || (cfg->n_pad % 128) != 0) return fail(nullptr, CL_EINVAL, "n_pad must be a multiple of 128 and >= num_envs");
  if (!is_parity(cfg->kind)) {
    if (cfg->substeps < 1 || cfg->substeps > 4096) return fail(nullptr, CL_EINVAL, "substeps out of range");
    if (!(cfg->dt > 0.0)) return fail(nullptr, CL_EINVAL, "dt must be > 0");
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(nullptr, CL_ENODEV, "no CUDA device: %s", cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, CL_ENODEV, "device %d out of range (%d devices)", cfg->device, ndev);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, cfg->device);
  if (e != cudaSuccess) return fail(nullptr, CL_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10) return fail(nullptr, CL_ENODEV, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);

  ctx = (cl_ctx*)calloc(1, sizeof(cl_ctx));
  if (!ctx) return fail(nullptr, CL_ENOMEM, "out of host memory");
  ctx->cfg = *cfg;
  ctx->lay = kLayouts[cfg->kind];
  ctx->sm_count = prop.multiProcessorCount;
  ctx->block = pick_block(cfg->num_envs, ctx->sm_count);
  if (const char* ov = getenv("CHAOS_B200_BLOCK")) {  // tuning override: 32..256, multiple of 32
    const int b = atoi(ov);
    if (b >= 32 && b <= 256 && (b % 32) == 0) ctx->block = b;
  }
  // testing / A-B override: CHAOS_B200_PLAIN=0 keeps rollouts on the generic kernel instantiation
  ctx->no_plain = (getenv("CHAOS_B200_PLAIN") != nullptr && getenv("CHAOS_B200_PLAIN")[0] == '0') ? 1 : 0;
  ctx->step_index = 0;
  e = cudaSetDevice(cfg->device);
  if (e != cudaSuccess) { int r = fail(nullptr, CL_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(e)); free(ctx); return r; }

  if (cfg->kind == CL_ENV_PMSM_SYNC) {
    // (float)(1 - beta**n): CPython float pow -> libm pow, then the weak-scalar rounding to
    // float32 that NumPy applies in `self.m_t / (1 - self.beta1 ** self.adam_step)`
    // (lorenz_env_try_pmsm.py:130-131).  The tables end where the value reaches 1.0f.
    const double betas[2] = {0.9, 0.999};
    float** dst[2] = {&ctx->d_bc1, &ctx->d_bc2};
    int* cnt[2] = {&ctx->bc1_n, &ctx->bc2_n};
    for (int k = 0; k < 2; ++k) {
      int n = 1;
      while ((float)(1.0 - pow(betas[k], (double)n)) != 1.0f && n < (1 << 20)) ++n;
      float* h = (float*)malloc(sizeof(float) * (size_t)n);
      if (!h) { free(ctx); return fail(nullptr, CL_ENOMEM, "out of host memory"); }
      for (int j = 0; j < n; ++j) h[j] = (float)(1.0 - pow(betas[k], (double)j));
      e = cudaMalloc((void**)dst[k], sizeof(float) * (size_t)n);
      if (e == cudaSuccess) e = cudaMemcpy(*dst[k], h, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice);
      free(h);
      if (e != cudaSuccess) { int r = fail(nullptr, CL_ECUDA, "bias table upload: %s", cudaGetErrorString(e)); free(ctx); return r; }
      *cnt[k] = n;
    }
  }
  {  // scratch that must exist before any CUDA-graph capture: dyn queue + device step counter
    const int64_t W = (cfg->num_envs + 31) / 32;
    e = cudaMalloc((void**)&ctx->d_dyn, sizeof(uint32_t) * (size_t)(W + 1));
    if (e == cudaSuccess) e = cudaMalloc((void**)&ctx->d_step, 2 * sizeof(uint64_t));
    if (e == cudaSuccess) e = cudaMemset(ctx->d_step, 0, 2 * sizeof(uint64_t));
    if (e != cudaSuccess) { int r = fail(nullptr, CL_ECUDA, "scratch allocation: %s", cudaGetErrorString(e)); free(ctx); return r; }
  }
  *out = ctx;
  return CL_OK;
}

static void copy_helper_stop(CopyHelper* c);

static void host_stage_free(cl_ctx* ctx) {
  HostStage& h = ctx->hs;
  if (!h.ready) return;
  copy_helper_stop(h.helper);
  h.helper = nullptr;
  cudaFreeHost(h.h_act);
  cudaFree(h.d_act); cudaFree(h.d_out);
  cudaFree(h.d_term); cudaFree(h.d_ler); cudaFree(h.d_lel);
  cudaFreeHost(h.h_ready);
  cudaFree(h.d_ready);
  for (int k = 0; k < kHostRing; ++k) {
    cudaFreeHost(h.slot[k].out);
    cudaFreeHost(h.slot[k].term_obs); cudaFreeHost(h.slot[k].last_ep_ret); cudaFreeHost(h.slot[k].last_ep_len);
  }
  cudaStreamDestroy(h.stream);
  cudaStreamDestroy(h.side);
  cudaEventDestroy(h.ev_fork);
  cudaEventDestroy(h.ev_join);
  h.ready = false;
}

extern "C" int cl_destroy(cl_ctx* ctx) {
  if (!ctx) return CL_OK;
  cudaSetDevice(ctx->cfg.device);
  host_stage_free(ctx);
  if (ctx->d_bc1) cudaFree(ctx->d_bc1);
  if (ctx->d_bc2) cudaFree(ctx->d_bc2);
  if (ctx->d_dyn) cudaFree(ctx->d_dyn);
  if (ctx->d_step) cudaFree(ctx->d_step);
  free(ctx);
  return CL_OK;
}

static int fill_params(cl_ctx* ctx, const cl_buffers* buf, const cl_io* io, KParams& p) {
  if (!buf || !buf->state || !buf->ep_len || !buf->ep_return || !buf->stats)
    return fail(ctx, CL_EINVAL, "cl_buffers: state/ep_len/ep_return/stats must be non-null");
  if (ctx->lay.n_int > 0 && !buf->aux_int) return fail(ctx, CL_EINVAL, "cl_buffers.aux_int required for this kind");
  memset(&p, 0, sizeof(p));
  const cl_config& c = ctx->cfg;
  p.n = c.num_envs; p.n_pad = c.n_pad; p.env_id_base = c.env_id_base;
  p.k0 = (uint32_t)c.seed; p.k1 = (uint32_t)(c.seed >> 32);
  p.step_index = ctx->step_index;
  p.no_plain = ctx->no_plain;
  if (ctx->graph_mode) p.step_ptr = ctx->d_step;
  p.max_steps = c.max_episode_steps; p.substeps = c.substeps; p.flags = c.flags;
  p.dt = c.dt; p.alpha = c.alpha; p.act_limit = c.act_limit; p.act_gain = c.act_gain;
  p.param_jitter = c.param_jitter;
  p.state = buf->state; p.aux_int = buf->aux_int; p.ep_len = buf->ep_len;
  p.ep_return = buf->ep_return; p.stats = buf->stats;
  p.bc1 = ctx->d_bc1; p.bc2 = ctx->d_bc2; p.bc1_n = ctx->bc1_n; p.bc2_n = ctx->bc2_n;
  if (!is_parity(c.kind)) {
    // same IEEE operations the kernel used to do per thread, done once here
    p.h = c.dt / (double)c.substeps; p.hh = 0.5 * p.h; p.h3 = p.h / 3.0; p.h6 = p.h / 6.0;
    p.hf = (float)p.h; p.hhf = 0.5f * p.hf; p.h3f = p.hf / 3.0f; p.h6f = p.hf / 6.0f;
    if (c.kind == CL_ENV_PMSM_RK4) { p.nom[0] = 5.46; p.nom[1] = 20.0; p.nom[2] = 0.0; }
    else { p.nom[0] = 10.0; p.nom[1] = 28.0; p.nom[2] = 8.0 / 3.0; }
    for (int k = 0; k < 3; ++k) p.nomf[k] = (float)p.nom[k];
    p.nom_br = p.nom[2] * p.nom[1];          // beta * rho, one rounding (see lorenz_rk4)
    p.nom_brf = p.nomf[2] * p.nomf[1];
    p.act_limit_f = (float)c.act_limit; p.act_gain_f = (float)c.act_gain;
  }
  if (io) {
    p.action = io->action; p.act_es = io->act_es; p.act_cs = io->act_cs;
    p.noise = io->noise;
    p.obs = io->obs; p.obs_es = io->obs_es; p.obs_cs = io->obs_cs;
    p.reward = io->reward; p.done = io->done; p.term_obs = io->term_obs;
    p.last_ep_ret = io->last_ep_ret; p.last_ep_len = io->last_ep_len; p.mask = io->mask;
  }
  return CL_OK;
}

__global__ void k_advance_step(uint64_t* step, uint64_t count) { *step += count; }

// Streamed host mode: the relay (cl::relay_lanes, kernels_common.cuh) as a kernel of its own on the side stream
// (CHAOS_B200_RELAY=kernel); by default it runs as block 0 of the step kernel.
__global__ void k_relay(const uint32_t* host_words, uint32_t* dev_words, uint32_t gen, uint32_t lanes, uint32_t spl,
                        uint32_t nslices, uint32_t* host_err) {
  cl::relay_lanes(host_words, dev_words, gen, lanes, spl, nslices, host_err);
}

// graph mode: the device-resident Philox step index (CUDA graphs) advances after each env kernel
static int advance_graph_step(cl_ctx* ctx, cudaStream_t st, uint64_t count) {
  if (!ctx->graph_mode) return CL_OK;
  k_advance_step<<<1, 1, 0, st>>>(ctx->d_step, count);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(ctx, CL_ECUDA, "step-index advance failed: %s", cudaGetErrorString(e));
  return CL_OK;
}

static int launch(cl_ctx* ctx, const KParams& p_in, int mode, cudaStream_t st) {
  KParams p = p_in;
  int32_t plain = 0;
  p.host_plain_out = &plain;
  cudaError_t e = is_parity(ctx->cfg.kind) ? cl_launch_parity(ctx->cfg.kind, p, mode, st, ctx->block)
                                           : cl_launch_northstar(ctx->cfg.kind, p, mode, st, ctx->block);
  if (e != cudaSuccess) return fail(ctx, CL_ECUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  ctx->launches += 1;
  ctx->plain_launches += (plain & 1);
  ctx->sm_launches += (plain >> 1) & 1;
  if (mode == cl::MODE_INIT) return CL_OK;
  return advance_graph_step(ctx, st, (mode == cl::MODE_ROLLOUT || mode == cl::MODE_ROLLOUT_DYN) ? (uint64_t)p.T : 1);
}

extern "C" int cl_init_persistent(cl_ctx* ctx, void* stream, const cl_buffers* buf) {
  if (!ctx) return fail(nullptr, CL_EINVAL, "null ctx");
  KParams p;
  int r = fill_params(ctx, buf, nullptr, p);
  if (r) return r;
  CU(cudaSetDevice(ctx->cfg.device));
  CU(cudaMemsetAsync(buf->stats, 0, sizeof(double) * CL_NSTATS, (cudaStream_t)stream));
  return launch(ctx, p, cl::MODE_INIT, (cudaStream_t)stream);
}

extern "C" int cl_reset(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io) {
  if (!ctx) return fail(nullptr, CL_EINVAL, "null ctx");
  KParams p;
  int r = fill_params(ctx, buf, io, p);
  if (r) return r;
  CU(cudaSetDevice(ctx->cfg.device));
  r = launch(ctx, p, cl::MODE_RESET, (cudaStream_t)stream);
  if (r == CL_OK) ctx->step_index += 1;
  return r;
}

extern "C" int cl_step(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io) {
  if (!ctx) return fail(nullptr, CL_EINVAL, "null ctx");
  if (!io || !io->action) return fail(ctx, CL_EINVAL, "cl_step: io.action is required");
  KParams p;
  int r = fill_params(ctx, buf, io, p);
  if (r) return r;
  p.reward_f32 = 0;
  CU(cudaSetDevice(ctx->cfg.device));
  r = launch(ctx, p, cl::MODE_STEP, (cudaStream_t)stream);
  if (r == CL_OK) ctx->step_index += 1;
  return r;
}

// Tensor map of a rollout's action tensor, f32 [T][A][row stride] with env stride 1: dims (x = envs,
// y = channels, z = intervals), box (32, A, chunk) = what one env-warp consumes in one chunk, fetched by
// k_rollout_sm with one cp.async.bulk.tensor per chunk.  The encoder is a driver entry point, looked up
// through the runtime (no link-time dependency on libcuda).  false -> the kernel copies row by row.
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static bool action_tensor_map(CUtensorMap* out, const float* base, uint64_t n_x, uint64_t n_ch, uint64_t T,
                              uint64_t row_stride, uint64_t t_stride, uint32_t chunk) {
  static encode_tiled_fn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (encode_tiled_fn)f;
  }
  if (!fn || chunk < 1 || chunk > 256 || n_ch > 256 || T < chunk) return false;
  const cuuint64_t dims[3] = {n_x, n_ch, T};
  const cuuint64_t strides[2] = {row_stride * sizeof(float), t_stride * sizeof(float)};   // of dims 1, 2 (bytes)
  const cuuint32_t box[3] = {32, (cuuint32_t)n_ch, chunk};
  const cuuint32_t estr[3] = {1, 1, 1};
  return fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Dynamic (env-warp x interval-chunk) scheduling pays off when the env-warps do not divide
// evenly over the 4 x SMs warp schedulers; CHAOS_B200_DYN=0/1 forces it off/on.
static bool want_dynamic(const cl_ctx* ctx, int T, int chunk) {
  const char* ov = getenv("CHAOS_B200_DYN");
  if (ov && ov[0] == '0') return false;
  const int64_t W = (ctx->cfg.num_envs + 31) / 32, nsched = (int64_t)ctx->sm_count * 4;
  if (T < 2 * chunk) return false;
  if (ov && ov[0] == '1') return true;
  if (W <= nsched) return false;
  if (W * (int64_t)((T + chunk - 1) / chunk) >= (int64_t)1 << 31) return false;  // task ids are 32-bit
  const double eff = (double)W / (double)(((W + nsched - 1) / nsched) * nsched);
  return eff < 0.95;
}

extern "C" int cl_rollout(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
                          const cl_rollout_desc* d) {
  if (!ctx) return fail(nullptr, CL_EINVAL, "null ctx");
  if (!io || !d || d->T < 1) return fail(ctx, CL_EINVAL, "cl_rollout: io/desc required, T >= 1");
  if (io->noise) return fail(ctx, CL_EINVAL, "cl_rollout: noise override is single-step only");
  KParams p;
  int r = fill_params(ctx, buf, io, p);
  if (r) return r;
  p.T = d->T; p.act_ts = d->act_ts; p.obs_ts = d->obs_ts; p.rew_ts = d->rew_ts; p.done_ts = d->done_ts;
  p.synth_amp = (float)d->synth_amp;
  cudaStream_t st = (cudaStream_t)stream;
  CU(cudaSetDevice(ctx->cfg.device));
  int chunk = CL_DYN_CHUNK_DEFAULT;
  if (const char* ov = getenv("CHAOS_B200_DYN_CHUNK")) { const int c = atoi(ov); if (c >= 1 && c <= 16) chunk = c; }
  int mode = cl::MODE_ROLLOUT;
  alignas(64) CUtensorMap tmap;      // lives until launch() below has copied it into the kernel's parameters
  if (want_dynamic(ctx, d->T, chunk)) {
    const int64_t W = (ctx->cfg.num_envs + 31) / 32;
    if (!ctx->dyn_bps) {
      int occ = 0;
      cudaError_t e = is_parity(ctx->cfg.kind) ? cl_dyn_occupancy_parity(ctx->cfg.kind, chunk, &occ)
                                               : cl_dyn_occupancy_northstar(ctx->cfg.kind, chunk, &occ);
      if (e != cudaSuccess) return fail(ctx, CL_ECUDA, "dyn occupancy query: %s", cudaGetErrorString(e));
      // keep the worker count below the env-warp count (see k_rollout_dyn: no dependency waits)
      int bps = (int)(W / ((int64_t)ctx->sm_count * 4));
      bps = bps < 1 ? 1 : (bps > 4 ? 4 : bps);
      if (const char* ov = getenv("CHAOS_B200_DYN_BPS")) { const int b = atoi(ov); if (b >= 1 && b <= 16) bps = b; }
      ctx->dyn_bps = occ < bps ? occ : bps;
    }
    if (ctx->dyn_bps >= 1) {
      CU(cudaMemsetAsync(ctx->d_dyn, 0, sizeof(uint32_t) * (size_t)(W + 1), st));
      p.dyn_counter = ctx->d_dyn;
      p.dyn_progress = ctx->d_dyn + 1;
      p.dyn_chunk = chunk;
      p.dyn_nchunks = (d->T + chunk - 1) / chunk;
      p.dyn_nwarps = (int32_t)W;
      // every SM gets its full set of resident worker blocks: only W tasks can run at any time
      // (one per env-warp), the surplus workers wait -- what matters is that each of the 592
      // warp schedulers always has at least one or two runnable workers
      const int64_t workers = (int64_t)ctx->sm_count * ctx->dyn_bps;
      const int64_t tasks = W * (int64_t)((d->T + chunk - 1) / chunk);
      p.dyn_grid = (int32_t)(workers * 4 < tasks ? workers : (tasks + 3) / 4);
      // bulk-copy staging needs unit env stride, 16 B alignment and whole 128 B rows in bounds
      p.dyn_tma = (io->action != nullptr && io->act_es == 1 && (io->act_cs % 4) == 0 && (d->act_ts % 4) == 0 &&
                   ((uintptr_t)io->action % 16) == 0 && io->act_cs >= W * 32) ? 1 : 0;
      // SM-local variant (k_rollout_sm, plain rollout shape only -- launch_env decides): one block per
      // SM owning W / SMs env-warps.  Workers = resident env-warps per block: a multiple of 4 (one per
      // scheduler and round) not above the smallest per-SM env-warp count, at most 16; the rest are guests.
      // CHAOS_B200_SM=0 keeps the global queue; CHAOS_B200_SM_WORKERS / _SM_CHUNK override (tuning).
      {
        const char* ov = getenv("CHAOS_B200_SM");
        if (!(ov && ov[0] == '0') && p.dyn_tma) {
          const int grid = (int)(W < ctx->sm_count ? W : ctx->sm_count);
          const int qn = (int)(W / grid), cmax = (int)((W + grid - 1) / grid);
          int workers = qn >= 4 ? 4 * (qn / 4) : qn;
          workers = workers > 16 ? 16 : workers;
          if (workers == 16 && qn < 20) workers = 12;   // 16..19 env-warps: 12 residents + 4..7 guests balance better than 16 + 0..3
          if (const char* w = getenv("CHAOS_B200_SM_WORKERS")) { const int k = atoi(w); if (k >= 1 && k <= 16) workers = k < qn ? k : qn; }
          // control intervals per chunk: 16 if the action double buffers of the block's env-warps fit
          // (each env-warp: 2 x chunk x ACT x 128 B), else 8, 4, ... (+0.8 % from 8 to 16, -2 % from 8 to 4)
          int sc = 16;
          const size_t per_warp = (size_t)ctx->lay.n_state * 32u * (size_t)ctx->lay.real_bytes + 32u * 12u + 28u;   // SmLayout
          while (sc > 1 && (size_t)cmax * (2u * (size_t)sc * (size_t)ctx->lay.act_dim * 128u + per_warp) + 256u > 200u * 1024u) sc /= 2;
          if (const char* w = getenv("CHAOS_B200_SM_CHUNK")) { const int k = atoi(w); if (k >= 1 && k <= 16) sc = k; }
          if (sc > d->T) sc = d->T;
          if (cmax <= 64) {
            p.sm_grid = grid; p.sm_workers = workers; p.sm_chunk = sc;
            p.sm_gdiv = 1;
            if (const char* w = getenv("CHAOS_B200_SM_GDIV")) { const int k = atoi(w); if (k >= 1 && k <= 16) p.sm_gdiv = k; }
            p.host_tmap = &tmap;
            p.sm_tmap_ok = action_tensor_map(&tmap, io->action, (uint64_t)W * 32, (uint64_t)ctx->lay.act_dim,
                                             (uint64_t)d->T, (uint64_t)io->act_cs, (uint64_t)d->act_ts, (uint32_t)sc) ? 1 : 0;
            const char* tm = getenv("CHAOS_B200_SM_TMAP");
            if (tm && tm[0] == '0') p.sm_tmap_ok = 0;
          }
        }
      }
      mode = cl::MODE_ROLLOUT_DYN;
      ctx->dyn_launches += 1;
    }
  }
  r = launch(ctx, p, mode, st);
  if (r == CL_OK) ctx->step_index += (uint64_t)d->T;
  return r;
}

// The fused policy kernels exist for hr_sync and pmsm_sync only.
static int check_policy_kind(cl_ctx* ctx, const char* fn, int kind) {
  if (kind == CL_ENV_HR_SYNC || kind == CL_ENV_PMSM_SYNC) return CL_OK;
  return fail(ctx, CL_EINVAL, "%s: env kind %d is not supported (hr_sync and pmsm_sync only)", fn, kind);
}

// The refusals the fused policy entry points share, in the order they make them.  fn names the entry point;
// objs lists the arguments it requires ("io/desc/policy/..."), objs_ok says whether those beyond io / desc /
// policy are there; with need_last, pol->obs_last is required as well.
static int policy_prelude(cl_ctx* ctx, const char* fn, const char* objs, bool objs_ok, const cl_io* io,
                          const cl_rollout_desc* d, const cl_policy* pol, bool need_last) {
  if (!ctx) return fail(nullptr, CL_EINVAL, "null ctx");
  const int r = check_policy_kind(ctx, fn, ctx->cfg.kind);
  if (r) return r;
  if (ctx->cfg.flags & CL_F_OBS_F64) return fail(ctx, CL_EINVAL, "%s: float32 observations only", fn);
  if (!io || !d || !pol || !objs_ok || d->T < 1) return fail(ctx, CL_EINVAL, "%s: %s required, T >= 1", fn, objs);
  if (io->action || io->noise) return fail(ctx, CL_EINVAL, "%s: io.action and io.noise must be NULL", fn);
  if (!pol->params || !pol->obs0 || (need_last && !pol->obs_last))
    return fail(ctx, CL_EINVAL, need_last ? "%s: params, obs0 and obs_last are required"
                                          : "%s: params and obs0 are required", fn);
  return CL_OK;
}

// The launch parameters of a fused policy window of d->T intervals, on the context's device.
static int policy_params(cl_ctx* ctx, const cl_buffers* buf, const cl_io* io, const cl_rollout_desc* d,
                         KParams& p) {
  const int r = fill_params(ctx, buf, io, p);
  if (r) return r;
  p.T = d->T; p.obs_ts = d->obs_ts; p.rew_ts = d->rew_ts; p.done_ts = d->done_ts;
  CU(cudaSetDevice(ctx->cfg.device));
  return CL_OK;
}

static bool collect_complete(const cl_collect* col) {
  return col->starts && col->obs && col->actions && col->rewards && col->values && col->log_probs &&
         col->episode_starts && col->last_values;
}

// After a fused policy launch: count it and advance the Philox step index by the window's T intervals.
static int policy_done(cl_ctx* ctx, cudaStream_t st, cudaError_t e, const char* what, int T) {
  if (e != cudaSuccess) return fail(ctx, CL_ECUDA, "%s launch failed: %s", what, cudaGetErrorString(e));
  ctx->launches += 1;
  const int r = advance_graph_step(ctx, st, (uint64_t)T);
  if (r == CL_OK) ctx->step_index += (uint64_t)T;
  return r;
}

extern "C" int cl_policy_rollout(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
                                 const cl_rollout_desc* d, const cl_policy* pol) {
  int r = policy_prelude(ctx, "cl_policy_rollout", "io/desc/policy", true, io, d, pol, false);
  if (r) return r;
  if ((pol->obs_mean == nullptr) != (pol->obs_var == nullptr))
    return fail(ctx, CL_EINVAL, "cl_policy_rollout: obs_mean and obs_var go together");
  if (pol->steady_start < 0 || pol->steady_start >= d->T)
    return fail(ctx, CL_EINVAL, "cl_policy_rollout: steady_start %d outside [0, T)", pol->steady_start);
  KParams p;
  if ((r = policy_params(ctx, buf, io, d, p))) return r;
  cudaStream_t st = (cudaStream_t)stream;
  const cudaError_t e = cl_launch_policy(ctx->cfg.kind, p, *pol, (float)ctx->lay.act_low, (float)ctx->lay.act_high,
                                         st, ctx->sm_count);
  return policy_done(ctx, st, e, "policy rollout", d->T);
}

extern "C" int cl_policy_collect(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
                                 const cl_rollout_desc* d, const cl_policy* pol, const cl_collect* col) {
  int r = policy_prelude(ctx, "cl_policy_collect", "io/desc/policy/collect", col != nullptr, io, d, pol, false);
  if (r) return r;
  if (pol->act_out || pol->metrics) return fail(ctx, CL_EINVAL, "cl_policy_collect: act_out and metrics must be NULL");
  if ((pol->obs_mean == nullptr) != (pol->obs_var == nullptr))
    return fail(ctx, CL_EINVAL, "cl_policy_collect: obs_mean and obs_var go together");
  if (!collect_complete(col))
    return fail(ctx, CL_EINVAL, "cl_policy_collect: starts, the six buffers and last_values are required");
  KParams p;
  if ((r = policy_params(ctx, buf, io, d, p))) return r;
  cudaStream_t st = (cudaStream_t)stream;
  const cudaError_t e = cl_launch_policy_collect(ctx->cfg.kind, p, *pol, *col, (float)ctx->lay.act_low,
                                                 (float)ctx->lay.act_high, st, ctx->sm_count);
  return policy_done(ctx, st, e, "policy collect", d->T);
}

extern "C" int cl_policy_collect_norm_scratch_bytes(int32_t kind, int64_t n, int64_t* out) {
  const int r = check_policy_kind(nullptr, "cl_policy_collect_norm_scratch_bytes", kind);
  if (r) return r;
  if (!out || n < 1) return fail(nullptr, CL_EINVAL, "cl_policy_collect_norm_scratch_bytes: n >= 1 and out required");
  *out = cl_policy_collect_norm_bytes(kLayouts[kind].obs_dim, n);
  return CL_OK;
}

extern "C" int cl_policy_collect_norm(cl_ctx* ctx, void* stream, const cl_buffers* buf, const cl_io* io,
                                      const cl_rollout_desc* d, const cl_policy* pol, const cl_collect* col,
                                      const cl_vecnorm_update* vn) {
  int r = policy_prelude(ctx, "cl_policy_collect_norm", "io/desc/policy/collect/vecnorm", col && vn, io, d, pol,
                         true);
  if (r) return r;
  if (pol->act_out || pol->metrics)
    return fail(ctx, CL_EINVAL, "cl_policy_collect_norm: act_out and metrics must be NULL");
  if (pol->obs_mean || pol->obs_var)
    return fail(ctx, CL_EINVAL, "cl_policy_collect_norm: pol.obs_mean / obs_var must be NULL (the statistics "
                "come from the vecnorm argument)");
  if (!collect_complete(col))
    return fail(ctx, CL_EINVAL, "cl_policy_collect_norm: starts, the six buffers and last_values are required");
  if (!vn->ret_mean || !vn->ret_var || !vn->ret_count || !vn->returns ||
      (vn->norm_obs && (!vn->obs_mean || !vn->obs_var || !vn->obs_count)))
    return fail(ctx, CL_EINVAL, "cl_policy_collect_norm: the ret_rms statistics, returns and (norm_obs) the "
                "obs_rms statistics are required");
  const int64_t need = cl_policy_collect_norm_bytes(ctx->lay.obs_dim, ctx->cfg.num_envs);
  if (!vn->scratch || vn->scratch_bytes < need)
    return fail(ctx, CL_EINVAL, "cl_policy_collect_norm: scratch of %lld bytes required, got %lld", (long long)need,
                (long long)vn->scratch_bytes);
  KParams p;
  if ((r = policy_params(ctx, buf, io, d, p))) return r;
  cudaStream_t st = (cudaStream_t)stream;
  const cudaError_t e = cl_launch_policy_collect_norm(ctx->cfg.kind, p, *pol, *col, *vn, (float)ctx->lay.act_low,
                                                      (float)ctx->lay.act_high, st, ctx->sm_count);
  return policy_done(ctx, st, e, "policy collect (training-mode VecNormalize)", d->T);
}

extern "C" int64_t cl_dyn_launch_count(const cl_ctx* ctx) { return ctx ? ctx->dyn_launches : 0; }
extern "C" int64_t cl_plain_launch_count(const cl_ctx* ctx) { return ctx ? ctx->plain_launches : 0; }
extern "C" int64_t cl_sm_launch_count(const cl_ctx* ctx) { return ctx ? ctx->sm_launches : 0; }

extern "C" int cl_derivatives(cl_ctx* ctx, void* stream, const void* state, const float* action,
                              void* out, int64_t n) {
  if (!ctx || !state || !out || n <= 0) return fail(ctx, CL_EINVAL, "cl_derivatives: bad argument");
  CU(cudaSetDevice(ctx->cfg.device));
  cudaError_t e = cl_launch_derivatives(ctx->cfg.kind, state, action, out, n, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(ctx, CL_ECUDA, "cl_derivatives: %s", cudaGetErrorString(e));
  ctx->launches += 1;
  return CL_OK;
}

extern "C" int cl_stats(cl_ctx* ctx, void* stream, const cl_buffers* buf, double* out8, int clear) {
  if (!ctx || !buf || !buf->stats || !out8) return fail(ctx, CL_EINVAL, "cl_stats: bad argument");
  CU(cudaSetDevice(ctx->cfg.device));
  CU(cudaMemcpyAsync(out8, buf->stats, sizeof(double) * CL_NSTATS, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (clear) CU(cudaMemsetAsync(buf->stats, 0, sizeof(double) * CL_NSTATS, (cudaStream_t)stream));
  return CL_OK;
}

extern "C" int cl_get_step_index(const cl_ctx* ctx, uint64_t* out) {
  if (!ctx || !out) return CL_EINVAL;
  if (ctx->graph_mode) {  // the device counter is authoritative (graph replays advance only it)
    if (cudaSetDevice(ctx->cfg.device) != cudaSuccess) return CL_ECUDA;
    if (cudaDeviceSynchronize() != cudaSuccess) return CL_ECUDA;
    if (cudaMemcpy(out, ctx->d_step, sizeof(uint64_t), cudaMemcpyDeviceToHost) != cudaSuccess) return CL_ECUDA;
    return CL_OK;
  }
  *out = ctx->step_index;
  return CL_OK;
}
extern "C" int cl_set_step_index(cl_ctx* ctx, uint64_t v) {
  if (!ctx) return CL_EINVAL;
  ctx->step_index = v;
  if (ctx->graph_mode) {
    if (cudaSetDevice(ctx->cfg.device) != cudaSuccess) return CL_ECUDA;
    if (cudaMemcpy(ctx->d_step, &v, sizeof(uint64_t), cudaMemcpyHostToDevice) != cudaSuccess) return CL_ECUDA;
  }
  return CL_OK;
}
extern "C" int cl_set_graph_mode(cl_ctx* ctx, int enable) {
  if (!ctx) return CL_EINVAL;
  if (cudaSetDevice(ctx->cfg.device) != cudaSuccess) return CL_ECUDA;
  if (cudaDeviceSynchronize() != cudaSuccess) return CL_ECUDA;
  if (enable && !ctx->graph_mode) {
    const uint64_t init[2] = {ctx->step_index, 0};
    if (cudaMemcpy(ctx->d_step, init, sizeof(init), cudaMemcpyHostToDevice) != cudaSuccess) return CL_ECUDA;
  } else if (!enable && ctx->graph_mode) {
    uint64_t v = 0;
    if (cudaMemcpy(&v, ctx->d_step, sizeof(uint64_t), cudaMemcpyDeviceToHost) != cudaSuccess) return CL_ECUDA;
    ctx->step_index = v;
  }
  ctx->graph_mode = enable ? 1 : 0;
  return CL_OK;
}
extern "C" int64_t cl_launch_count(const cl_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" int cl_block_size(const cl_ctx* ctx) { return ctx ? ctx->block : 0; }

// ---- host-buffer path ------------------------------------------------------------------

// Default data-movement mode of the host path per (env kind, batch size), from the measured table
// profiles/r02_e2e_host_modes.jsonl (tools/e2e_modes.py: lorenz_rk4 / hr_sync / pmsm_sync x {4,096, 16,384,
// 65,536} envs x {DMA chain, zero-copy, streamed 8 / 32 slices}, a caller-owned action array each step).
// What decides is the size of the action array (kind enters through its action dimension): the DMA chain
// never wins, streamed wins once the staging copy is long enough to hide a relay launch behind.
static void host_mode_default(int kind, int64_t n, int* mode, int* slices) {
  const int64_t action_bytes = n * (int64_t)kLayouts[kind].act_dim * 4;
  // With the relay inside the step kernel streaming costs no second launch, so it pays from smaller arrays than
  // with the separate relay kernel (384 KB then).  A-B-A-B on one env, caller-owned array, us per step zero-copy vs
  // streamed (profiles/r02f4_e2e_small_ab.jsonl, r02f3_e2e_host_modes.jsonl): 48 KB of actions 32.5-35.3 vs 33.3-35.7,
  // 64 KB 39.3 vs 40.4, 96 KB 40.7-42.5 vs 39.1-40.5, 128 KB 36.3-36.9 vs 33.4-33.9, 192 KB 38.9-41.9 vs 34.1-36.9,
  // 768 KB 109.7 vs 64.8, 3 MB 377 vs 195.
  if (action_bytes >= 96 * 1024) {
    *mode = CL_HOST_STREAMED;
    int k = (int)(n / 2048);           // finer slices keep paying up to the relay's poll period (~4 us of staging)
    *slices = k < 1 ? 1 : (k > 64 ? 64 : k);
  } else {
    *mode = CL_HOST_ZEROCOPY;
    *slices = 1;
  }
}

static int host_stage_init(cl_ctx* ctx) {
  HostStage& h = ctx->hs;
  if (h.ready) return CL_OK;
  const size_t N = (size_t)ctx->cfg.num_envs, NP = (size_t)ctx->cfg.n_pad;
  const size_t A = (size_t)ctx->lay.act_dim, O = (size_t)ctx->lay.obs_dim;
  CU(cudaSetDevice(ctx->cfg.device));
  CU(cudaStreamCreateWithFlags(&h.stream, cudaStreamNonBlocking));
  CU(cudaHostAlloc((void**)&h.h_act, N * A * sizeof(float), cudaHostAllocDefault));
  CU(cudaMalloc((void**)&h.d_act, N * A * sizeof(float)));
  h.wd_bytes = (((N + 31) / 32) + 7) / 8 * 8;
  const size_t wd_off = (N * O * sizeof(float) + N * sizeof(float) + N + 7) / 8 * 8;
  h.out_bytes = wd_off + h.wd_bytes;
  CU(cudaMalloc((void**)&h.d_out, h.out_bytes));
  h.d_warp_done = h.d_out + wd_off;
  CU(cudaHostAlloc((void**)&h.h_ready, 80 * sizeof(uint32_t), cudaHostAllocDefault));
  memset(h.h_ready, 0, 80 * sizeof(uint32_t));
  h.h_err = h.h_ready + 72;
  h.gen = 0;
  CU(cudaMalloc((void**)&h.d_ready, CL_STAGE_MAX_LANES * sizeof(uint32_t)));
  CU(cudaMemset(h.d_ready, 0, CL_STAGE_MAX_LANES * sizeof(uint32_t)));
  h.d_obs = (float*)h.d_out;
  h.d_rew = (float*)(h.d_out + N * O * sizeof(float));
  h.d_done = (uint8_t*)(h.d_out + N * O * sizeof(float) + N * sizeof(float));
  CU(cudaMalloc((void**)&h.d_term, N * O * sizeof(float)));
  CU(cudaMalloc((void**)&h.d_ler, NP * sizeof(double)));
  CU(cudaMalloc((void**)&h.d_lel, NP * sizeof(int32_t)));
  CU(cudaMemset(h.d_term, 0, N * O * sizeof(float)));
  CU(cudaMemset(h.d_ler, 0, NP * sizeof(double)));
  CU(cudaMemset(h.d_lel, 0, NP * sizeof(int32_t)));
  for (int k = 0; k < kHostRing; ++k) {
    CU(cudaHostAlloc((void**)&h.slot[k].out, h.out_bytes, cudaHostAllocDefault));
    h.slot[k].obs = (float*)h.slot[k].out;
    h.slot[k].reward = (float*)(h.slot[k].out + N * O * sizeof(float));
    h.slot[k].done = (uint8_t*)(h.slot[k].out + N * O * sizeof(float) + N * sizeof(float));
    h.slot[k].warp_done = h.slot[k].out + wd_off;
    CU(cudaHostAlloc((void**)&h.slot[k].term_obs, N * O * sizeof(float), cudaHostAllocDefault));
    CU(cudaHostAlloc((void**)&h.slot[k].last_ep_ret, N * sizeof(double), cudaHostAllocDefault));
    CU(cudaHostAlloc((void**)&h.slot[k].last_ep_len, N * sizeof(int32_t), cudaHostAllocDefault));
  }
  h.cur = 0;
  h.pending = false;
  CU(cudaStreamCreateWithFlags(&h.side, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&h.ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&h.ev_join, cudaEventDisableTiming));
  // default: zero-copy (one launch, no copies: 23 / 73 us per step at 4,096 / 65,536 Lorenz envs
  // vs 31 / 88 us for the DMA chain).  The sliced pipeline only pays when the caller's ndarray has
  // to be staged at >= 262,144 envs: each slice costs ~9 us of host-side launch time
  // (profiles/r01_e2e_host_modes.jsonl).  CHAOS_B200_HOST_MODE=dma|zerocopy|pipelined and
  // CHAOS_B200_HOST_SLICES=k override (tuning); CHAOS_B200_ZEROCOPY=0 is the older spelling of dma.
  host_mode_default(ctx->cfg.kind, (int64_t)N, &h.mode, &h.slices);
  if (const char* ov = getenv("CHAOS_B200_ZEROCOPY")) { if (ov[0] == '0') h.mode = CL_HOST_DMA; }
  if (const char* ov = getenv("CHAOS_B200_HOST_MODE")) {
    if (!strcmp(ov, "dma")) h.mode = CL_HOST_DMA;
    else if (!strcmp(ov, "zerocopy")) h.mode = CL_HOST_ZEROCOPY;
    else if (!strcmp(ov, "pipelined")) { h.mode = CL_HOST_PIPELINED; if (h.slices < 2) h.slices = 2; }
    else if (!strcmp(ov, "streamed")) h.mode = CL_HOST_STREAMED;
  }
  if (const char* ov = getenv("CHAOS_B200_HOST_SLICES")) { const int k = atoi(ov); if (k >= 1 && k <= 64) h.slices = k; }
  h.helper = copy_helper_start(N * A * sizeof(float));
  { const char* ov = getenv("CHAOS_B200_RELAY"); h.relay_kernel = (ov && !strcmp(ov, "kernel")) ? 1 : 0; }
  h.ready = true;
  return CL_OK;
}

static cudaStream_t host_stream(cl_ctx* ctx, void* stream) {
  // stream == (void*)-1 selects the context's own non-blocking stream
  return stream == (void*)(intptr_t)-1 ? ctx->hs.stream : (cudaStream_t)stream;
}

extern "C" int cl_host_action_staging(cl_ctx* ctx, float** act) {
  if (!ctx || !act) return fail(ctx, CL_EINVAL, "bad argument");
  int r = host_stage_init(ctx);
  if (r) return r;
  *act = ctx->hs.h_act;
  return CL_OK;
}

static int host_step_launch(cl_ctx* ctx, cudaStream_t st, const cl_buffers* buf, const float* action_host);

extern "C" int cl_step_host_async(cl_ctx* ctx, void* stream, const cl_buffers* buf, const float* action_host) {
  if (!ctx) return fail(nullptr, CL_EINVAL, "null ctx");
  int r = host_stage_init(ctx);
  if (r) return r;
  HostStage& h = ctx->hs;
  if (h.pending) return fail(ctx, CL_EINVAL, "cl_step_host_async called twice without cl_step_host_wait");
  if (!buf) return fail(ctx, CL_EINVAL, "cl_buffers required");
  CU(cudaSetDevice(ctx->cfg.device));
  h.redo_buf = *buf;   // cl_step_host_wait redoes a called-off streamed step from the staging buffer
  return host_step_launch(ctx, host_stream(ctx, stream), buf, action_host);
}

static int host_step_launch(cl_ctx* ctx, cudaStream_t st, const cl_buffers* buf, const float* action_host) {
  HostStage& h = ctx->hs;
  int r = CL_OK;
  const size_t N = (size_t)ctx->cfg.num_envs;
  const size_t A = (size_t)ctx->lay.act_dim, O = (size_t)ctx->lay.obs_dim;
  const bool stage_copy = action_host && action_host != h.h_act;
  // graph capture cannot contain CPU-side staging: captured steps read the pinned buffer as it is
  int mode = ((h.mode == CL_HOST_PIPELINED || h.mode == CL_HOST_STREAMED) && ctx->graph_mode) ? CL_HOST_ZEROCOPY : h.mode;
  if (mode == CL_HOST_STREAMED && !stage_copy) mode = CL_HOST_ZEROCOPY;   // the caller wrote the pinned buffer itself
  const bool host_out = mode != CL_HOST_DMA;       // kernel writes obs / reward / done to pinned host memory
  const bool host_in = mode == CL_HOST_ZEROCOPY || mode == CL_HOST_STREAMED;   // kernel reads the actions from pinned host memory
  h.cur = (h.cur + 1) % kHostRing;
  HostSlot& s = h.slot[h.cur];
  cl_io io;
  memset(&io, 0, sizeof(io));
  io.action = host_in ? h.h_act : h.d_act; io.act_es = (int64_t)A; io.act_cs = 1;
  io.obs = host_out ? s.obs : h.d_obs; io.obs_es = (int64_t)O; io.obs_cs = 1;
  io.reward = host_out ? s.reward : h.d_rew; io.done = host_out ? s.done : h.d_done;
  // finished episodes: terminal observation and Monitor numbers go straight to the host slot too
  // (whole rows of the warps concerned), so a step that ends episodes needs no extra copies
  io.term_obs = host_out ? s.term_obs : h.d_term;
  io.last_ep_ret = host_out ? s.last_ep_ret : h.d_ler; io.last_ep_len = host_out ? s.last_ep_len : h.d_lel;
  h.extras_on_host = host_out;
  KParams p;
  r = fill_params(ctx, buf, &io, p);
  if (r) return r;
  p.reward_f32 = 1;
  p.flags &= ~CL_F_OBS_F64;
  // per-env-warp "an episode ended" flags: cleared here, set by the kernel, scanned by cl_step_host_wait
  // (N / 32 bytes instead of the N done flags)
  if (host_out) { memset(s.warp_done, 0, h.wd_bytes); p.warp_done = s.warp_done; p.host_rows = 1; }
  else { CU(cudaMemsetAsync(h.d_warp_done, 0, h.wd_bytes, st)); p.warp_done = h.d_warp_done; }
  if (mode == CL_HOST_STREAMED) {
    // 1. launch the step kernel, whose blocks wait for the slice they read; its block 0 is the relay that mirrors
    //    the pinned "slices staged" words into device memory (or k_relay on the side stream, CHAOS_B200_RELAY=kernel);
    // 2. stage the caller's array into the pinned buffer: the slices are dealt out to staging lanes (one copy
    //    thread each, host_copy.h), every lane publishes its count after each slice.  The final counts are
    //    stored whatever happens in between, so both kernels always terminate (and their waits are bounded anyway).
    const int blk = ctx->block;
    int slices = h.slices < 1 ? 1 : (h.slices > 64 ? 64 : h.slices);
    size_t per = ((N + (size_t)slices - 1) / (size_t)slices + (size_t)blk - 1) / (size_t)blk * (size_t)blk;   // whole blocks
    h.gen = (h.gen + 1) & 0x00FFFFFFu;
    if (h.gen == 0) h.gen = 1;
    *h.h_err = 0u;
    const uint32_t nsl = (uint32_t)((N + per - 1) / per);
    uint32_t spl = 1;
    const uint32_t lanes = stage_plan(h.helper, nsl, &spl);
    for (uint32_t k = 0; k < lanes; ++k)
      __atomic_store_n(&h.h_ready[k * CL_STAGE_WORD_STRIDE], h.gen << 8, __ATOMIC_RELEASE);
    // whatever happens below, the relay (and any block already running) must get to see every lane complete
    auto publish_all = [&]() {
      for (uint32_t k = 0; k < lanes; ++k)
        __atomic_store_n(&h.h_ready[k * CL_STAGE_WORD_STRIDE], (h.gen << 8) | stage_lane_count(k, spl, nsl), __ATOMIC_RELEASE);
    };
    p.act_ready = h.d_ready; p.act_gen = h.gen; p.act_slice_envs = (int32_t)per; p.act_lane_slices = (int32_t)spl;
    p.host_err = h.h_err;
    if (h.relay_kernel) {
      k_relay<<<1, 32, 0, h.side>>>(h.h_ready, h.d_ready, h.gen, lanes, spl, nsl, h.h_err);
      if (cudaGetLastError() != cudaSuccess) {
        publish_all();
        return fail(ctx, CL_ECUDA, "relay kernel launch failed");
      }
    } else {
      p.act_host_words = h.h_ready; p.act_lanes = (int32_t)lanes; p.act_nslices = (int32_t)nsl;
    }
    r = launch(ctx, p, cl::MODE_STEP, st);
    if (r == CL_OK)
      stage_slices(h.helper, (unsigned char*)h.h_act, (const unsigned char*)action_host, per * A * sizeof(float),
                   N * A * sizeof(float), nsl, h.gen, h.h_ready);
    publish_all();
    if (r) return r;
  } else if (mode == CL_HOST_PIPELINED && h.slices > 1) {
    // slice j runs on stream (j & 1): [DMA its actions in] -> [kernel: step, write results to host].
    // The user's array is staged into pinned memory slice by slice too, so that host memcpy
    // overlaps the device work of the slices already enqueued.
    const size_t per = ((N + (size_t)h.slices - 1) / (size_t)h.slices + 255) / 256 * 256;  // whole blocks / warps
    CU(cudaEventRecord(h.ev_fork, st));
    CU(cudaStreamWaitEvent(h.side, h.ev_fork, 0));
    int j = 0;
    for (size_t b = 0; b < N; b += per, ++j) {
      const size_t e = b + per < N ? b + per : N;
      cudaStream_t sj = (j & 1) ? h.side : st;
      if (stage_copy) memcpy(h.h_act + b * A, action_host + b * A, (e - b) * A * sizeof(float));
      CU(cudaMemcpyAsync(h.d_act + b * A, h.h_act + b * A, (e - b) * A * sizeof(float), cudaMemcpyHostToDevice, sj));
      p.i_begin = (int64_t)b;
      p.n = (int64_t)e;
      r = launch(ctx, p, cl::MODE_STEP, sj);
      if (r) return r;
    }
    CU(cudaEventRecord(h.ev_join, h.side));
    CU(cudaStreamWaitEvent(st, h.ev_join, 0));
  } else {
    if (stage_copy) stage_copy_bytes(h.h_act, action_host, N * A * sizeof(float));
    if (!host_in) CU(cudaMemcpyAsync(h.d_act, h.h_act, N * A * sizeof(float), cudaMemcpyHostToDevice, st));
    r = launch(ctx, p, cl::MODE_STEP, st);
    if (r) return r;
  }
  ctx->step_index += 1;
  if (!host_out) CU(cudaMemcpyAsync(s.out, h.d_out, h.out_bytes, cudaMemcpyDeviceToHost, st));
  h.pending = true;
  return CL_OK;
}

extern "C" int cl_host_set_zero_copy(cl_ctx* ctx, int enable) {
  return cl_host_set_mode(ctx, enable ? CL_HOST_ZEROCOPY : CL_HOST_DMA, 1);
}

extern "C" int cl_host_set_mode(cl_ctx* ctx, int mode, int slices) {
  if (!ctx) return CL_EINVAL;
  if (mode < CL_HOST_DMA || mode > CL_HOST_STREAMED || slices < 1 || slices > 64)
    return fail(ctx, CL_EINVAL, "cl_host_set_mode: mode %d / slices %d out of range", mode, slices);
  int r = host_stage_init(ctx);
  if (r) return r;
  if (ctx->hs.pending) return fail(ctx, CL_EINVAL, "cl_host_set_mode with a step in flight");
  ctx->hs.mode = mode;
  ctx->hs.slices = slices;
  return CL_OK;
}

static int host_wait_common(cl_ctx* ctx, void* stream, int64_t* n_done_out) {
  HostStage& h = ctx->hs;
  if (!h.ready || !h.pending) return fail(ctx, CL_EINVAL, "cl_step_host_wait without a pending cl_step_host_async");
  cudaStream_t st = host_stream(ctx, stream);
  CU(cudaSetDevice(ctx->cfg.device));
  CU(cudaStreamSynchronize(st));
  h.pending = false;
  const size_t N = (size_t)ctx->cfg.num_envs, O = (size_t)ctx->lay.obs_dim;
  HostSlot& s = h.slot[h.cur];
  if (*h.h_err) {
    const uint32_t code = *h.h_err;
    *h.h_err = 0u;
    CU(cudaStreamSynchronize(h.side));
    if (code != 2u) return fail(ctx, CL_ECUDA, "streamed host step: staging stalled for 2 s after a partial publication");
    // Called off before any block stored anything (k_relay): launches are synchronous here, streaming
    // cannot work.  Redo the step from the staging buffer (complete by now) as a plain zero-copy step --
    // same Philox step index, same result slot -- and keep this context out of streamed mode.
    h.mode = CL_HOST_ZEROCOPY;
    h.streamed_fallbacks += 1;
    ctx->step_index -= 1;
    h.cur = (h.cur + kHostRing - 1) % kHostRing;
    int r = host_step_launch(ctx, st, &h.redo_buf, nullptr);
    if (r) return r;
    CU(cudaStreamSynchronize(st));
    h.pending = false;
  }
  // finished episodes: scan the per-env-warp flags (N / 32 bytes, 8 at a time); count the done
  // flags only inside flagged warps
  int64_t nd = 0;
  const size_t W = (N + 31) / 32;
  for (size_t w8 = 0; w8 < h.wd_bytes; w8 += 8) {
    uint64_t word;
    memcpy(&word, s.warp_done + w8, 8);
    if (!word) continue;
    for (size_t w = w8; w < w8 + 8 && w < W; ++w) {
      if (!s.warp_done[w]) continue;
      const size_t lo = w * 32, hi = lo + 32 < N ? lo + 32 : N;
      for (size_t i = lo; i < hi; ++i) nd += (s.done[i] != 0);
    }
  }
  if (nd > 0 && !h.extras_on_host) {  // DMA mode: fetch the terminal observations and Monitor numbers
    CU(cudaMemcpyAsync(s.term_obs, h.d_term, N * O * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(s.last_ep_ret, h.d_ler, N * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(s.last_ep_len, h.d_lel, N * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  *n_done_out = nd;
  return CL_OK;
}

extern "C" int cl_step_host_wait_view(cl_ctx* ctx, void* stream, cl_host_view* v) {
  if (!ctx || !v) return fail(ctx, CL_EINVAL, "bad argument");
  int64_t nd = 0;
  int r = host_wait_common(ctx, stream, &nd);
  if (r) return r;
  HostSlot& s = ctx->hs.slot[ctx->hs.cur];
  v->obs = s.obs; v->reward = s.reward; v->done = s.done; v->term_obs = s.term_obs;
  v->last_ep_ret = s.last_ep_ret; v->last_ep_len = s.last_ep_len; v->n_done = nd;
  return CL_OK;
}

extern "C" int cl_step_host_wait(cl_ctx* ctx, void* stream, float* obs_host, float* reward_host,
                                 uint8_t* done_host, float* term_obs_host, double* last_ep_ret_host,
                                 int32_t* last_ep_len_host, int64_t* n_done) {
  if (!ctx) return fail(nullptr, CL_EINVAL, "null ctx");
  int64_t nd = 0;
  int r = host_wait_common(ctx, stream, &nd);
  if (r) return r;
  const size_t N = (size_t)ctx->cfg.num_envs, O = (size_t)ctx->lay.obs_dim;
  HostSlot& s = ctx->hs.slot[ctx->hs.cur];
  if (obs_host) memcpy(obs_host, s.obs, N * O * sizeof(float));
  if (reward_host) memcpy(reward_host, s.reward, N * sizeof(float));
  if (done_host) memcpy(done_host, s.done, N);
  if (nd > 0) {
    if (term_obs_host) memcpy(term_obs_host, s.term_obs, N * O * sizeof(float));
    if (last_ep_ret_host) memcpy(last_ep_ret_host, s.last_ep_ret, N * sizeof(double));
    if (last_ep_len_host) memcpy(last_ep_len_host, s.last_ep_len, N * sizeof(int32_t));
  }
  if (n_done) *n_done = nd;
  return CL_OK;
}

extern "C" int cl_reset_host(cl_ctx* ctx, void* stream, const cl_buffers* buf, float* obs_host) {
  if (!ctx || !obs_host) return fail(ctx, CL_EINVAL, "bad argument");
  int r = host_stage_init(ctx);
  if (r) return r;
  HostStage& h = ctx->hs;
  const size_t N = (size_t)ctx->cfg.num_envs, O = (size_t)ctx->lay.obs_dim;
  cudaStream_t st = host_stream(ctx, stream);
  cl_io io;
  memset(&io, 0, sizeof(io));
  io.obs = h.d_obs; io.obs_es = (int64_t)O; io.obs_cs = 1;
  KParams p;
  r = fill_params(ctx, buf, &io, p);
  if (r) return r;
  p.flags &= ~CL_F_OBS_F64;
  CU(cudaSetDevice(ctx->cfg.device));
  r = launch(ctx, p, cl::MODE_RESET, st);
  if (r) return r;
  ctx->step_index += 1;
  h.cur = (h.cur + 1) % kHostRing;
  CU(cudaMemcpyAsync(h.slot[h.cur].obs, h.d_obs, N * O * sizeof(float), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  memcpy(obs_host, h.slot[h.cur].obs, N * O * sizeof(float));
  return CL_OK;
}

extern "C" int64_t cl_host_streamed_fallbacks(const cl_ctx* ctx) { return ctx ? ctx->hs.streamed_fallbacks : 0; }

extern "C" int64_t cl_host_h2d_bytes(const cl_ctx* ctx) {
  return ctx ? ctx->cfg.num_envs * ctx->lay.act_dim * (int64_t)sizeof(float) : 0;
}
extern "C" int64_t cl_host_d2h_bytes(const cl_ctx* ctx) {
  return ctx ? ctx->cfg.num_envs * (ctx->lay.obs_dim * (int64_t)sizeof(float) + (int64_t)sizeof(float) + 1) : 0;
}

// ---- measurement -----------------------------------------------------------------------

extern "C" int cl_measure_fma_peak(int32_t device, int32_t dtype_bytes, double seconds, double* tflops) {
  cl_ctx* ctx = nullptr;
  if (!tflops || (dtype_bytes != 8 && dtype_bytes != 4)) return fail(nullptr, CL_EINVAL, "bad argument");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int block = 256, grid = prop.multiProcessorCount * 8;
  void* sink = nullptr;
  CU(cudaMalloc(&sink, 64));
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  int iters = 2000;
  double best = 0.0, spent = 0.0;
  // warm-up + adaptive repetition: best of the launches that fit in `seconds`
  for (int rep = 0; rep < 64; ++rep) {
    CU(cudaEventRecord(e0, 0));
    CU(cl_fma_peak_launch(dtype_bytes, grid, block, iters, sink, 0));
    CU(cudaEventRecord(e1, 0));
    CU(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8.0 * 16.0 * (double)iters * (double)grid * (double)block;
    const double tf = fl / ((double)ms * 1e-3) * 1e-12;
    if (rep > 0 && tf > best) best = tf;
    if (rep > 0) spent += (double)ms * 1e-3;
    if (ms < 20.f) iters *= 2;
    if (spent >= seconds && rep >= 3) break;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  *tflops = best;
  return CL_OK;
}

// ---- host-side test hooks ----------------------------------------------------------------

extern "C" void cl_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  cl::u32x4 c;
  c.x = ctr[0]; c.y = ctr[1]; c.z = ctr[2]; c.w = ctr[3];
  const cl::u32x4 r = cl::philox4x32_10(c, key[0], key[1]);
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

extern "C" double cl_uniform53(uint32_t a, uint32_t b, double lo, double hi) {
  return cl::uniform53(a, b, lo, hi);
}
