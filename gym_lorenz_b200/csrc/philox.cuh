// Philox4x32-10 counter-based generator (Salmon, Moraes, Dror, Shaw: "Parallel random
// numbers: as easy as 1, 2, 3", SC'11) plus the uniform / normal mappings used by the
// env kernels.  Written from the published algorithm; verified against the Random123
// known-answer vectors in tests/test_philox.py.
//
// Stream layout (GPU-count invariant, see DESIGN.md "RNG"):
//   key     = (seed_lo, seed_hi)
//   counter = (global_env_id_lo, global_env_id_hi, step_index, purpose_tag + block)
// i.e. one independent subsequence per *global* env index, advanced by the global step
// index, so a slab of envs produces the same numbers no matter which rank owns it.
//
// The reference draws from NumPy's global MT19937 / a PCG64 Generator
// (dynamic.py:37, lorenz_env_try.py:55-67, lorenz_env_try_pmsm.py:64-65,80); those
// streams cannot be reproduced by a counter-based generator, so parity tests inject
// states and noise, and reset is checked distributionally + exactly against
// the CPU checker's independent restatement of this same mapping.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define CL_HD __host__ __device__ __forceinline__
#else
#define CL_HD static inline
#endif

namespace cl {

enum PhiloxTag : uint32_t {
  TAG_RESET  = 0x00000000u,  // + block index 0..3 (initial conditions)
  TAG_NOISE  = 0x10000000u,  // + block index 0..1 (per-step process noise)
  TAG_ACTION = 0x20000000u,  // synthetic random actions of the fused rollout
  TAG_PARAM  = 0x30000000u,  // per-env parameter randomisation
  TAG_POLICY = 0x40000000u,  // Gaussian policy noise of the rollout collector (cl_policy_collect)
};

struct u32x4 { uint32_t x, y, z, w; };

CL_HD void mulhilo32(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
  lo = a * b;
  hi = __umulhi(a, b);
#else
  uint64_t p = (uint64_t)a * (uint64_t)b;
  lo = (uint32_t)p;
  hi = (uint32_t)(p >> 32);
#endif
}

CL_HD u32x4 philox4x32_10(u32x4 c, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  const uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    mulhilo32(M0, c.x, hi0, lo0);
    mulhilo32(M1, c.z, hi1, lo1);
    u32x4 n;
    n.x = hi1 ^ c.y ^ k0;
    n.y = lo1;
    n.z = hi0 ^ c.w ^ k1;
    n.w = lo0;
    c = n;
    k0 += W0;
    k1 += W1;
  }
  return c;
}

// Per-env stream handle.
struct Stream {
  uint32_t id_lo, id_hi, step, k0, k1;
  CL_HD u32x4 draw(uint32_t tag_block) const {
    u32x4 c;
    c.x = id_lo; c.y = id_hi; c.z = step; c.w = tag_block;
    return philox4x32_10(c, k0, k1);
  }
};

// 53-bit uniform in [0,1): same construction as NumPy's random_double
// ((a >> 5) * 2^26 + (b >> 6)) / 2^53, from two 32-bit words.
CL_HD double u01_53(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  // the same 53-bit integer assembled from two exact 32-bit conversions ((a >> 5) * 2^26 + (b >> 6) < 2^53 is
  // exact in double): a 64-bit integer -> double conversion is a multi-instruction sequence on the GPU
  return __fma_rn((double)(a >> 5), 67108864.0, (double)(b >> 6)) * (1.0 / 9007199254740992.0);
#else
  return (double)(((uint64_t)(a >> 5) << 26) | (uint64_t)(b >> 6)) * (1.0 / 9007199254740992.0);
#endif
}

// uniform(lo, hi) as NumPy evaluates it: lo + (hi - lo) * u  (two roundings, no FMA).
CL_HD double uniform53(uint32_t a, uint32_t b, double lo, double hi) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(lo, __dmul_rn(hi - lo, u01_53(a, b)));
#else
  volatile double t = (hi - lo) * u01_53(a, b);
  return lo + t;
#endif
}

// 24-bit uniform in [0,1) as float (exact).
CL_HD float u01_24(uint32_t a) { return (float)(a >> 8) * (1.0f / 16777216.0f); }

}  // namespace cl
