// Shared helpers for the sm_100a kernels of libibm_b200.so.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ibm_b200.h"

namespace ibm {

void set_error(const char* fmt, ...);
int check_arch();                       // IBM_OK iff current device is sm_100
int sm_count();
// 1 if the launch being prepared should walk its rows / tiles in DESCENDING order (see ibm_set_walk_order); launches
// streaming less than 48 MB neither alternate nor count
int next_walk_reverse(int64_t bytes_streamed);

#define IBM_CHECK_ARG(cond, ...)                       \
  do {                                                 \
    if (!(cond)) {                                     \
      ibm::set_error(__VA_ARGS__);                     \
      return IBM_E_ARG;                                \
    }                                                  \
  } while (0)

#define IBM_CHECK_CUDA(expr)                                                            \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      ibm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return IBM_E_CUDA;                                                                \
    }                                                                                   \
  } while (0)

#define IBM_CHECK_ARCH()            \
  do {                              \
    int _a = ibm::check_arch();     \
    if (_a != IBM_OK) return _a;    \
  } while (0)

#define IBM_LAUNCH_CHECK() IBM_CHECK_CUDA(cudaGetLastError())

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static inline bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3) == 0; }
// a softmax scale the attention kernels handle: they take the row maximum of the raw scores and scale afterwards
static inline bool attn_scale_ok(float s) { return s > 0.f && s < INFINITY; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

// streaming 16-byte accesses (data touched once: bypass L1 allocation)
__device__ __forceinline__ uint4 ld_stream16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream16(void* p, uint4 v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
  uint4 r = ld_stream16(p);
  return make_float4(__uint_as_float(r.x), __uint_as_float(r.y), __uint_as_float(r.z), __uint_as_float(r.w));
}
__device__ __forceinline__ void st_stream_f4(float* p, float4 v) {
  st_stream16(p, make_uint4(__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w)));
}

// The CoP contact test of the reference evaluator (mask_by_threes on the label force, threshold 10.0 at
// RegressionLossEvaluator.py:205-209): ||f|| > thr, strict, the norm accumulated as (a*a + b*b) + c*c without FMA
// contraction like the reference's fp32 torch.norm.  norm3_gt2 is the same predicate without the square root, with
// thr2 = norm3_threshold_sq(thr) from the host; the loss and ensemble kernels share both so their contact decisions agree.
__device__ __forceinline__ bool norm3_gt2(float a, float b, float c, float thr2) {
  return __fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), __fmul_rn(c, c)) > thr2;
}
// largest fp32 x with sqrtf(x) <= thr, so that (sqrtf(n2) > thr)  <=>  (n2 > x) bit for bit (sqrtf is correctly rounded and
// monotonic, so this is exact); -1 for a negative threshold, which every norm exceeds
static inline float norm3_threshold_sq(float thr) {
  if (thr < 0.f) return -1.f;
  float x = thr * thr;
  while (sqrtf(nextafterf(x, INFINITY)) <= thr) x = nextafterf(x, INFINITY);
  while (x > 0.f && sqrtf(x) > thr) x = nextafterf(x, -INFINITY);
  return x;
}

// activations and their derivatives expressed through the activation OUTPUT y
__device__ __forceinline__ float act_apply(float x, int act) {
  switch (act) {
    case IBM_ACT_RELU: return fmaxf(x, 0.f);
    case IBM_ACT_SIGMOID: return 1.f / (1.f + __expf(-x));
    case IBM_ACT_TANH: return tanhf(x);
    case IBM_ACT_ELU: return x > 0.f ? x : expm1f(x);
    case IBM_ACT_SILU: return x / (1.f + __expf(-x));
    default: return x;
  }
}
__device__ __forceinline__ float act_grad_from_output(float y, int act) {
  switch (act) {
    case IBM_ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case IBM_ACT_SIGMOID: return y * (1.f - y);
    case IBM_ACT_TANH: return 1.f - y * y;
    case IBM_ACT_ELU: return y > 0.f ? 1.f : y + 1.f;
    default: return 1.f;
  }
}
__device__ __forceinline__ float act_grad_from_input(float x, int act) {
  switch (act) {
    case IBM_ACT_RELU: return x > 0.f ? 1.f : 0.f;
    case IBM_ACT_SIGMOID: { float s = 1.f / (1.f + __expf(-x)); return s * (1.f - s); }
    case IBM_ACT_TANH: { float t = tanhf(x); return 1.f - t * t; }
    case IBM_ACT_ELU: return x > 0.f ? 1.f : __expf(x);
    case IBM_ACT_SILU: { float s = 1.f / (1.f + __expf(-x)); return s * (1.f + x * (1.f - s)); }
    default: return 1.f;
  }
}

// Philox4x32-10 counter RNG + Box-Muller (self-contained; no cuRAND dependency)
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint64_t offset, uint64_t idx) {
  uint64_t c = offset;
  uint4 r = philox4x32_10(make_uint4((uint32_t)idx, (uint32_t)(idx >> 32), (uint32_t)c, (uint32_t)(c >> 32)),
                          make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float k = 2.3283064365386963e-10f;  // 2^-32
  float u0 = (r.x + 0.5f) * k, u1 = (r.y + 0.5f) * k, u2 = (r.z + 0.5f) * k, u3 = (r.w + 0.5f) * k;
  float r0 = sqrtf(-2.f * __logf(u0)), r1 = sqrtf(-2.f * __logf(u2));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * u1, &s0, &c0);
  __sincosf(6.283185307179586f * u3, &s1, &c1);
  return make_float4(r0 * c0, r0 * s0, r1 * c1, r1 * s1);
}

}  // namespace ibm
