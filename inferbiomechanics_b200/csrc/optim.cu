// Fused optimizer step over the flat fp32 parameter arena.  One launch updates parameters and
// optimizer state in place, applies the data-parallel 1/world_size gradient scale, and refreshes
// the bf16 shadow weights the tcgen05 GEMMs read.  HBM-bound (RMSprop: 12 B read + 10 B written
// per parameter; an exponential moving average of the weights adds 4 B read + 4 B written).
//
// Replaces torch.optim.{RMSprop,Adam,SGD,Adagrad,Adadelta,Adamax}(lr) with torch defaults as
// constructed at /root/reference/src/cli/train.py:183-197 and stepped at :284.
//
// Builder-owned additions: the global gradient norm and clip coefficient of
// torch.nn.utils.clip_grad_norm_ (grad_norm_kernel, one 4 B read per parameter, deterministic fp64
// reduction), and an optimizer instantiation that applies that coefficient and a warm-up / cosine
// learning-rate schedule, both read on the device so that captured steps replay.
#include "common.cuh"

namespace ibm {

constexpr int kThreads = 256;

struct OptArgs {
  float lr, gscale;
  float bc1, bc2_sqrt;   // Adam / Adamax bias corrections for this step
  const long long* step_dev;   // optional device-resident step count (CUDA-graph replays): the corrections are derived from it
  float* ema;            // EMA instantiation only: fp32 arena with the parameters' offsets
  double ema_decay;      // the EMA's decay cap
  float ema_w;           // 1 - d_n of this step (derived from step_dev when given)
  // SCHED instantiation only
  long long step;        // the 1-based step count when step_dev is null
  const float* clip;     // optional {total norm, clip coefficient} written by grad_norm_kernel
  int sched;             // 0 constant, 1 cosine after the warm-up
  long long warmup, total;
  double lr_ratio;       // lr_min / lr
};

// Learning-rate factor of the 1-based step n: linear warm-up n / W for n <= W, then 1 (constant) or
// r + (1 - r) * (1 + cos(pi * p)) / 2 with p = clamp((n - W) / (S - W), 0, 1) (cosine).
__host__ __device__ inline double lr_lambda(int sched, long long warmup, long long total, double r, double n) {
  if (warmup > 0 && n <= (double)warmup) return n / (double)warmup;
  if (sched == 0) return 1.0;
  const double p = fmin(fmax((n - (double)warmup) / (double)(total - warmup), 0.0), 1.0);
  return r + (1.0 - r) * (0.5 * (1.0 + cos(3.14159265358979323846 * p)));
}

// torch_ema's use_num_updates warm-up: d_n = min(decay, (1 + n) / (10 + n)), n = the 1-based step count, in double
__host__ __device__ inline float ema_weight(double decay, double n) {
  const double d = fmin(decay, (1.0 + n) / (10.0 + n));
  return (float)(1.0 - d);
}

template <int KIND>
__device__ __forceinline__ void opt_update(float& p, float g, float& s0, float& s1, const OptArgs& a) {
  if (KIND == 0) {            // RMSprop(alpha=.99, eps=1e-8)
    s0 = fmaf(0.99f, s0, 0.01f * g * g);               // 1-alpha evaluated in fp32 like torch's python float → 0.010000000000000009
    p -= a.lr * (g / (sqrtf(s0) + 1e-8f));
  } else if (KIND == 1) {     // Adam(.9, .999, 1e-8)
    s0 = s0 + (1.f - 0.9f) * (g - s0);
    s1 = fmaf(0.999f, s1, (1.f - 0.999f) * g * g);
    const float denom = sqrtf(s1) / a.bc2_sqrt + 1e-8f;
    p -= (a.lr / a.bc1) * (s0 / denom);
  } else if (KIND == 2) {     // SGD
    p -= a.lr * g;
  } else if (KIND == 3) {     // Adagrad(eps=1e-10)
    s0 = fmaf(g, g, s0);
    p -= a.lr * (g / (sqrtf(s0) + 1e-10f));
  } else if (KIND == 4) {     // Adadelta(rho=.9, eps=1e-6)
    s0 = fmaf(0.9f, s0, (1.f - 0.9f) * g * g);
    const float delta = sqrtf(s1 + 1e-6f) / sqrtf(s0 + 1e-6f) * g;
    s1 = fmaf(0.9f, s1, (1.f - 0.9f) * delta * delta);
    p -= a.lr * delta;
  } else {                    // Adamax(.9, .999, 1e-8)
    s0 = s0 + (1.f - 0.9f) * (g - s0);
    s1 = fmaxf(0.999f * s1, fabsf(g) + 1e-8f);
    p -= (a.lr / a.bc1) * (s0 / s1);
  }
}

__device__ __forceinline__ float ema_update(float e, float p, float w) { return fmaf(w, p - e, e); }

// the averaged gradient times the clip coefficient, torch's order (clip_grad_norm_ then step); __fmul_rn is never
// contracted into a later add, so a coefficient of exactly 1 leaves the gradient, and the update, unchanged
template <bool SCHED>
__device__ __forceinline__ float clipped(float g, float cf) {
  if constexpr (SCHED) return __fmul_rn(g, cf);
  return g;
}

template <int KIND, bool EMA, bool SCHED>
__global__ void __launch_bounds__(kThreads)
optimizer_kernel(float* __restrict__ param, const float* __restrict__ grad, float* __restrict__ st0,
                 float* __restrict__ st1, __nv_bfloat16* __restrict__ pb, long long n, OptArgs a) {
  if constexpr (KIND == 1 || KIND == 5) {
    if (a.step_dev != nullptr) {
      // one thread per block evaluates the two powers in double precision (as the host does for a by-value step)
      __shared__ float s_bc[2];
      if (threadIdx.x == 0) {
        const double st = (double)__ldg(a.step_dev);
        s_bc[0] = (float)(1.0 - pow(0.9, st));
        s_bc[1] = (float)sqrt(1.0 - pow(0.999, st));
      }
      __syncthreads();
      a.bc1 = s_bc[0];
      a.bc2_sqrt = s_bc[1];
    }
  }
  if constexpr (EMA) {
    if (a.step_dev != nullptr) {
      __shared__ float s_w;
      if (threadIdx.x == 0) s_w = ema_weight(a.ema_decay, (double)__ldg(a.step_dev));
      __syncthreads();
      a.ema_w = s_w;
    }
  }
  float cf = 1.f;         // clip coefficient (SCHED only)
  if constexpr (SCHED) {
    // thread 0 evaluates the schedule in double from the step this launch performs, and reads the clip coefficient
    __shared__ float s_sched[2];
    if (threadIdx.x == 0) {
      const double st = a.step_dev != nullptr ? (double)__ldg(a.step_dev) : (double)a.step;
      s_sched[0] = (float)((double)a.lr * lr_lambda(a.sched, a.warmup, a.total, a.lr_ratio, st));
      s_sched[1] = a.clip != nullptr ? a.clip[1] : 1.f;
    }
    __syncthreads();
    a.lr = s_sched[0];
    cf = s_sched[1];
  }
  float* __restrict__ ema = a.ema;
  const long long n4 = n >> 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  constexpr bool kS0 = KIND != 2, kS1 = (KIND == 1 || KIND == 4 || KIND == 5);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 p = *reinterpret_cast<const float4*>(param + 4 * i);
    float4 g = ld_stream_f4(grad + 4 * i);
    float4 s0 = kS0 ? *reinterpret_cast<const float4*>(st0 + 4 * i) : make_float4(0, 0, 0, 0);
    float4 s1 = kS1 ? *reinterpret_cast<const float4*>(st1 + 4 * i) : make_float4(0, 0, 0, 0);
    opt_update<KIND>(p.x, clipped<SCHED>(g.x * a.gscale, cf), s0.x, s1.x, a);
    opt_update<KIND>(p.y, clipped<SCHED>(g.y * a.gscale, cf), s0.y, s1.y, a);
    opt_update<KIND>(p.z, clipped<SCHED>(g.z * a.gscale, cf), s0.z, s1.z, a);
    opt_update<KIND>(p.w, clipped<SCHED>(g.w * a.gscale, cf), s0.w, s1.w, a);
    *reinterpret_cast<float4*>(param + 4 * i) = p;
    if (kS0) *reinterpret_cast<float4*>(st0 + 4 * i) = s0;
    if (kS1) *reinterpret_cast<float4*>(st1 + 4 * i) = s1;
    if (pb) *reinterpret_cast<uint2*>(pb + 4 * i) = make_uint2(pack_bf16x2(p.x, p.y), pack_bf16x2(p.z, p.w));
    if constexpr (EMA) {
      float4 e = *reinterpret_cast<const float4*>(ema + 4 * i);
      e = make_float4(ema_update(e.x, p.x, a.ema_w), ema_update(e.y, p.y, a.ema_w), ema_update(e.z, p.z, a.ema_w),
                      ema_update(e.w, p.w, a.ema_w));
      *reinterpret_cast<float4*>(ema + 4 * i) = e;
    }
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float p = param[i], s0 = kS0 ? st0[i] : 0.f, s1 = kS1 ? st1[i] : 0.f;
    opt_update<KIND>(p, clipped<SCHED>(grad[i] * a.gscale, cf), s0, s1, a);
    param[i] = p;
    if (kS0) st0[i] = s0;
    if (kS1) st1[i] = s1;
    if (pb) pb[i] = __float2bfloat16_rn(p);
    if constexpr (EMA) ema[i] = ema_update(ema[i], p, a.ema_w);
  }
}

template <bool EMA, bool SCHED>
static void launch_optimizer(int32_t kind, int grid, cudaStream_t s, float* param, const float* grad, float* state0, float* state1,
                             __nv_bfloat16* pb, long long n, const OptArgs& a) {
  switch (kind) {
    case 0: optimizer_kernel<0, EMA, SCHED><<<grid, kThreads, 0, s>>>(param, grad, state0, state1, pb, n, a); break;
    case 1: optimizer_kernel<1, EMA, SCHED><<<grid, kThreads, 0, s>>>(param, grad, state0, state1, pb, n, a); break;
    case 2: optimizer_kernel<2, EMA, SCHED><<<grid, kThreads, 0, s>>>(param, grad, state0, state1, pb, n, a); break;
    case 3: optimizer_kernel<3, EMA, SCHED><<<grid, kThreads, 0, s>>>(param, grad, state0, state1, pb, n, a); break;
    case 4: optimizer_kernel<4, EMA, SCHED><<<grid, kThreads, 0, s>>>(param, grad, state0, state1, pb, n, a); break;
    default: optimizer_kernel<5, EMA, SCHED><<<grid, kThreads, 0, s>>>(param, grad, state0, state1, pb, n, a); break;
  }
}

// ---- global gradient norm (torch.nn.utils.clip_grad_norm_) ------------------------------------------------------------
constexpr int kNormThreads = 512;
constexpr int kNormMaxBlocks = 1024;    // size of the caller's partials buffer (ibm_b200.h)

// fixed-order fp64 sum over the block (warp shuffles, then warp 0 over the warp sums); the result is valid in thread 0
__device__ __forceinline__ double block_sum_f64(double v) {
  __shared__ double s_w[kNormThreads / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) s_w[w] = v;
  __syncthreads();
  v = l < kNormThreads / 32 ? s_w[l] : 0.0;
  if (w == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  }
  return v;
}

// Sum of squares over the arena in fp64 (per thread, per block), one partial per block; the last block to finish sums the
// partials in a fixed partition and order, so the result depends on the grid only, never on the blocks' timing.
__global__ void __launch_bounds__(kNormThreads)
grad_norm_kernel(const float* __restrict__ grad, long long n, float gscale, float max_norm, float* __restrict__ out,
                 double* __restrict__ partials, unsigned int* __restrict__ counter, double* __restrict__ record) {
  double acc = 0.0;
  const long long n4 = n >> 2;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 g = ld_stream_f4(grad + 4 * i);
    acc = fma((double)g.x, (double)g.x, acc);
    acc = fma((double)g.y, (double)g.y, acc);
    acc = fma((double)g.z, (double)g.z, acc);
    acc = fma((double)g.w, (double)g.w, acc);
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const double g = (double)grad[i];
    acc = fma(g, g, acc);
  }
  acc = block_sum_f64(acc);
  __shared__ bool is_last;
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = acc;
    __threadfence();
    is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  double v = 0.0;
  for (unsigned int j = threadIdx.x; j < gridDim.x; j += blockDim.x) v += __ldcg(partials + j);
  v = block_sum_f64(v);
  if (threadIdx.x == 0) {
    // clip_grad_norm_ in fp32 from the fp32-rounded total: coef = min(1, max_norm / (total + 1e-6)); a NaN total gives a
    // NaN coefficient, as torch's clamp does (fminf would return 1)
    const float total = (float)(sqrt(v) * (double)gscale);
    const float c = max_norm / (total + 1e-6f);
    const float coef = c > 1.f ? 1.f : c;
    out[0] = total;
    out[1] = coef;
    if (record != nullptr) {
      record[0] += (double)total;
      record[1] += 1.0;
      record[2] += coef < 1.f ? 1.0 : 0.0;
    }
    *counter = 0u;
  }
}

}  // namespace ibm

struct SchedArgs {
  const float* clip;
  int32_t sched;
  int64_t warmup, total;
  float lr_min;
};

static int optimizer_step_impl(int32_t kind, float* param, const float* grad, float* state0, float* state1, void* param_bf16,
                               float* ema, int64_t n, float lr, float grad_scale, float ema_decay, int64_t step,
                               const int64_t* step_dev, void* stream, const SchedArgs* sa = nullptr);

extern "C" int ibm_optimizer_step(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                                  void* param_bf16, int64_t n, float lr, float grad_scale, int64_t step, void* stream) {
  return optimizer_step_impl(kind, param, grad, state0, state1, param_bf16, nullptr, n, lr, grad_scale, 0.f, step, nullptr, stream);
}

extern "C" int ibm_optimizer_step_dev(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                                      void* param_bf16, int64_t n, float lr, float grad_scale, const int64_t* step_dev, void* stream) {
  if (step_dev == nullptr) {
    ibm::set_error("optimizer_step_dev: null step counter");
    return IBM_E_ARG;
  }
  return optimizer_step_impl(kind, param, grad, state0, state1, param_bf16, nullptr, n, lr, grad_scale, 0.f, 1, step_dev, stream);
}

extern "C" int ibm_optimizer_step_ema(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                                      void* param_bf16, float* ema, int64_t n, float lr, float grad_scale, float ema_decay,
                                      int64_t step, const int64_t* step_dev, void* stream) {
  if (ema == nullptr) {
    ibm::set_error("optimizer_step_ema: null EMA arena");
    return IBM_E_ARG;
  }
  return optimizer_step_impl(kind, param, grad, state0, state1, param_bf16, ema, n, lr, grad_scale, ema_decay,
                             step_dev ? 1 : step, step_dev, stream);
}

extern "C" int ibm_optimizer_step_sched(int32_t kind, float* param, const float* grad, float* state0, float* state1,
                                        void* param_bf16, float* ema, int64_t n, float lr, float grad_scale, float ema_decay,
                                        int64_t step, const int64_t* step_dev, const float* clip, int32_t sched,
                                        int64_t warmup_steps, int64_t total_steps, float lr_min, void* stream) {
  IBM_CHECK_ARG(sched == 0 || sched == 1, "optimizer_step_sched: unknown schedule %d (0 constant, 1 cosine)", (int)sched);
  IBM_CHECK_ARG(warmup_steps >= 0, "optimizer_step_sched: warmup_steps must be >= 0, got %lld", (long long)warmup_steps);
  IBM_CHECK_ARG(sched == 0 || total_steps > warmup_steps,
                "optimizer_step_sched: the cosine schedule needs total_steps > warmup_steps, got %lld <= %lld",
                (long long)total_steps, (long long)warmup_steps);
  IBM_CHECK_ARG(lr_min >= 0.f && lr_min <= lr, "optimizer_step_sched: lr_min must be in [0, lr], got %g (lr %g)", (double)lr_min,
                (double)lr);
  IBM_CHECK_ARG(reinterpret_cast<uintptr_t>(clip) % 4 == 0, "optimizer_step_sched: misaligned clip record");
  const SchedArgs sa{clip, sched, warmup_steps, total_steps, lr_min};
  return optimizer_step_impl(kind, param, grad, state0, state1, param_bf16, ema, n, lr, grad_scale, ema_decay,
                             step_dev ? 1 : step, step_dev, stream, &sa);
}

extern "C" int ibm_grad_clip_coef(const float* grad, int64_t n, float grad_scale, float max_norm, float* out, double* partials,
                                  uint32_t* counter, double* record, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(grad && out && partials && counter && n > 0, "grad_clip_coef: bad argument");
  IBM_CHECK_ARG(aligned16(grad), "grad_clip_coef: the gradient arena must be 16-byte aligned");
  IBM_CHECK_ARG(max_norm > 0.f, "grad_clip_coef: max_norm must be > 0, got %g", (double)max_norm);
  long long need = ceil_div(n / 4 + 1, kNormThreads);
  long long cap = (long long)sm_count() * 4;
  if (cap > kNormMaxBlocks) cap = kNormMaxBlocks;
  const int grid = (int)(need < cap ? need : cap);
  grad_norm_kernel<<<grid, kNormThreads, 0, static_cast<cudaStream_t>(stream)>>>(grad, n, grad_scale, max_norm, out, partials,
                                                                                  counter, record);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

static int optimizer_step_impl(int32_t kind, float* param, const float* grad, float* state0, float* state1, void* param_bf16,
                               float* ema, int64_t n, float lr, float grad_scale, float ema_decay, int64_t step,
                               const int64_t* step_dev, void* stream, const SchedArgs* sa) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(kind >= 0 && kind <= 5, "optimizer_step: unknown optimizer kind %d", kind);
  IBM_CHECK_ARG(param && grad && n > 0 && step >= 1, "optimizer_step: bad argument");
  IBM_CHECK_ARG(kind == 2 || state0, "optimizer_step: state0 required");
  IBM_CHECK_ARG(!(kind == 1 || kind == 4 || kind == 5) || state1, "optimizer_step: state1 required");
  IBM_CHECK_ARG(aligned16(param) && aligned16(grad) && (!state0 || aligned16(state0)) && (!state1 || aligned16(state1)) &&
                    (!ema || aligned16(ema)) && (!param_bf16 || (reinterpret_cast<uintptr_t>(param_bf16) % 8 == 0)),
                "optimizer_step: arenas must be 16-byte aligned");
  IBM_CHECK_ARG(!ema || (ema_decay > 0.f && ema_decay < 1.f), "optimizer_step: EMA decay must be in (0, 1), got %g",
                (double)ema_decay);
  OptArgs a;
  a.lr = lr;
  a.gscale = grad_scale;
  a.bc1 = (float)(1.0 - pow(0.9, (double)step));
  a.bc2_sqrt = (float)sqrt(1.0 - pow(0.999, (double)step));
  a.step_dev = reinterpret_cast<const long long*>(step_dev);
  a.ema = ema;
  a.ema_decay = (double)ema_decay;
  a.ema_w = ema_weight(a.ema_decay, (double)step);
  a.step = step;
  a.clip = sa ? sa->clip : nullptr;
  a.sched = sa ? sa->sched : 0;
  a.warmup = sa ? sa->warmup : 0;
  a.total = sa ? sa->total : 0;
  a.lr_ratio = sa && lr > 0.f ? (double)sa->lr_min / (double)lr : 0.0;
  long long need = ceil_div(n / 4 + 1, kThreads);
  long long cap = (long long)sm_count() * 16;
  const int grid = (int)(need < cap ? need : cap);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  auto* pb = static_cast<__nv_bfloat16*>(param_bf16);
  if (sa != nullptr) {
    if (ema)
      launch_optimizer<true, true>(kind, grid, s, param, grad, state0, state1, pb, n, a);
    else
      launch_optimizer<false, true>(kind, grid, s, param, grad, state0, state1, pb, n, a);
  } else if (ema) {
    launch_optimizer<true, false>(kind, grid, s, param, grad, state0, state1, pb, n, a);
  } else {
    launch_optimizer<false, false>(kind, grid, s, param, grad, state0, state1, pb, n, a);
  }
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}
