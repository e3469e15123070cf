// DDPM elementwise kernels: q_sample, posterior (reverse) step, sinusoidal timestep embedding,
// and the time/position embedding add.  Builder-owned spec (DESIGN.md D-1) — the reference has no
// diffusion code (only /root/reference/src/.gitignore:10).  All HBM-bound, 16-byte vectorised:
//   q_sample        reads x0, eps (fp32), writes x_t fp32 (+ bf16 scatter)  = 360*F B/window
//   posterior step  reads x_t, x0_hat, z, writes x_{t-1}                    = 480*F B/window/step
#include "common.cuh"

namespace ibm {

constexpr int kThreads = 256;

// ---- q_sample --------------------------------------------------------------------------------
// Vector path: per_win % 4 == 0 so the four lanes of a float4 share one window (one table lookup).
template <bool kVec>
__global__ void __launch_bounds__(kThreads)
q_sample_kernel(const float* __restrict__ x0, const float* __restrict__ eps, const int32_t* __restrict__ t,
                const float* __restrict__ sa, const float* __restrict__ sb, long long n, long long per_win,
                float* __restrict__ xt, __nv_bfloat16* __restrict__ xt_bf16, long long bf16_ld,
                uint64_t seed, uint64_t offset, float* __restrict__ eps_out) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  if (kVec) {
    const long long n4 = n >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
      const long long e = i << 2;
      const long long w = e / per_win;
      const int tt = __ldg(t + w);
      const float a = __ldg(sa + tt), b = __ldg(sb + tt);
      float4 x = ld_stream_f4(x0 + e);
      float4 z = eps ? ld_stream_f4(eps + e) : philox_normal4(seed, offset, (uint64_t)i);
      if (!eps && eps_out) st_stream_f4(eps_out + e, z);
      float4 r = make_float4(fmaf(a, x.x, b * z.x), fmaf(a, x.y, b * z.y), fmaf(a, x.z, b * z.z), fmaf(a, x.w, b * z.w));
      if (xt) st_stream_f4(xt + e, r);
      if (xt_bf16) {
        // rows of 30 channels: pairs never straddle a row because 30 is even
        long long m0 = e / 30, c0 = e - m0 * 30;
        *reinterpret_cast<uint32_t*>(xt_bf16 + m0 * bf16_ld + c0) = pack_bf16x2(r.x, r.y);
        long long e1 = e + 2, m1 = e1 / 30, c1 = e1 - m1 * 30;
        *reinterpret_cast<uint32_t*>(xt_bf16 + m1 * bf16_ld + c1) = pack_bf16x2(r.z, r.w);
      }
    }
  } else {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
      const long long w = e / per_win;
      const int tt = __ldg(t + w);
      const float a = __ldg(sa + tt), b = __ldg(sb + tt);
      float z;
      if (eps) z = __ldg(eps + e);
      else {
        float4 z4 = philox_normal4(seed, offset, (uint64_t)(e >> 2));
        int k = (int)(e & 3);
        z = k == 0 ? z4.x : k == 1 ? z4.y : k == 2 ? z4.z : z4.w;
        if (eps_out) eps_out[e] = z;
      }
      float r = fmaf(a, __ldg(x0 + e), b * z);
      if (xt) xt[e] = r;
      if (xt_bf16) {
        long long m = e / 30, c = e - m * 30;
        xt_bf16[m * bf16_ld + c] = __float2bfloat16_rn(r);
      }
    }
  }
}

// ---- posterior step --------------------------------------------------------------------------
// One float2 per thread-iteration: 30 is even so a pair never straddles a row; x0_hat has its own
// leading dimension (the head GEMM writes 32-float rows).  kSucc: the next timestep is t_succ[t]
// (a respaced DDIM sequence) instead of t-1; the instantiation without it is the DDPM chain.  kGuided: x0h holds 2M
// rows, conditional then unconditional, combined as u + s (c - u) (classifier-free guidance); the bf16 rows go to both
// halves of the concat buffer.  gscale follows the parameters of the unguided instantiations so they keep their parameter
// offsets.  kKnown (inpainting): after the guided combination, channel c of row m takes known[m, c] instead of the prediction
// where bit c of kmask[m] is set (bits 30-31 are ignored); a select, so a NaN in an unknown entry of `known` never reaches
// the output.  known / kmask come after gscale for the same reason.  kMulti (DPM-Solver++(2M), always with kSucc): no noise
// term; the update adds coef_prev[t] x0_prev (the previous step's prediction, read only when coef_prev[t] != 0, so the
// uninitialised buffer of the first step is never read) and stores this step's prediction, after the guided combination and
// the known-entry select, into x0_prev in place.  coef_prev / x0_prev come last for the same reason.
template <bool kSucc, bool kGuided, bool kKnown, bool kMulti>
__global__ void __launch_bounds__(kThreads)
posterior_kernel(const float* __restrict__ x0h, long long x0_ld, const float* __restrict__ xt,
                 const float* __restrict__ z, const int32_t* __restrict__ t_dev, const float* __restrict__ c1t,
                 const float* __restrict__ c2t, const float* __restrict__ sig, long long M,
                 float* __restrict__ xprev, __nv_bfloat16* __restrict__ xp_bf16, long long bf16_ld,
                 uint64_t seed, uint64_t offset, int32_t* __restrict__ t_next,
                 const int32_t* __restrict__ t_succ, float gscale, const float* __restrict__ known,
                 const int32_t* __restrict__ kmask, const float* __restrict__ coef_prev, float* __restrict__ x0_prev) {
  const int tt = __ldg(t_dev);
  const float c1 = __ldg(c1t + tt), c2 = __ldg(c2t + tt);
  const float s = !kMulti && tt > 0 ? __ldg(sig + tt) : 0.f;
  const float cp = kMulti ? __ldg(coef_prev + tt) : 0.f;
  const long long npair = M * 15;
  const long long stride = (long long)gridDim.x * blockDim.x;
#pragma unroll (kKnown ? 1 : 2)   // unrolled twice, the kKnown loop spills 8 bytes (CUDA 12.9)
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < npair; p += stride) {
    const long long m = p / 15, c = (p - m * 15) * 2;
    float2 a = *reinterpret_cast<const float2*>(x0h + m * x0_ld + c);
    if (kGuided) {
      const float2 u = *reinterpret_cast<const float2*>(x0h + (M + m) * x0_ld + c);
      a.x = fmaf(gscale, a.x - u.x, u.x);
      a.y = fmaf(gscale, a.y - u.y, u.y);
    }
    if (kKnown) {
      const uint32_t w = (uint32_t)__ldg(kmask + m) >> c;
      if (w & 3u) {
        const float2 y = __ldg(reinterpret_cast<const float2*>(known + 2 * p));
        if (w & 1u) a.x = y.x;
        if (w & 2u) a.y = y.y;
      }
    }
    const float2 x = *reinterpret_cast<const float2*>(xt + 2 * p);
    float2 r;
    if (kMulti) {
      r.x = fmaf(c1, a.x, c2 * x.x);
      r.y = fmaf(c1, a.y, c2 * x.y);
      float2* const q = reinterpret_cast<float2*>(x0_prev + 2 * p);
      if (cp != 0.f) {                      // tt is uniform per launch, so is this branch
        const float2 d = *q;
        r.x = fmaf(cp, d.x, r.x);
        r.y = fmaf(cp, d.y, r.y);
      }
      *q = a;
    } else {
      float2 n;
      if (z) n = *reinterpret_cast<const float2*>(z + 2 * p);
      else {
        // counter offset includes the step so a CUDA-graph replay (frozen arguments) still draws fresh noise
        float4 z4 = philox_normal4(seed, offset + (uint64_t)tt, (uint64_t)(p >> 1));
        n = (p & 1) ? make_float2(z4.z, z4.w) : make_float2(z4.x, z4.y);
      }
      r.x = fmaf(c1, a.x, c2 * x.x);
      r.y = fmaf(c1, a.y, c2 * x.y);
      if (tt > 0) { r.x = fmaf(s, n.x, r.x); r.y = fmaf(s, n.y, r.y); }
    }
    if (xprev) *reinterpret_cast<float2*>(xprev + 2 * p) = r;
    if (xp_bf16) {
      const uint32_t v = pack_bf16x2(r.x, r.y);
      *reinterpret_cast<uint32_t*>(xp_bf16 + m * bf16_ld + c) = v;
      if (kGuided) *reinterpret_cast<uint32_t*>(xp_bf16 + (M + m) * bf16_ld + c) = v;
    }
  }
  if (t_next && blockIdx.x == 0 && threadIdx.x == 0) *t_next = kSucc ? __ldg(t_succ + tt) : tt - 1;
}

// ---- per-window condition dropout (classifier-free guidance training) -------------------------------------------------
// One block per window (grid-stride): every thread derives the window's keep bit from word 0 of Philox draw b, so a kept
// window costs one draw and no memory traffic.  A dropped window's F rows are cleared in 8-column groups: a group that lies
// inside [col0, col0 + ncols) is one 16-byte store when the rows are 16-byte aligned (kVec), a group cut by the range edge
// is stored element by element so neighbouring columns (x_t, pad) are never written.
template <bool kVec>
__global__ void __launch_bounds__(kThreads)
cond_dropout_kernel(__nv_bfloat16* __restrict__ xc, long long ld, long long B, int F, int col0, int ncols,
                    uint32_t thresh, int drop_all, uint64_t seed, uint64_t offset, uint8_t* __restrict__ keep_out) {
  const int g0 = col0 >> 3, g1 = (col0 + ncols - 1) >> 3, col1 = col0 + ncols;
  const int ng = g1 - g0 + 1;
  const long long items = (long long)F * ng;
  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    bool drop = true;
    if (!drop_all) {
      const uint4 r = philox4x32_10(make_uint4((uint32_t)b, (uint32_t)(b >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)),
                                    make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
      drop = r.x < thresh;
    }
    if (keep_out && threadIdx.x == 0) keep_out[b] = drop ? 0 : 1;
    if (!drop) continue;
    __nv_bfloat16* base = xc + b * F * ld;
    for (long long i = threadIdx.x; i < items; i += blockDim.x) {
      const long long f = i / ng;
      const int c = (g0 + (int)(i - f * ng)) << 3;
      __nv_bfloat16* row = base + f * ld;
      if (kVec && c >= col0 && c + 8 <= col1) {
        *reinterpret_cast<uint4*>(row + c) = make_uint4(0u, 0u, 0u, 0u);
      } else {
        const int lo = c > col0 ? c : col0, hi = c + 8 < col1 ? c + 8 : col1;
        for (int k = lo; k < hi; ++k) row[k] = __ushort_as_bfloat16((unsigned short)0);
      }
    }
  }
}

// ---- sinusoidal timestep embedding -----------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
timestep_embed_kernel(const int32_t* __restrict__ t, int t_is_scalar, long long B, int dim,
                      __nv_bfloat16* __restrict__ out) {
  const int half = dim >> 1;
  const long long n = B * half;
  const float neg_log = -9.210340371976184f / (float)half;   // -ln(10000)/half
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / half;
    const int k = (int)(i - b * half);
    const float tv = (float)__ldg(t + (t_is_scalar ? 0 : b));
    const float ang = tv * expf(neg_log * (float)k);
    float s, c;
    sincosf(ang, &s, &c);
    out[b * dim + k] = __float2bfloat16_rn(s);
    out[b * dim + half + k] = __float2bfloat16_rn(c);
  }
}

// ---- h += temb[b] + pos[f] -------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
add_time_pos_kernel(__nv_bfloat16* __restrict__ h, long long ld, const __nv_bfloat16* __restrict__ temb,
                    long long temb_ld, const float* __restrict__ pos, long long M, int F, int d,
                    const int* __restrict__ t_row) {
  const int d8 = d >> 3;
  const long long n = M * d8;
  const long long fixed_row = t_row ? (long long)__ldg(t_row) : -1;   // one table row for every window (sampling)
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / d8;
    const int c = (int)(i - m * d8) * 8;
    const long long b = m / F;
    const int f = (int)(m - b * F);
    uint4 hv = *reinterpret_cast<const uint4*>(h + m * ld + c);
    const uint4 tv = __ldg(reinterpret_cast<const uint4*>(temb + (fixed_row >= 0 ? fixed_row : b) * temb_ld + c));
    const float4 p0 = __ldg(reinterpret_cast<const float4*>(pos + (long long)f * d + c));
    const float4 p1 = __ldg(reinterpret_cast<const float4*>(pos + (long long)f * d + c + 4));
    float2 a, e;
    a = unpack_bf16x2(hv.x); e = unpack_bf16x2(tv.x); hv.x = pack_bf16x2(a.x + e.x + p0.x, a.y + e.y + p0.y);
    a = unpack_bf16x2(hv.y); e = unpack_bf16x2(tv.y); hv.y = pack_bf16x2(a.x + e.x + p0.z, a.y + e.y + p0.w);
    a = unpack_bf16x2(hv.z); e = unpack_bf16x2(tv.z); hv.z = pack_bf16x2(a.x + e.x + p1.x, a.y + e.y + p1.y);
    a = unpack_bf16x2(hv.w); e = unpack_bf16x2(tv.w); hv.w = pack_bf16x2(a.x + e.x + p1.z, a.y + e.y + p1.w);
    *reinterpret_cast<uint4*>(h + m * ld + c) = hv;
  }
}

// backward: block = (window group, 64-column slab); thread (r, cpair) ; dtemb per window, dpos via
// register accumulation over the block's windows then one fp32 atomic per (f, col) per block.
constexpr int kTpWin = 8;   // windows per block
__global__ void __launch_bounds__(kThreads)
add_time_pos_bwd_kernel(const __nv_bfloat16* __restrict__ dh, long long ld, __nv_bfloat16* __restrict__ dtemb,
                        long long temb_ld, float* __restrict__ dpos, long long B, int F, int d) {
  // thread layout: 32 column-pairs (64 cols) x 8 frame lanes
  const int cp = threadIdx.x & 31, fl = threadIdx.x >> 5;
  const int col = blockIdx.y * 64 + cp * 2;
  __shared__ float2 tsum[8][32];
  if (col >= d) return;   // d is a multiple of 8 and slabs are 64 wide: whole warps exit together only if d%64==0
  const long long b0 = (long long)blockIdx.x * kTpWin;
  for (int f0 = 0; f0 < F; f0 += 8) {
    const int f = f0 + fl;
    float2 pacc = make_float2(0.f, 0.f);
    if (f < F) {
      for (int w = 0; w < kTpWin; ++w) {
        const long long b = b0 + w;
        if (b >= B) break;
        float2 v = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(dh + (b * F + f) * ld + col));
        pacc.x += v.x; pacc.y += v.y;
      }
      atomicAdd(dpos + (long long)f * d + col, pacc.x);
      atomicAdd(dpos + (long long)f * d + col + 1, pacc.y);
    }
  }
  // dtemb[b, col] = sum_f dh[b, f, col]
  for (int w = 0; w < kTpWin; ++w) {
    const long long b = b0 + w;
    if (b >= B) break;                 // uniform across the block
    float2 acc = make_float2(0.f, 0.f);
    for (int f = fl; f < F; f += 8) {
      float2 v = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(dh + (b * F + f) * ld + col));
      acc.x += v.x; acc.y += v.y;
    }
    tsum[fl][cp] = acc;
    __syncthreads();
    if (fl == 0) {
      float2 s = tsum[0][cp];
#pragma unroll
      for (int k = 1; k < 8; ++k) { s.x += tsum[k][cp].x; s.y += tsum[k][cp].y; }
      *reinterpret_cast<uint32_t*>(dtemb + b * temb_ld + col) = pack_bf16x2(s.x, s.y);
    }
    __syncthreads();
  }
}

// One pass over dh for all three reductions of the stem's backward: dtemb[b] = sum_f dh[b, f] (bf16, per window), dpos[f] +=
// sum_b dh[b, f] (fp32) and, optionally, dbias += sum_{b, f} dh[b, f] (the in-projection's bias gradient, which used to cost a
// second full read of dh).  Block = kFusedW windows x 512 columns: thread (cc, fl) owns the 16-byte column chunk cc and the
// frames fl, fl + 4, ...; every thread has up to K independent 16-byte loads in flight per window, dpos partial sums live in
// registers over the block's windows and leave as vector atomics (8 KB x F per block instead of per window).
constexpr int kFusedW = 16;
template <int K>
__global__ void __launch_bounds__(kThreads)
add_time_pos_bwd_fused_kernel(const __nv_bfloat16* __restrict__ dh, long long ld, __nv_bfloat16* __restrict__ dtemb,
                              long long temb_ld, float* __restrict__ dpos, float* __restrict__ dbias, long long B, int F, int d) {
  const int cc = threadIdx.x & 63, fl = threadIdx.x >> 6;
  const int col = (blockIdx.y * 64 + cc) * 8;
  const bool active = col < d;
  __shared__ float red[4][64][9];
  float pacc[K][8], bacc[8];
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) pacc[k][j] = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) bacc[j] = 0.f;
  const long long b0 = (long long)blockIdx.x * kFusedW;
  for (int w = 0; w < kFusedW; ++w) {
    const long long b = b0 + w;
    if (b >= B) break;                                   // uniform across the block
    float tacc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) tacc[j] = 0.f;
    uint4 u[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int f = fl + 4 * k;
      u[k] = (active && f < F) ? ld_stream16(dh + (b * F + f) * ld + col) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float2 t;
      t = unpack_bf16x2(u[k].x); pacc[k][0] += t.x; pacc[k][1] += t.y; tacc[0] += t.x; tacc[1] += t.y;
      t = unpack_bf16x2(u[k].y); pacc[k][2] += t.x; pacc[k][3] += t.y; tacc[2] += t.x; tacc[3] += t.y;
      t = unpack_bf16x2(u[k].z); pacc[k][4] += t.x; pacc[k][5] += t.y; tacc[4] += t.x; tacc[5] += t.y;
      t = unpack_bf16x2(u[k].w); pacc[k][6] += t.x; pacc[k][7] += t.y; tacc[6] += t.x; tacc[7] += t.y;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) red[fl][cc][j] = tacc[j];
    __syncthreads();
    if (fl == 0 && active) {
      float s8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s8[j] = red[0][cc][j] + red[1][cc][j] + red[2][cc][j] + red[3][cc][j];
        bacc[j] += s8[j];
      }
      *reinterpret_cast<uint4*>(dtemb + b * temb_ld + col) =
          make_uint4(pack_bf16x2(s8[0], s8[1]), pack_bf16x2(s8[2], s8[3]), pack_bf16x2(s8[4], s8[5]), pack_bf16x2(s8[6], s8[7]));
    }
    __syncthreads();
  }
  if (!active) return;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int f = fl + 4 * k;
    if (f < F) {
      float4* p = reinterpret_cast<float4*>(dpos + (long long)f * d + col);
      atomicAdd(p, make_float4(pacc[k][0], pacc[k][1], pacc[k][2], pacc[k][3]));
      atomicAdd(p + 1, make_float4(pacc[k][4], pacc[k][5], pacc[k][6], pacc[k][7]));
    }
  }
  if (dbias != nullptr && fl == 0) {
    float4* p = reinterpret_cast<float4*>(dbias + col);
    atomicAdd(p, make_float4(bacc[0], bacc[1], bacc[2], bacc[3]));
    atomicAdd(p + 1, make_float4(bacc[4], bacc[5], bacc[6], bacc[7]));
  }
}

static int ew_grid(long long n_items) {
  long long need = ceil_div(n_items, kThreads);
  long long cap = (long long)sm_count() * 16;
  return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

}  // namespace ibm

extern "C" int ibm_q_sample(const float* x0, const float* eps, const int32_t* t, const float* sqrt_abar,
                            const float* sqrt_1m_abar, int64_t B, int64_t per_win, float* xt_f32, void* xt_bf16,
                            int64_t bf16_ld, uint64_t seed, uint64_t offset, float* eps_out, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x0 && t && sqrt_abar && sqrt_1m_abar, "q_sample: null argument");
  IBM_CHECK_ARG(B > 0 && per_win > 0, "q_sample: empty input");
  IBM_CHECK_ARG(xt_f32 || xt_bf16, "q_sample: no output requested");
  IBM_CHECK_ARG(!xt_bf16 || (per_win % 30 == 0 && bf16_ld % 2 == 0 && bf16_ld >= 30), "q_sample: bf16 scatter needs per_win %% 30 == 0 and even ld");
  const long long n = B * per_win;
  const bool vec = (per_win % 4 == 0) && aligned16(x0) && (!eps || aligned16(eps)) && (!xt_f32 || aligned16(xt_f32)) &&
                   (!eps_out || aligned16(eps_out));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* xb = static_cast<__nv_bfloat16*>(xt_bf16);
  if (vec)
    q_sample_kernel<true><<<ew_grid(n / 4), kThreads, 0, s>>>(x0, eps, t, sqrt_abar, sqrt_1m_abar, n, per_win, xt_f32, xb,
                                                            bf16_ld, seed, offset, eps_out);
  else
    q_sample_kernel<false><<<ew_grid(n), kThreads, 0, s>>>(x0, eps, t, sqrt_abar, sqrt_1m_abar, n, per_win, xt_f32, xb,
                                                         bf16_ld, seed, offset, eps_out);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_ddpm_posterior_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                                       const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                                       const float* sigma, int64_t M, float* x_prev, void* xprev_bf16, int64_t bf16_ld,
                                       uint64_t seed, uint64_t offset, int32_t* t_next_dev, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x0_hat && x_t && t_dev && coef_x0 && coef_xt && sigma, "posterior_step: null argument");
  IBM_CHECK_ARG(M > 0 && x0_ld >= 30 && x0_ld % 2 == 0, "posterior_step: bad shape (M=%lld ld=%lld)", (long long)M, (long long)x0_ld);
  IBM_CHECK_ARG(x_prev || xprev_bf16, "posterior_step: no output requested");
  IBM_CHECK_ARG(!xprev_bf16 || (bf16_ld % 2 == 0 && bf16_ld >= 30), "posterior_step: bf16 ld must be even");
  posterior_kernel<false, false, false, false><<<ew_grid(M * 15 / 2), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x0_hat, x0_ld, x_t, z, t_dev, coef_x0, coef_xt, sigma, M, x_prev, static_cast<__nv_bfloat16*>(xprev_bf16), bf16_ld,
      seed, offset, t_next_dev, nullptr, 0.f, nullptr, nullptr, nullptr, nullptr);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_ddpm_respaced_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                                      const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                                      const float* sigma, int64_t M, float* x_prev, void* xprev_bf16, int64_t bf16_ld,
                                      uint64_t seed, uint64_t offset, int32_t* t_next_dev, const int32_t* t_succ,
                                      void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x0_hat && x_t && t_dev && coef_x0 && coef_xt && sigma && t_succ, "respaced_step: null argument");
  IBM_CHECK_ARG(M > 0 && x0_ld >= 30 && x0_ld % 2 == 0, "respaced_step: bad shape (M=%lld ld=%lld)", (long long)M, (long long)x0_ld);
  IBM_CHECK_ARG(x_prev || xprev_bf16, "respaced_step: no output requested");
  IBM_CHECK_ARG(!xprev_bf16 || (bf16_ld % 2 == 0 && bf16_ld >= 30), "respaced_step: bf16 ld must be even");
  posterior_kernel<true, false, false, false><<<ew_grid(M * 15 / 2), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x0_hat, x0_ld, x_t, z, t_dev, coef_x0, coef_xt, sigma, M, x_prev, static_cast<__nv_bfloat16*>(xprev_bf16), bf16_ld,
      seed, offset, t_next_dev, t_succ, 0.f, nullptr, nullptr, nullptr, nullptr);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_ddpm_guided_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                                    const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                                    const float* sigma, int64_t M, float* x_prev, void* xprev_bf16, int64_t bf16_ld,
                                    uint64_t seed, uint64_t offset, int32_t* t_next_dev, const int32_t* t_succ,
                                    float guidance_scale, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x0_hat && x_t && t_dev && coef_x0 && coef_xt && sigma, "guided_step: null argument");
  IBM_CHECK_ARG(M > 0 && x0_ld >= 30 && x0_ld % 2 == 0, "guided_step: bad shape (M=%lld ld=%lld)", (long long)M, (long long)x0_ld);
  IBM_CHECK_ARG(x_prev || xprev_bf16, "guided_step: no output requested");
  IBM_CHECK_ARG(!xprev_bf16 || (bf16_ld % 2 == 0 && bf16_ld >= 30), "guided_step: bf16 ld must be even");
  IBM_CHECK_ARG(guidance_scale >= 0.f && guidance_scale <= 3.402823466e38f, "guided_step: guidance scale must be finite and >= 0, got %g",
                (double)guidance_scale);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  auto* xb = static_cast<__nv_bfloat16*>(xprev_bf16);
  if (t_succ)
    posterior_kernel<true, true, false, false><<<ew_grid(M * 15 / 2), kThreads, 0, s>>>(x0_hat, x0_ld, x_t, z, t_dev, coef_x0, coef_xt, sigma, M,
                                                                        x_prev, xb, bf16_ld, seed, offset, t_next_dev, t_succ,
                                                                        guidance_scale, nullptr, nullptr, nullptr, nullptr);
  else
    posterior_kernel<false, true, false, false><<<ew_grid(M * 15 / 2), kThreads, 0, s>>>(x0_hat, x0_ld, x_t, z, t_dev, coef_x0, coef_xt, sigma, M,
                                                                         x_prev, xb, bf16_ld, seed, offset, t_next_dev, nullptr,
                                                                         guidance_scale, nullptr, nullptr, nullptr, nullptr);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_ddpm_inpaint_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const float* z,
                                     const int32_t* t_dev, const float* coef_x0, const float* coef_xt,
                                     const float* sigma, int64_t M, float* x_prev, void* xprev_bf16, int64_t bf16_ld,
                                     uint64_t seed, uint64_t offset, int32_t* t_next_dev, const int32_t* t_succ,
                                     float guidance_scale, int32_t guided, const float* known, const int32_t* known_mask,
                                     void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x0_hat && x_t && t_dev && coef_x0 && coef_xt && sigma, "inpaint_step: null argument");
  IBM_CHECK_ARG(known && known_mask, "inpaint_step: null known values or known mask");
  IBM_CHECK_ARG(reinterpret_cast<uintptr_t>(known) % 8 == 0, "inpaint_step: known values must be 8-byte aligned");
  IBM_CHECK_ARG(M > 0 && x0_ld >= 30 && x0_ld % 2 == 0, "inpaint_step: bad shape (M=%lld ld=%lld)", (long long)M, (long long)x0_ld);
  IBM_CHECK_ARG(x_prev || xprev_bf16, "inpaint_step: no output requested");
  IBM_CHECK_ARG(!xprev_bf16 || (bf16_ld % 2 == 0 && bf16_ld >= 30), "inpaint_step: bf16 ld must be even");
  IBM_CHECK_ARG(guidance_scale >= 0.f && guidance_scale <= 3.402823466e38f, "inpaint_step: guidance scale must be finite and >= 0, got %g",
                (double)guidance_scale);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  auto* xb = static_cast<__nv_bfloat16*>(xprev_bf16);
  const int grid = ew_grid(M * 15 / 2);
#define IBM_INPAINT_LAUNCH(SUCC, GUIDED)                                                                                       \
  posterior_kernel<SUCC, GUIDED, true, false><<<grid, kThreads, 0, s>>>(x0_hat, x0_ld, x_t, z, t_dev, coef_x0, coef_xt, sigma, M,     \
                                                                 x_prev, xb, bf16_ld, seed, offset, t_next_dev, t_succ,         \
                                                                 guidance_scale, known, known_mask, nullptr, nullptr)
  if (t_succ) {
    if (guided) IBM_INPAINT_LAUNCH(true, true);
    else IBM_INPAINT_LAUNCH(true, false);
  } else {
    if (guided) IBM_INPAINT_LAUNCH(false, true);
    else IBM_INPAINT_LAUNCH(false, false);
  }
#undef IBM_INPAINT_LAUNCH
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_ddpm_multistep_step(const float* x0_hat, int64_t x0_ld, const float* x_t, const int32_t* t_dev,
                                       const float* coef_x0, const float* coef_xt, const float* coef_prev,
                                       const int32_t* t_succ, int64_t M, float* x0_prev, float* x_prev, void* xprev_bf16,
                                       int64_t bf16_ld, int32_t* t_next_dev, float guidance_scale, int32_t guided,
                                       const float* known, const int32_t* known_mask, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x0_hat && x_t && t_dev && coef_x0 && coef_xt && coef_prev && t_succ && x0_prev, "multistep_step: null argument");
  IBM_CHECK_ARG(reinterpret_cast<uintptr_t>(x0_prev) % 8 == 0, "multistep_step: x0_prev must be 8-byte aligned");
  IBM_CHECK_ARG(x0_prev != x_prev && x0_prev != x_t && x0_prev != x0_hat,
                "multistep_step: x0_prev must not be x_prev, x_t or x0_hat");
  IBM_CHECK_ARG(!known == !known_mask, "multistep_step: known values and known mask go together");
  IBM_CHECK_ARG(reinterpret_cast<uintptr_t>(known) % 8 == 0, "multistep_step: known values must be 8-byte aligned");
  IBM_CHECK_ARG(M > 0 && x0_ld >= 30 && x0_ld % 2 == 0, "multistep_step: bad shape (M=%lld ld=%lld)", (long long)M, (long long)x0_ld);
  IBM_CHECK_ARG(x_prev || xprev_bf16, "multistep_step: no output requested");
  IBM_CHECK_ARG(!xprev_bf16 || (bf16_ld % 2 == 0 && bf16_ld >= 30), "multistep_step: bf16 ld must be even");
  IBM_CHECK_ARG(guidance_scale >= 0.f && guidance_scale <= 3.402823466e38f, "multistep_step: guidance scale must be finite and >= 0, got %g",
                (double)guidance_scale);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  auto* xb = static_cast<__nv_bfloat16*>(xprev_bf16);
  const int grid = ew_grid(M * 15 / 2);
#define IBM_MULTISTEP_LAUNCH(GUIDED, KNOWN)                                                                                    \
  posterior_kernel<true, GUIDED, KNOWN, true><<<grid, kThreads, 0, s>>>(x0_hat, x0_ld, x_t, nullptr, t_dev, coef_x0, coef_xt,  \
                                                                        nullptr, M, x_prev, xb, bf16_ld, 0, 0, t_next_dev,      \
                                                                        t_succ, guidance_scale, known, known_mask, coef_prev,  \
                                                                        x0_prev)
  if (known) {
    if (guided) IBM_MULTISTEP_LAUNCH(true, true);
    else IBM_MULTISTEP_LAUNCH(false, true);
  } else {
    if (guided) IBM_MULTISTEP_LAUNCH(true, false);
    else IBM_MULTISTEP_LAUNCH(false, false);
  }
#undef IBM_MULTISTEP_LAUNCH
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_cond_dropout(void* xc_bf16, int64_t ld, int64_t B, int32_t F, int32_t col0, int32_t ncols, float p,
                                uint64_t seed, uint64_t offset, uint8_t* keep_out, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(xc_bf16 && B > 0 && F > 0 && col0 >= 0 && ncols > 0 && (int64_t)col0 + ncols <= ld,
                "cond_dropout: bad shape (B=%lld F=%d col0=%d ncols=%d ld=%lld)", (long long)B, F, col0, ncols, (long long)ld);
  IBM_CHECK_ARG(p > 0.f, "cond_dropout: p must be > 0 (p = 0 drops nothing and launches nothing), got %g", (double)p);
  const int drop_all = p >= 1.f;
  const uint32_t thresh = drop_all ? 0u : (uint32_t)(p * 4294967296.0);   // the keep rule of dropout_kernel
  const int grid = (int)(B < (int64_t)sm_count() * 16 ? B : (int64_t)sm_count() * 16);
  auto* xc = static_cast<__nv_bfloat16*>(xc_bf16);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (ld % 8 == 0 && aligned16(xc_bf16))
    cond_dropout_kernel<true><<<grid, kThreads, 0, s>>>(xc, ld, B, F, col0, ncols, thresh, drop_all, seed, offset, keep_out);
  else
    cond_dropout_kernel<false><<<grid, kThreads, 0, s>>>(xc, ld, B, F, col0, ncols, thresh, drop_all, seed, offset, keep_out);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_timestep_embed(const int32_t* t, int32_t t_is_scalar, int64_t B, int32_t dim, void* out_bf16,
                                  void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(t && out_bf16 && B > 0 && dim > 0 && dim % 2 == 0, "timestep_embed: bad argument");
  timestep_embed_kernel<<<ew_grid(B * (dim / 2)), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      t, t_is_scalar, B, dim, static_cast<__nv_bfloat16*>(out_bf16));
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_add_time_pos(void* h_bf16, int64_t ld, const void* temb_bf16, int64_t temb_ld, const float* pos,
                                int64_t M, int32_t F, int32_t d, const int32_t* t_row_dev, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(h_bf16 && temb_bf16 && pos && M > 0 && F > 0 && M % F == 0, "add_time_pos: bad argument");
  IBM_CHECK_ARG(d % 8 == 0 && ld % 8 == 0 && temb_ld % 8 == 0 && aligned16(h_bf16) && aligned16(temb_bf16) && aligned16(pos),
                "add_time_pos: d, ld must be multiples of 8 and pointers 16-byte aligned");
  add_time_pos_kernel<<<ew_grid(M * (d / 8)), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<__nv_bfloat16*>(h_bf16), ld, static_cast<const __nv_bfloat16*>(temb_bf16), temb_ld, pos, M, F, d, t_row_dev);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_add_time_pos_bwd(const void* dh_bf16, int64_t ld, void* dtemb_bf16, int64_t temb_ld, float* dpos,
                                    int64_t M, int32_t F, int32_t d, float* dbias, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(dh_bf16 && dtemb_bf16 && dpos && M > 0 && F > 0 && M % F == 0, "add_time_pos_bwd: bad argument");
  const long long B = M / F;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  auto* dh = static_cast<const __nv_bfloat16*>(dh_bf16);
  auto* dt = static_cast<__nv_bfloat16*>(dtemb_bf16);
  if (d % 8 == 0 && ld % 8 == 0 && temb_ld % 8 == 0 && F <= 64 && aligned16(dh_bf16) && aligned16(dtemb_bf16) && aligned16(dpos) &&
      (dbias == nullptr || aligned16(dbias))) {
    dim3 grid((unsigned)ceil_div(B, kFusedW), (unsigned)ceil_div(d, 512));
    if (F <= 52) add_time_pos_bwd_fused_kernel<13><<<grid, kThreads, 0, s>>>(dh, ld, dt, temb_ld, dpos, dbias, B, F, d);
    else add_time_pos_bwd_fused_kernel<16><<<grid, kThreads, 0, s>>>(dh, ld, dt, temb_ld, dpos, dbias, B, F, d);
    IBM_LAUNCH_CHECK();
    return IBM_OK;
  }
  IBM_CHECK_ARG(dbias == nullptr, "add_time_pos_bwd: the bias-gradient output needs the fused path (d %% 8 == 0, F <= 64, 16-byte aligned rows)");
  IBM_CHECK_ARG(d % 64 == 0 && ld % 2 == 0 && temb_ld % 2 == 0, "add_time_pos_bwd: d must be a multiple of 64");
  dim3 grid((unsigned)ceil_div(B, kTpWin), (unsigned)(d / 64));
  add_time_pos_bwd_kernel<<<grid, kThreads, 0, s>>>(dh, ld, dt, temb_ld, dpos, B, F, d);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}
