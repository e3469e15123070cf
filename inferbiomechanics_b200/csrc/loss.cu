// Fused regression loss evaluator (forward + backward) — one launch each.
//
// Replaces the ~25 ATen launches + 7 `.item()` syncs per call of
//   /root/reference/src/loss/RegressionLossEvaluator.py:160-221 (step 1: four squared-diff means,
//   the 10 N CoP mask, the component-selected sum) and :230-263 (step 2.2: six last-frame reports).
// HBM-bound: algorithmic traffic 240*F bytes/window forward, +120*F bytes/window for the
// backward write (bf16 grads: +60*F).
//
// Fast path ("pair" kernels, used whenever all strides are even and pointers 8-byte aligned — every
// layout this package produces): 16 lanes per (window, frame) row, lane p owns the channel PAIR
// (2p, 2p+1) of the 30-channel row [CoP6|F6|tau6|W12] (lane 15 idles, and does the last-frame report
// arithmetic), so every access is an 8-byte vector access, a half-warp reads 120 contiguous bytes, the
// CoP mask comes from the force-label lanes of the same row by warp shuffle (no re-loads), and the
// index arithmetic is shared by two elements.  4 rows are batched per loop trip for memory-level
// parallelism.  Generic path (any strides): one thread per (row, channel).
// Column sums: per-thread register accumulators (a thread always owns the same channels) → smem →
// per-block partials → the last-arriving block reduces in fp64 in a fixed order (deterministic, no
// float atomics).
#include <math.h>

#include "common.cuh"

namespace ibm {

struct LossParams {
  const float* out[4];
  const float* lab[4];
  long long osb[4], osf[4], lsb[4], lsf[4];
  float w[30];
  long long B, F;
  float thr;
  float thr2;      // largest fp32 x with sqrtf(x) <= thr: (sqrtf(n2) > thr)  <=>  (n2 > thr2), bit for bit
};

struct GradParams {
  void* g[4];
  long long gsb[4], gsf[4];
};

constexpr int kRowsPerBlock = 8;      // generic path: 8 rows x 30 channels = 240 active threads of 256
constexpr int kPairRows = 16;         // pair path: 16 rows x 16 lanes
constexpr int kBatch = 8;             // rows in flight per thread (pair path)
constexpr int kLossThreads = 256;
constexpr int kResult = 40;           // floats per partial / result

__device__ __forceinline__ void ch_to_qc(int ch, int& q, int& c) {
  if (ch < 6) { q = 0; c = ch; }
  else if (ch < 12) { q = 1; c = ch - 6; }
  else if (ch < 18) { q = 2; c = ch - 12; }
  else { q = 3; c = ch - 18; }
}

// mask_by_threes on the label force (…Evaluator.py:85-108, threshold 10.0 at :205-209): strict >,
// norm accumulated as (a*a + b*b) + c*c without FMA contraction like the reference's fp32 torch.norm.
__device__ __forceinline__ bool norm3_gt(float a, float b, float c, float thr) {
  float n2 = __fadd_rn(__fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b)), __fmul_rn(c, c));
  return sqrtf(n2) > thr;
}
// the same predicate without the square root is norm3_gt2 (common.cuh), shared with the ensemble kernel
__device__ __forceinline__ bool force_mask(const float* f3, float thr) {
  return norm3_gt(__ldg(f3), __ldg(f3 + 1), __ldg(f3 + 2), thr);
}

// Last-arriving block: fixed-order fp64 reduction of all block partials (6 threads per value, then a
// fixed 6-term sum: deterministic for a given grid), then the final means / loss (SURVEY §9.1, §9.2).
__device__ __forceinline__ void final_reduce(const float* __restrict__ partials, float* __restrict__ result,
                                             const LossParams& p, int t, unsigned int* __restrict__ counter) {
  __shared__ double slice[37][6];
  __shared__ double fin[kResult];
  if (t < 37 * 6) {
    const int k = t / 6, sl = t % 6;
    double s = 0.0;
#pragma unroll 8
    for (unsigned int j = sl; j < gridDim.x; j += 6) s += (double)__ldcg(partials + (size_t)j * kResult + k);
    slice[k][sl] = s;
  }
  __syncthreads();
  if (t < 37) fin[t] = ((slice[t][0] + slice[t][1]) + (slice[t][2] + slice[t][3])) + (slice[t][4] + slice[t][5]);
  __syncthreads();
  if (t == 0) {
    const double N = (double)(p.B * p.F), Bd = (double)p.B;
    double loss = 0.0;
    for (int c = 0; c < 30; ++c) {
      double v = fin[c] / N;
      result[1 + c] = (float)v;
      loss += (double)p.w[c] * v;
    }
    result[0] = (float)loss;
    result[31] = (float)(fin[30] / (2.0 * Bd));                       // force
    result[32] = (float)(fin[31] / (2.0 * Bd));                       // moment
    result[33] = (float)(fin[32] / (2.0 * Bd));                       // cop
    result[34] = (float)(0.5 * (fin[33] / Bd + fin[34] / Bd));        // wrench moment
    result[35] = (float)(fin[35] / (2.0 * Bd));                       // wrench
    result[36] = (float)(fin[36] / Bd);                               // com acc
    result[37] = result[38] = result[39] = 0.f;
    *counter = 0u;
  }
}

// block partials → global; returns true in the last-arriving block
__device__ __forceinline__ bool publish_and_elect(unsigned int* __restrict__ counter, int t) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (t == 0) is_last = (atomicAdd(counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// the 6 report sums of one last-frame row from its 30 masked diffs d and the raw force values (…:119-158, 230-263)
__device__ __forceinline__ void report_row(const float* d, const float* of, const float* lf, float (&rep)[7]) {
  auto n3 = [&](int i) { return sqrtf(d[i] * d[i] + d[i + 1] * d[i + 1] + d[i + 2] * d[i + 2]); };
  rep[0] += n3(6) + n3(9);                  // force
  rep[1] += n3(12) + n3(15);                // moment
  rep[2] += n3(0) + n3(3);                  // masked CoP
  rep[3] += n3(18);                         // wrench moment, left
  rep[4] += n3(24);                         // wrench moment, right
  float w0 = 0.f, w1 = 0.f;
#pragma unroll
  for (int c = 0; c < 6; ++c) { w0 = fmaf(d[18 + c], d[18 + c], w0); w1 = fmaf(d[24 + c], d[24 + c], w1); }
  rep[5] += sqrtf(w0) + sqrtf(w1);          // wrench v=6
  const float cx = (of[0] + of[3]) - (lf[0] + lf[3]);
  const float cy = (of[1] + of[4]) - (lf[1] + lf[4]);
  const float cz = (of[2] + of[5]) - (lf[2] + lf[5]);
  rep[6] += sqrtf(cx * cx + cy * cy + cz * cz);   // CoM acc
}

// =============================================================================================
// fast path: channel pairs
// =============================================================================================
__device__ __forceinline__ void pair_to_qc(int pr, int& q, int& c) {
  if (pr < 3) { q = 0; c = 2 * pr; }
  else if (pr < 6) { q = 1; c = 2 * pr - 6; }
  else if (pr < 9) { q = 2; c = 2 * pr - 12; }
  else { q = 3; c = 2 * pr - 18; }
}

// CoP mask of this lane's two channels from the force labels held by lanes 3,4,5 of the same 16-lane row group
__device__ __forceinline__ void pair_masks(float2 l, int lane, int pr, float thr2, bool& m0, bool& m1) {
  const int base = lane & 16;
  const float f0 = __shfl_sync(0xffffffffu, l.x, base + 3), f1 = __shfl_sync(0xffffffffu, l.y, base + 3);
  const float f2 = __shfl_sync(0xffffffffu, l.x, base + 4), f3 = __shfl_sync(0xffffffffu, l.y, base + 4);
  const float f4 = __shfl_sync(0xffffffffu, l.x, base + 5), f5 = __shfl_sync(0xffffffffu, l.y, base + 5);
  const bool g0 = norm3_gt2(f0, f1, f2, thr2), g1 = norm3_gt2(f3, f4, f5, thr2);
  // pair 0 = channels (0,1) → group 0,0; pair 1 = (2,3) → 0,1; pair 2 = (4,5) → 1,1; other pairs unmasked
  m0 = pr >= 3 ? true : (pr == 2 ? g1 : g0);
  m1 = pr >= 3 ? true : (pr == 0 ? g0 : g1);
}

template <bool kBwd, bool kBf16>
__global__ void __launch_bounds__(kLossThreads)
loss_pair_kernel(const LossParams p, const GradParams gp, const float* __restrict__ upstream, float* __restrict__ result,
                 float* __restrict__ partials, unsigned int* __restrict__ counter) {
  __shared__ float red[kLossThreads][2];
  __shared__ float rep_s[kPairRows][8];
  __shared__ float scratch[kPairRows][44];          // last-frame rows: 30 diffs + 6 o_force + 6 l_force
  const int t = threadIdx.x, lane = t & 31;
  const int pr = t & 15, r = t >> 4;                // channel pair, row slot
  const bool active = pr < 15;
  int q, c;
  pair_to_qc(active ? pr : 0, q, c);
  const long long M = p.B * p.F;
  const float* __restrict__ ob = p.out[q] + c;
  const float* __restrict__ lb = p.lab[q] + c;
  const long long osb = p.osb[q], osf = p.osf[q], lsb = p.lsb[q], lsf = p.lsf[q];
  const long long S = (long long)gridDim.x * kPairRows;
  float a0 = 0.f, a1 = 0.f;
  float rep[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float sc0 = 0.f, sc1 = 0.f;
  if (kBwd) {
    const float up = upstream ? __ldg(upstream) : 1.f;
    sc0 = p.w[2 * (active ? pr : 0)] * up / (float)M;
    sc1 = p.w[2 * (active ? pr : 0) + 1] * up / (float)M;
  }
  const unsigned F32 = (unsigned)p.F;
  const unsigned dSb = (unsigned)(S / p.F), dSf = (unsigned)(S % p.F);
  // the loop bound is WARP-uniform (first row of the warp): the two half-warps own different rows but must
  // reach the shuffles together; per-lane validity is the `m < M` test below
  for (long long mw = (long long)blockIdx.x * kPairRows + ((t >> 5) << 1); mw < M; mw += S * kBatch) {
    const long long m0 = mw + (r & 1);
    float2 o[kBatch], l[kBatch];
    long long goff[kBatch];
    unsigned fr[kBatch];
    // one division per batch; the other rows of the batch are S apart: (b, f) advance by (S / F, S % F) with a carry
    unsigned b = (unsigned)((unsigned long long)m0 / F32), f = (unsigned)(m0 - (long long)b * F32);
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      const long long m = m0 + u * S;
      o[u] = make_float2(0.f, 0.f);
      l[u] = make_float2(0.f, 0.f);
      fr[u] = 0xffffffffu;
      if (m < M) {
        fr[u] = f;
        if (active) {
          o[u] = *reinterpret_cast<const float2*>(ob + b * osb + f * osf);
          l[u] = *reinterpret_cast<const float2*>(lb + b * lsb + f * lsf);
          if (kBwd) goff[u] = b * gp.gsb[q] + f * gp.gsf[q] + c;
        }
      }
      b += dSb;
      f += dSf;
      if (f >= F32) { f -= F32; ++b; }
    }
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      bool k0, k1;
      pair_masks(l[u], lane, pr, p.thr2, k0, k1);         // whole warp participates (shuffles)
      float d0 = o[u].x - l[u].x, d1 = o[u].y - l[u].y;
      if (!k0) d0 = 0.f;
      if (!k1) d1 = 0.f;
      if (kBwd) {
        if (active && fr[u] != 0xffffffffu) {
          const float g0 = (2.f * d0) * sc0, g1 = (2.f * d1) * sc1;
          if (kBf16) *reinterpret_cast<uint32_t*>(reinterpret_cast<__nv_bfloat16*>(gp.g[q]) + goff[u]) = pack_bf16x2(g0, g1);
          else *reinterpret_cast<float2*>(reinterpret_cast<float*>(gp.g[q]) + goff[u]) = make_float2(g0, g1);
        }
      } else {
        a0 = fmaf(d0, d0, a0);
        a1 = fmaf(d1, d1, a1);
        // last-frame rows also feed the six report norms: park the row in smem, lane 15 of the row does the sums
        const bool last = fr[u] == F32 - 1;
        if (__any_sync(0xffffffffu, last)) {
          if (last && active) {
            scratch[r][2 * pr] = d0;
            scratch[r][2 * pr + 1] = d1;
            if (pr >= 3 && pr < 6) {
              scratch[r][30 + 2 * (pr - 3)] = o[u].x; scratch[r][31 + 2 * (pr - 3)] = o[u].y;
              scratch[r][36 + 2 * (pr - 3)] = l[u].x; scratch[r][37 + 2 * (pr - 3)] = l[u].y;
            }
          }
          __syncwarp();
          if (last && pr == 15) report_row(scratch[r], scratch[r] + 30, scratch[r] + 36, rep);
          __syncwarp();
        }
      }
    }
  }
  if (kBwd) return;

  red[t][0] = a0;
  red[t][1] = a1;
  if (pr == 15) {
#pragma unroll
    for (int k = 0; k < 7; ++k) rep_s[r][k] = rep[k];
  }
  __syncthreads();
  float* mine = partials + (size_t)blockIdx.x * kResult;
  if (t < 30) {                                     // channel t = pair t/2, component t&1: sum over the 16 row slots
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kPairRows; ++k) s += red[k * 16 + (t >> 1)][t & 1];
    mine[t] = s;
  } else if (t >= 32 && t < 39) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kPairRows; ++k) s += rep_s[k][t - 32];
    mine[30 + (t - 32)] = s;
  }
  if (publish_and_elect(counter, t)) final_reduce(partials, result, p, t, counter);
}

// =============================================================================================
// generic path: one thread per (row, channel), any strides
// =============================================================================================
__global__ void __launch_bounds__(kLossThreads)
loss_fwd_generic_kernel(const LossParams p, float* __restrict__ result, float* __restrict__ partials,
                        unsigned int* __restrict__ counter) {
  __shared__ float red[kLossThreads];
  __shared__ float rep_s[kLossThreads / 32][7];
  const int t = threadIdx.x;
  const long long M = p.B * p.F;
  float acc = 0.f;
  if (t < kRowsPerBlock * 30) {
    const int ch = t % 30, r = t / 30;
    int q, c;
    ch_to_qc(ch, q, c);
    const float* __restrict__ ob = p.out[q] + c;
    const float* __restrict__ lb = p.lab[q] + c;
    const float* __restrict__ fb = p.lab[1] + (c / 3) * 3;
    const long long osb = p.osb[q], osf = p.osf[q], lsb = p.lsb[q], lsf = p.lsf[q];
    const long long fsb = p.lsb[1], fsf = p.lsf[1];
    const long long S = (long long)gridDim.x * kRowsPerBlock;
    const long long dS_b = S / p.F, dS_f = S % p.F;
    long long m = (long long)blockIdx.x * kRowsPerBlock + r;
    long long b = m / p.F, f = m % p.F;
#pragma unroll 4
    for (; m < M; m += S) {
      float d = __ldg(ob + b * osb + f * osf) - __ldg(lb + b * lsb + f * lsf);
      if (q == 0 && !force_mask(fb + b * fsb + f * fsf, p.thr)) d = 0.f;
      acc = fmaf(d, d, acc);
      b += dS_b;
      f += dS_f;
      if (f >= p.F) { f -= p.F; ++b; }
    }
  }
  red[t] = acc;
  // last-frame report norms: windows dealt round-robin over blocks so every SM carries a few of these rows
  float rep[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  {
    const long long f = p.F - 1;
    for (long long b = (long long)blockIdx.x + (long long)t * gridDim.x; b < p.B; b += (long long)gridDim.x * kLossThreads) {
      float d[30], of[6], lf[6];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int C = q == 3 ? 12 : 6, base = q == 3 ? 18 : 6 * q;
        const float* o = p.out[q] + b * p.osb[q] + f * p.osf[q];
        const float* l = p.lab[q] + b * p.lsb[q] + f * p.lsf[q];
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const float ov = __ldg(o + c), lv = __ldg(l + c);
          d[base + c] = ov - lv;
          if (q == 1) { of[c] = ov; lf[c] = lv; }
        }
      }
#pragma unroll
      for (int g = 0; g < 2; ++g)
        if (!norm3_gt(lf[3 * g], lf[3 * g + 1], lf[3 * g + 2], p.thr)) { d[3 * g] = 0.f; d[3 * g + 1] = 0.f; d[3 * g + 2] = 0.f; }
      report_row(d, of, lf, rep);
    }
  }
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const float v = warp_sum(rep[k]);
    if ((t & 31) == 0) rep_s[t >> 5][k] = v;
  }
  __syncthreads();
  float* mine = partials + (size_t)blockIdx.x * kResult;
  if (t < 30) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kRowsPerBlock; ++k) s += red[t + 30 * k];
    mine[t] = s;
  } else if (t >= 32 && t < 39) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kLossThreads / 32; ++k) s += rep_s[k][t - 32];
    mine[30 + (t - 32)] = s;
  }
  if (publish_and_elect(counter, t)) final_reduce(partials, result, p, t, counter);
}

template <bool kBf16>
__global__ void __launch_bounds__(kLossThreads)
loss_bwd_generic_kernel(const LossParams p, const GradParams gp, const float* __restrict__ upstream) {
  const int t = threadIdx.x;
  if (t >= kRowsPerBlock * 30) return;
  const long long M = p.B * p.F;
  const int ch = t % 30, r = t / 30;
  int q, c;
  ch_to_qc(ch, q, c);
  const float up = upstream ? __ldg(upstream) : 1.f;
  const float scale = p.w[ch] * up / (float)M;
  const float* __restrict__ ob = p.out[q] + c;
  const float* __restrict__ lb = p.lab[q] + c;
  const float* __restrict__ fb = p.lab[1] + (c / 3) * 3;
  const long long osb = p.osb[q], osf = p.osf[q], lsb = p.lsb[q], lsf = p.lsf[q];
  const long long fsb = p.lsb[1], fsf = p.lsf[1];
  const long long gsb = gp.gsb[q], gsf = gp.gsf[q];
  const long long S = (long long)gridDim.x * kRowsPerBlock;
  const long long dS_b = S / p.F, dS_f = S % p.F;
  long long m = (long long)blockIdx.x * kRowsPerBlock + r;
  long long b = m / p.F, f = m % p.F;
#pragma unroll 4
  for (; m < M; m += S) {
    float d = __ldg(ob + b * osb + f * osf) - __ldg(lb + b * lsb + f * lsf);
    if (q == 0 && !force_mask(fb + b * fsb + f * fsf, p.thr)) d = 0.f;
    const float g = (2.f * d) * scale;
    if (kBf16) reinterpret_cast<__nv_bfloat16*>(gp.g[q])[b * gsb + f * gsf + c] = __float2bfloat16_rn(g);
    else reinterpret_cast<float*>(gp.g[q])[b * gsb + f * gsf + c] = g;
    b += dS_b;
    f += dS_f;
    if (f >= p.F) { f -= p.F; ++b; }
  }
}

// =============================================================================================
// rows30 path (denoiser / Groundlink pipelines): outputs fp32 [M, 32] (the head GEMM's 128-byte rows),
// labels fp32 [M, 30], gradients bf16 [M, 32].  A warp streams 32 consecutive rows of each matrix into
// shared memory with coalesced 16-/8-byte accesses (4 KB + 3.75 KB contiguous), then each lane owns ONE
// row and reads it back with vector LDS (row strides 36 / 34 floats: conflict-free for 16-/8-byte
// accesses), so index arithmetic, the CoP mask and the last-frame test are paid once per 30 elements.
// =============================================================================================
constexpr int kSO = 36;          // smem row stride of the output tile (floats)
constexpr int kSL = 34;          // smem row stride of the label tile (floats)
constexpr int kRowStages = 3;    // cp.async ring depth per warp: two 32-row chunks in flight behind the one in use

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}

template <bool kBwd>
__global__ void __launch_bounds__(kLossThreads)
loss_rows_kernel(const float* __restrict__ out, const float* __restrict__ lab, __nv_bfloat16* __restrict__ grad,
                 const LossParams p, const float* __restrict__ upstream, float* __restrict__ result,
                 float* __restrict__ partials, unsigned int* __restrict__ counter) {
  extern __shared__ __align__(16) float smem_rows[];    // per warp and stage: out tile [32][36], lab tile [32][34]
  __shared__ float wsum[kLossThreads / 32][40];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  float* ring = smem_rows + wid * (kRowStages * 32 * (kSO + kSL));
  const long long M = p.B * p.F;
  const unsigned F32 = (unsigned)p.F;
  const long long n_chunks = (M + 31) >> 5;
  const long long warps = ((long long)gridDim.x * kLossThreads) >> 5;
  float acc[30];
#pragma unroll
  for (int c = 0; c < 30; ++c) acc[c] = 0.f;
  float rep[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float wsc[30];
  if (kBwd) {
    const float up = (upstream ? __ldg(upstream) : 1.f) / (float)M;
#pragma unroll
    for (int c = 0; c < 30; ++c) wsc[c] = 2.f * p.w[c] * up;
  }

  // stage a 32-row chunk with cp.async: out rows are 8 x 16 B, label rows 15 x 8 B, both contiguous in HBM
  auto stage_chunk = [&](long long ck, int st) {
    if (ck < n_chunks) {
      const long long m0 = ck << 5;
      const int rows = (int)min((long long)32, M - m0);
      float* so = ring + st * (32 * (kSO + kSL));
      float* sl = so + 32 * kSO;
      const float4* go = reinterpret_cast<const float4*>(out + m0 * 32);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = k * 32 + lane;                    // float4 index inside the 32-row block
        if (i < rows * 8) cp_async_16(so + (i >> 3) * kSO + (i & 7) * 4, go + i);
      }
      const float2* gl = reinterpret_cast<const float2*>(lab + m0 * 30);
#pragma unroll
      for (int k = 0; k < 15; ++k) {
        const int i = k * 32 + lane;                    // float2 index: row = i / 15
        const int r = i / 15;
        if (i < rows * 15) cp_async_8(sl + r * kSL + (i - r * 15) * 2, gl + i);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");   // one group per slot, empty past the end
  };
  const long long ck0 = (long long)blockIdx.x * (kLossThreads / 32) + wid;
#pragma unroll
  for (int i = 0; i < kRowStages - 1; ++i) stage_chunk(ck0 + i * warps, i);
  int it = 0;
  for (long long ck = ck0; ck < n_chunks; ck += warps, ++it) {
    const long long m0 = ck << 5;
    const int rows = (int)min((long long)32, M - m0);
    // the slot freed by the previous iteration (every lane passed its trailing __syncwarp) takes the chunk 2 ahead
    stage_chunk(ck + (kRowStages - 1) * warps, (it + kRowStages - 1) % kRowStages);
    asm volatile("cp.async.wait_group %0;" ::"n"(kRowStages - 1) : "memory");
    __syncwarp();
    const float* so = ring + (it % kRowStages) * (32 * (kSO + kSL));
    const float* sl = so + 32 * kSO;
    // ---- one row per lane ----
    if (lane < rows) {
      float o[32], l[30];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float4 v = *reinterpret_cast<const float4*>(so + lane * kSO + 4 * k);
        o[4 * k] = v.x; o[4 * k + 1] = v.y; o[4 * k + 2] = v.z; o[4 * k + 3] = v.w;
      }
#pragma unroll
      for (int k = 0; k < 15; ++k) {
        const float2 v = *reinterpret_cast<const float2*>(sl + lane * kSL + 2 * k);
        l[2 * k] = v.x; l[2 * k + 1] = v.y;
      }
      const bool g0 = norm3_gt2(l[6], l[7], l[8], p.thr2), g1 = norm3_gt2(l[9], l[10], l[11], p.thr2);
      float d[30];
#pragma unroll
      for (int c = 0; c < 30; ++c) {
        d[c] = o[c] - l[c];
        if (c < 3 && !g0) d[c] = 0.f;
        if (c >= 3 && c < 6 && !g1) d[c] = 0.f;
      }
      if (kBwd) {
        uint4* gr = reinterpret_cast<uint4*>(grad + (m0 + lane) * 32);
        float g[32];
#pragma unroll
        for (int c = 0; c < 30; ++c) g[c] = d[c] * wsc[c];
        g[30] = g[31] = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          gr[k] = make_uint4(pack_bf16x2(g[8 * k], g[8 * k + 1]), pack_bf16x2(g[8 * k + 2], g[8 * k + 3]),
                             pack_bf16x2(g[8 * k + 4], g[8 * k + 5]), pack_bf16x2(g[8 * k + 6], g[8 * k + 7]));
      } else {
#pragma unroll
        for (int c = 0; c < 30; ++c) acc[c] = fmaf(d[c], d[c], acc[c]);
        const unsigned f = (unsigned)(m0 + lane) % F32;       // M < 2^31 (checked on the host)
        if (f == F32 - 1) report_row(d, o + 6, l + 6, rep);
      }
    }
    __syncwarp();
  }
  if (kBwd) return;

#pragma unroll
  for (int c = 0; c < 30; ++c) {
    const float v = warp_sum(acc[c]);
    if (lane == 0) wsum[wid][c] = v;
  }
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const float v = warp_sum(rep[k]);
    if (lane == 0) wsum[wid][30 + k] = v;
  }
  __syncthreads();
  if (t < 37) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kLossThreads / 32; ++w) s += wsum[w][t];
    partials[(size_t)blockIdx.x * kResult + t] = s;
  }
  if (publish_and_elect(counter, t)) final_reduce(partials, result, p, t, counter);
}

// ------------------------------------------- host side -------------------------------------------
static int fill_params(LossParams& p, const void* const* h_out, const int64_t* os, const void* const* h_lab,
                       const int64_t* ls, int64_t B, int64_t F, const float* w, float thr) {
  IBM_CHECK_ARG(h_out && os && h_lab && ls && w, "regression_loss: null argument");
  // ValueError cases of the reference helpers (…Evaluator.py:74-79): empty tensors
  IBM_CHECK_ARG(B > 0 && F > 0, "regression_loss: Output and label tensors must not be empty (B=%lld F=%lld)",
                (long long)B, (long long)F);
  for (int q = 0; q < 4; ++q) {
    IBM_CHECK_ARG(h_out[q] && h_lab[q], "regression_loss: null tensor %d", q);
    p.out[q] = static_cast<const float*>(h_out[q]);
    p.lab[q] = static_cast<const float*>(h_lab[q]);
    p.osb[q] = os[2 * q]; p.osf[q] = os[2 * q + 1];
    p.lsb[q] = ls[2 * q]; p.lsf[q] = ls[2 * q + 1];
  }
  for (int c = 0; c < 30; ++c) p.w[c] = w[c];
  p.B = B; p.F = F; p.thr = thr;
  p.thr2 = norm3_threshold_sq(thr);
  return IBM_OK;
}

// rows30 detection: the four quantity views are column slices (0,6,12,18) of one row-major matrix with
// row-linear (window, frame) indexing
static bool rows30(const float* const ptr[4], const long long sb[4], const long long sf[4], long long F, long long& ld) {
  ld = sf[0];
  if (ld < 30 || (ld & 1)) return false;
  for (int q = 0; q < 4; ++q) {
    if (sf[q] != ld || sb[q] != F * ld) return false;
    if (ptr[q] != ptr[0] + (q == 3 ? 18 : 6 * q)) return false;
  }
  return aligned16(ptr[0]);
}

static bool pairable(const LossParams& p, const GradParams* gp, size_t gelem) {
  if (p.B * p.F >= (1ll << 31)) return false;
  for (int q = 0; q < 4; ++q) {
    if ((p.osb[q] | p.osf[q] | p.lsb[q] | p.lsf[q]) & 1) return false;
    if ((reinterpret_cast<uintptr_t>(p.out[q]) | reinterpret_cast<uintptr_t>(p.lab[q])) & 7) return false;
    if (gp) {
      if ((gp->gsb[q] | gp->gsf[q]) & 1) return false;
      if (reinterpret_cast<uintptr_t>(gp->g[q]) & (2 * gelem - 1)) return false;
    }
  }
  return true;
}

constexpr size_t kRowsSmem = (size_t)(kLossThreads / 32) * kRowStages * 32 * (kSO + kSL) * sizeof(float);   // 215 040 B

static int rows_grid(int64_t rows) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(loss_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRowsSmem);
    cudaFuncSetAttribute(loss_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRowsSmem);
    attr_set = true;
  }
  int64_t need = ceil_div(rows, 32 * (kLossThreads / 32));
  int64_t cap = (int64_t)sm_count();            // one block (its ring is 210 KB) per SM
  int64_t maxp = (int64_t)(ibm_workspace_bytes() - 256) / (kResult * sizeof(float));
  if (cap > maxp) cap = maxp;
  return (int)(need < cap ? (need < 1 ? 1 : need) : cap);
}

static int loss_grid(int64_t rows, int rows_per_block) {
  int64_t need = ceil_div(rows, rows_per_block);
  int64_t cap = (int64_t)sm_count() * 8;
  int64_t maxp = (int64_t)(ibm_workspace_bytes() - 256) / (kResult * sizeof(float));
  if (cap > maxp) cap = maxp;
  return (int)(need < cap ? (need < 1 ? 1 : need) : cap);
}

}  // namespace ibm

extern "C" int ibm_regression_loss_fwd(const void* const* h_out, const int64_t* h_out_strides,
                                       const void* const* h_lab, const int64_t* h_lab_strides, int64_t B,
                                       int64_t F, const float* h_weights, float threshold, float* result,
                                       void* workspace, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  LossParams p;
  int rc = fill_params(p, h_out, h_out_strides, h_lab, h_lab_strides, B, F, h_weights, threshold);
  if (rc) return rc;
  IBM_CHECK_ARG(result && workspace, "regression_loss_fwd: null result/workspace");
  unsigned int* counter = static_cast<unsigned int*>(workspace);
  float* partials = reinterpret_cast<float*>(static_cast<char*>(workspace) + 256);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  long long ldo = 0, ldl = 0;
  if (B * F < (1ll << 31) && rows30(p.out, p.osb, p.osf, F, ldo) && rows30(p.lab, p.lsb, p.lsf, F, ldl) && ldo == 32 && ldl == 30) {
    const int grid = rows_grid(B * F);
    loss_rows_kernel<false><<<grid, kLossThreads, kRowsSmem, s>>>(p.out[0], p.lab[0], nullptr, p, nullptr, result, partials, counter);
  } else if (pairable(p, nullptr, 0)) {
    GradParams none = {};
    loss_pair_kernel<false, false><<<loss_grid(ceil_div(B * F, kBatch), kPairRows), kLossThreads, 0, s>>>(p, none, nullptr, result,
                                                                                                        partials, counter);
  } else {
    loss_fwd_generic_kernel<<<loss_grid(B * F, kRowsPerBlock), kLossThreads, 0, s>>>(p, result, partials, counter);
  }
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_regression_loss_bwd(const void* const* h_out, const int64_t* h_out_strides,
                                       const void* const* h_lab, const int64_t* h_lab_strides, int64_t B,
                                       int64_t F, const float* h_weights, float threshold, const float* upstream,
                                       void* const* h_grad, const int64_t* h_grad_strides, int32_t grad_dtype,
                                       void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  LossParams p;
  int rc = fill_params(p, h_out, h_out_strides, h_lab, h_lab_strides, B, F, h_weights, threshold);
  if (rc) return rc;
  IBM_CHECK_ARG(h_grad && h_grad_strides, "regression_loss_bwd: null grad");
  IBM_CHECK_ARG(grad_dtype == IBM_F32 || grad_dtype == IBM_BF16, "regression_loss_bwd: bad grad dtype %d", grad_dtype);
  GradParams gp;
  for (int q = 0; q < 4; ++q) {
    IBM_CHECK_ARG(h_grad[q], "regression_loss_bwd: null grad tensor %d", q);
    gp.g[q] = h_grad[q];
    gp.gsb[q] = h_grad_strides[2 * q];
    gp.gsf[q] = h_grad_strides[2 * q + 1];
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool bf = grad_dtype == IBM_BF16;
  long long ldo = 0, ldl = 0, ldg = gp.gsf[0];
  bool grows = ldg >= 30 && !(ldg & 1) && aligned16(gp.g[0]);
  for (int q = 0; q < 4 && grows; ++q)
    grows = gp.gsf[q] == ldg && gp.gsb[q] == F * ldg &&
            static_cast<char*>(gp.g[q]) == static_cast<char*>(gp.g[0]) + (q == 3 ? 18 : 6 * q) * (bf ? 2 : 4);
  if (grows && bf && ldg == 32 && B * F < (1ll << 31) && rows30(p.out, p.osb, p.osf, F, ldo) && rows30(p.lab, p.lsb, p.lsf, F, ldl) &&
      ldo == 32 && ldl == 30) {
    loss_rows_kernel<true><<<rows_grid(B * F), kLossThreads, kRowsSmem, s>>>(p.out[0], p.lab[0], static_cast<__nv_bfloat16*>(gp.g[0]), p,
                                                                              upstream, nullptr, nullptr, nullptr);
  } else if (pairable(p, &gp, bf ? 2 : 4)) {
    const int grid = loss_grid(ceil_div(B * F, kBatch), kPairRows);
    if (bf) loss_pair_kernel<true, true><<<grid, kLossThreads, 0, s>>>(p, gp, upstream, nullptr, nullptr, nullptr);
    else loss_pair_kernel<true, false><<<grid, kLossThreads, 0, s>>>(p, gp, upstream, nullptr, nullptr, nullptr);
  } else {
    const int grid = loss_grid(B * F, kRowsPerBlock);
    if (bf) loss_bwd_generic_kernel<true><<<grid, kLossThreads, 0, s>>>(p, gp, upstream);
    else loss_bwd_generic_kernel<false><<<grid, kLossThreads, 0, s>>>(p, gp, upstream);
  }
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}
