// Whole-sequence softmax attention per (window, head), forward and backward.
//
// Replaces nn.MultiheadAttention's scaled-dot-product core at
//   /root/reference/src/models/TransformerBaseline.py:12-13,29 (3 heads x 36 at d=108, fp64 in the
//   reference) and SimpleAttention (…:51-70, unscaled, value dim 3), and serves the builder-owned
//   denoiser (8 heads x 64).  Sequences are short (T = 50 … 200 frames) so K and V of one
//   (window, head) live entirely in shared memory and the T x T score matrix never leaves
//   registers; long streams scale by sharding windows, not the sequence (SURVEY §5).
//
// The projections around it are tcgen05 GEMMs (gemm_sm100.cu).  The score/PV products here are
// <2 % of the layer FLOPs at these sizes and use warp-level mma.sync.m16n8k16 (bf16 in, fp32
// accumulate) with an online softmax; one CTA = 4 warps = 64 query rows.
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "mma_sync.cuh"

namespace ibm {
namespace attn {

constexpr int kThreads = 128;

// cooperative tile load: rows [r0, r0+nrows) x W columns (W % 8 == 0) into smem with row stride LDS;
// rows >= r_valid are zero-filled.
template <int W, int LDS>
__device__ __forceinline__ void load_tile(__nv_bfloat16* dst, const __nv_bfloat16* src, int64_t ld, int nrows, int r_valid) {
  constexpr int CPR = W / 8;
  for (int i = threadIdx.x; i < nrows * CPR; i += kThreads) {
    const int r = i / CPR, c = (i - r * CPR) * 8;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r < r_valid) v = *reinterpret_cast<const uint4*>(src + (int64_t)r * ld + c);
    *reinterpret_cast<uint4*>(dst + r * LDS + c) = v;
  }
}

// ---------------------------------------- forward ----------------------------------------------
template <int HQ, int HV>
__global__ void __launch_bounds__(kThreads)
attn_fwd_kernel(const __nv_bfloat16* __restrict__ q, int64_t ldq, const __nv_bfloat16* __restrict__ k, int64_t ldk,
                const __nv_bfloat16* __restrict__ v, int64_t ldv, __nv_bfloat16* __restrict__ o, int64_t ldo, int T,
                int H, int q_tiles, float scale_log2) {
  constexpr int LK = HQ + kPad, LV = HV + kPad;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  const int Tpad = (T + 63) & ~63;
  __nv_bfloat16* Ks = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* Vs = Ks + Tpad * LK;

  const int qt = blockIdx.x % q_tiles;
  const int wh = blockIdx.x / q_tiles;
  const int h = wh % H;
  const int64_t win = wh / H;
  const int64_t row0 = win * T;
  load_tile<HQ, LK>(Ks, k + row0 * ldk + h * HQ, ldk, Tpad, T);
  load_tile<HV, LV>(Vs, v + row0 * ldv + h * HV, ldv, Tpad, T);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int qr = qt * 64 + warp * 16 + g;            // this thread's rows: qr and qr + 8
  // Q fragments straight from global (each element read exactly once per CTA)
  uint32_t qa[HQ / 16][4];
  {
    const __nv_bfloat16* q0 = q + (row0 + qr) * ldq + h * HQ;
    const __nv_bfloat16* q1 = q0 + 8 * ldq;
#pragma unroll
    for (int kk = 0; kk < HQ / 16; ++kk) {
      qa[kk][0] = qr < T ? *reinterpret_cast<const uint32_t*>(q0 + kk * 16 + 2 * t) : 0u;
      qa[kk][1] = qr + 8 < T ? *reinterpret_cast<const uint32_t*>(q1 + kk * 16 + 2 * t) : 0u;
      qa[kk][2] = qr < T ? *reinterpret_cast<const uint32_t*>(q0 + kk * 16 + 8 + 2 * t) : 0u;
      qa[kk][3] = qr + 8 < T ? *reinterpret_cast<const uint32_t*>(q1 + kk * 16 + 8 + 2 * t) : 0u;
    }
  }
  __syncthreads();

  float oacc[HV / 8][4];
#pragma unroll
  for (int j = 0; j < HV / 8; ++j) oacc[j][0] = oacc[j][1] = oacc[j][2] = oacc[j][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

  for (int kb = 0; kb < Tpad; kb += 64) {
    float s[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < HQ / 16; ++kk) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const __nv_bfloat16* kp = Ks + (kb + j * 8 + g) * LK + kk * 16 + 2 * t;
        mma16816(s[j], qa[kk], *reinterpret_cast<const uint32_t*>(kp), *reinterpret_cast<const uint32_t*>(kp + 8));
      }
    }
    // scale into log2 domain, mask keys >= T, running max
    float mx0 = m0, mx1 = m1;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int key = kb + j * 8 + 2 * t;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const bool ok = key + (e & 1) < T;
        s[j][e] = ok ? s[j][e] * scale_log2 : -INFINITY;
      }
      mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
      mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float corr0 = exp2f(m0 - mx0), corr1 = exp2f(m1 - mx1);     // m = -inf on first block → 0
    m0 = mx0; m1 = mx1;
    float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[j][0] = exp2f(s[j][0] - m0); s[j][1] = exp2f(s[j][1] - m0);
      s[j][2] = exp2f(s[j][2] - m1); s[j][3] = exp2f(s[j][3] - m1);
      rs0 += s[j][0] + s[j][1];
      rs1 += s[j][2] + s[j][3];
    }
    l0 = l0 * corr0 + rs0;
    l1 = l1 * corr1 + rs1;
#pragma unroll
    for (int j = 0; j < HV / 8; ++j) { oacc[j][0] *= corr0; oacc[j][1] *= corr0; oacc[j][2] *= corr1; oacc[j][3] *= corr1; }
    // O += P V   (P from the score accumulators: C-fragment layout == A-fragment layout)
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
      pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
      pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int j = 0; j < HV / 8; ++j) {
        uint32_t b0, b1;
        ldsm_x2_trans(b0, b1, Vs + (kb + kk * 16 + (lane & 15)) * LV + j * 8);
        mma16816(oacc[j], pa, b0, b1);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float inv0 = 1.f / l0, inv1 = 1.f / l1;
  __nv_bfloat16* o0 = o + (row0 + qr) * ldo + h * HV + 2 * t;
  __nv_bfloat16* o1 = o0 + 8 * ldo;
#pragma unroll
  for (int j = 0; j < HV / 8; ++j) {
    if (qr < T) *reinterpret_cast<uint32_t*>(o0 + j * 8) = pack_bf16x2(oacc[j][0] * inv0, oacc[j][1] * inv0);
    if (qr + 8 < T) *reinterpret_cast<uint32_t*>(o1 + j * 8) = pack_bf16x2(oacc[j][2] * inv1, oacc[j][3] * inv1);
  }
}

// ------------------------------- pipelined kernels (T <= 64) -----------------------------------
// One CTA = 4 warps = the 64 (padded) query rows of one (window, head).  CTAs are persistent over the windows of ONE
// head: the Q/K/V (and dO) tiles of the next window stream into the other half of a two-stage shared-memory ring with
// cp.async while the current window is computed, so the kernel is bound by HBM rather than by load latency (the
// one-shot kernels above/before measured 2.5 TB/s forward, 2.0 TB/s backward; profiles/r01a).  Rows >= T of every
// tile are zero for the whole kernel: they are cleared once and the loads only touch rows < T.
template <int W, int LDS>
__device__ __forceinline__ void load_tile_async(__nv_bfloat16* dst, const __nv_bfloat16* src, int64_t ld, int T) {
  constexpr int CPR = W / 8;
  if constexpr ((CPR & (CPR - 1)) == 0) {
    // a thread keeps its 16-byte column and walks down the rows: one pointer bump per copy
    constexpr int RPP = kThreads / CPR;               // rows per pass
    const int r0 = threadIdx.x / CPR, c = (threadIdx.x % CPR) * 8;
    const __nv_bfloat16* sp = src + (int64_t)r0 * ld + c;
    __nv_bfloat16* dp = dst + r0 * LDS + c;
#pragma unroll
    for (int p = 0; p < 64 / RPP; ++p) {
      if (r0 + p * RPP < T) cp_async16(dp + p * RPP * LDS, sp);
      sp += (int64_t)RPP * ld;
    }
  } else {
    for (int i = threadIdx.x; i < T * CPR; i += kThreads) {
      const int r = i / CPR, c = (i - r * CPR) * 8;
      cp_async16(dst + r * LDS + c, src + (int64_t)r * ld + c);
    }
  }
}
// a warp's 16 staged rows (row stride LDS) → global rows, 16 bytes per lane, whole 128-byte lines per 8 lanes
template <int W, int LDS>
__device__ __forceinline__ void store_rows16(const __nv_bfloat16* stage, __nv_bfloat16* dst, int64_t ld, int r_first, int T, int lane) {
  constexpr int CPR = W / 8;
#pragma unroll
  for (int i = lane; i < 16 * CPR; i += 32) {
    const int r = i / CPR, c = (i - r * CPR) * 8;
    if (r_first + r < T)
      st_stream16(dst + (int64_t)(r_first + r) * ld + c, *reinterpret_cast<const uint4*>(stage + (r_first + r) * LDS + c));
  }
}

// acc[16 x 64] += A[16 x HD] · B[64 x HD]^T.  A: 16 rows starting at `Arows` (row stride LA); B: 64 rows (stride LB).
// Key blocks j with j*8 >= T are skipped (their columns are masked afterwards).
template <int HD, int LA, int LB>
__device__ __forceinline__ void mma_abt(float (&acc)[8][4], const __nv_bfloat16* Arows, const __nv_bfloat16* Bs, int lane, int T) {
  const __nv_bfloat16* ap = Arows + (lane & 15) * LA + (lane >> 4) * 8;
  const __nv_bfloat16* bp = Bs + (lane & 7) * LB + (lane >> 3) * 8;
#pragma unroll
  for (int k2 = 0; k2 < HD / 32; ++k2) {
    uint32_t a0[4], a1[4];
    ldsm_x4(a0, ap + k2 * 32);
    ldsm_x4(a1, ap + k2 * 32 + 16);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j * 8 < T) {
        uint32_t b[4];
        ldsm_x4(b, bp + j * 8 * LB + k2 * 32);
        mma16816(acc[j], a0, b[0], b[1]);
        mma16816(acc[j], a1, b[2], b[3]);
      }
    }
  }
  if constexpr ((HD / 16) % 2 == 1) {
    constexpr int kk = HD / 16 - 1;
    uint32_t a0[4];
    ldsm_x4(a0, ap + kk * 16);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j * 8 < T) {
        uint32_t b0, b1;
        ldsm_x2(b0, b1, Bs + (j * 8 + (lane & 7)) * LB + kk * 16 + ((lane >> 3) & 1) * 8);
        mma16816(acc[j], a0, b0, b1);
      }
    }
  }
}
// scale into the log2 domain, mask keys >= T, row max over the quad, exponentials and row sums.  Returns 1/rowsum.
__device__ __forceinline__ void softmax_rows(float (&s)[8][4], int t, int T, float scale_log2, float& inv0, float& inv1) {
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (j * 8 + 8 <= T) {
      mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
      mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
    } else {
      const int key = j * 8 + 2 * t;
#pragma unroll
      for (int e = 0; e < 4; ++e) s[j][e] = (key + (e & 1) < T) ? s[j][e] : -INFINITY;
      if (j * 8 < T) {
        mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
        mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
      }
    }
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  // scale > 0, so max(scale*s) = scale*max(s): one FFMA per element feeds ex2
  const float o0 = mx0 * scale_log2, o1 = mx1 * scale_log2;
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (j * 8 < T) {
      s[j][0] = ex2(fmaf(s[j][0], scale_log2, -o0)); s[j][1] = ex2(fmaf(s[j][1], scale_log2, -o0));
      s[j][2] = ex2(fmaf(s[j][2], scale_log2, -o1)); s[j][3] = ex2(fmaf(s[j][3], scale_log2, -o1));
      l0 += s[j][0] + s[j][1];
      l1 += s[j][2] + s[j][3];
    } else {
      s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  inv0 = 1.f / l0;
  inv1 = 1.f / l1;
}

template <int HD>
__global__ void __launch_bounds__(kThreads, 4)
attn_fwd_pipe_kernel(const __nv_bfloat16* __restrict__ q, int64_t ldq, const __nv_bfloat16* __restrict__ k, int64_t ldk,
                     const __nv_bfloat16* __restrict__ v, int64_t ldv, __nv_bfloat16* __restrict__ o, int64_t ldo, int T,
                     int H, int64_t n_win, float scale_log2, int rev) {
  constexpr int LD = HD + kPad;
  constexpr int TILE = 64 * LD;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  __nv_bfloat16* base = reinterpret_cast<__nv_bfloat16*>(smem_attn);          // [2 stages][Q | K | V]
  const int h = blockIdx.x % H;
  const int64_t cta = blockIdx.x / H, ctas = gridDim.x / H;
  for (int i = threadIdx.x; i < 2 * 3 * TILE / 8; i += kThreads) reinterpret_cast<uint4*>(base)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  auto load_item = [&](int64_t win, int stage) {
    const int64_t row0 = (rev ? n_win - 1 - win : win) * T;       // rev: windows from the last one down (ibm_set_walk_order)
    __nv_bfloat16* Qs = base + stage * 3 * TILE;
    load_tile_async<HD, LD>(Qs, q + row0 * ldq + h * HD, ldq, T);
    load_tile_async<HD, LD>(Qs + TILE, k + row0 * ldk + h * HD, ldk, T);
    load_tile_async<HD, LD>(Qs + 2 * TILE, v + row0 * ldv + h * HD, ldv, T);
  };
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = warp * 16 + g;                      // this thread's query rows: r0 and r0 + 8
  int64_t win = cta;
  if (win < n_win) load_item(win, 0);
  cp_async_commit();
  for (int it = 0; win < n_win; win += ctas, ++it) {
    const int st = it & 1;
    if (win + ctas < n_win) load_item(win + ctas, st ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    __nv_bfloat16* Qs = base + st * 3 * TILE;
    const __nv_bfloat16* Ks = Qs + TILE;
    const __nv_bfloat16* Vs = Qs + 2 * TILE;

    float s[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
    mma_abt<HD, LD, LD>(s, Qs + warp * 16 * LD, Ks, lane, T);
    float inv0, inv1;
    softmax_rows(s, t, T, scale_log2, inv0, inv1);
    float oacc[HD / 8][4];
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) oacc[j][0] = oacc[j][1] = oacc[j][2] = oacc[j][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      if (kk * 16 < T) {
        uint32_t pa[4];
        pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
        pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
        pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
        mma_ab16<HD, LD>(oacc, pa, Vs + kk * 16 * LD, lane);
      }
    }
    // O → this warp's own (now dead) Q rows → coalesced 16-byte stores.  Rows >= T stay zero.
    __syncwarp();
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) {
      if (r0 < T) *reinterpret_cast<uint32_t*>(Qs + r0 * LD + j * 8 + 2 * t) = pack_bf16x2(oacc[j][0] * inv0, oacc[j][1] * inv0);
      if (r0 + 8 < T) *reinterpret_cast<uint32_t*>(Qs + (r0 + 8) * LD + j * 8 + 2 * t) = pack_bf16x2(oacc[j][2] * inv1, oacc[j][3] * inv1);
    }
    __syncwarp();
    store_rows16<HD, LD>(Qs, o + (rev ? n_win - 1 - win : win) * T * ldo + h * HD, ldo, warp * 16, T, lane);
    __syncthreads();                                 // stage st is free for the load issued next iteration
  }
}

// ------------------------------- long windows (64 < T <= 256) ----------------------------------
// The analysis pass of the TransformerBaseline runs T = 200 frames per window (BASELINE configs[4];
// TransformerBaseline.py:12,29 at 3 heads x 36 -> 48 padded).  One CTA = ceil(T/16) warps = ALL query rows of one
// (window, head): K and V are fetched once per (window, head) instead of once per 64-row query tile, and only
// ceil(T/16)*16 query rows / ceil(T/8)*8 keys are computed (T = 200: 208 x 200 instead of the one-shot kernel's
// 256 x 256, i.e. 61 % -> 96 % useful tensor work).  CTAs are persistent over the windows of one head with a two-stage
// cp.async ring for K/V, Q fragments come straight from global memory, scores stay in registers (online softmax over
// 64-key chunks, ex2.approx), fragments via ldmatrix.
template <int HQ, int HV, int NJ, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB)
attn_fwd_long_kernel(const __nv_bfloat16* __restrict__ q, int64_t ldq, const __nv_bfloat16* __restrict__ k, int64_t ldk,
                     const __nv_bfloat16* __restrict__ v, int64_t ldv, __nv_bfloat16* __restrict__ o, int64_t ldo, int T,
                     int H, int64_t n_win, float scale_log2) {
  constexpr int LDK = HQ + kPad, LDV = HV + kPad;      // HQ = width of q/k rows, HV = width of v/o rows (equal for MHA heads)
  constexpr int CPRK = HQ / 8, CPRV = HV / 8;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  const int nthreads = blockDim.x;
  const int Tp = (nthreads >> 5) * 16;                  // rows covered by the CTA's warps: (T + 15) & ~15
  const int tileK = Tp * LDK, tileV = Tp * LDV;
  __nv_bfloat16* base = reinterpret_cast<__nv_bfloat16*>(smem_attn);          // [2 stages][K | V]
  const int h = blockIdx.x % H;
  const int64_t cta = blockIdx.x / H, ctas = gridDim.x / H;
  for (int i = threadIdx.x; i < 2 * (tileK + tileV) / 8; i += nthreads) reinterpret_cast<uint4*>(base)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();                                      // rows >= T stay zero for the whole kernel
  auto load_item = [&](int64_t win, int stage) {
    const int64_t row0 = win * T;
    __nv_bfloat16* Ks = base + stage * (tileK + tileV);
    const __nv_bfloat16* ksrc = k + row0 * ldk + h * HQ;
    const __nv_bfloat16* vsrc = v + row0 * ldv + h * HV;
    for (int i = threadIdx.x; i < T * CPRK; i += nthreads) {
      const int r = i / CPRK, c = (i - r * CPRK) * 8;
      cp_async16(Ks + r * LDK + c, ksrc + (int64_t)r * ldk + c);
    }
    for (int i = threadIdx.x; i < T * CPRV; i += nthreads) {
      const int r = i / CPRV, c = (i - r * CPRV) * 8;
      cp_async16(Ks + tileK + r * LDV + c, vsrc + (int64_t)r * ldv + c);
    }
  };
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int qr = warp * 16 + g;                         // this thread's query rows: qr and qr + 8
  int64_t win = cta;
  if (win < n_win) load_item(win, 0);
  cp_async_commit();
  for (int it = 0; win < n_win; win += ctas, ++it) {
    const int st = it & 1;
    if (win + ctas < n_win) load_item(win + ctas, st ^ 1);
    cp_async_commit();
    // this warp's 16 query rows as A fragments of m16n8k16, straight from global (every element is read exactly once;
    // issued before the wait so the latency overlaps the K/V arrival and the other CTA's math)
    uint32_t qa[HQ / 16][4];
    {
      const __nv_bfloat16* q0 = q + (win * T + qr) * ldq + h * HQ + 2 * t;
      const __nv_bfloat16* q1 = q0 + 8 * ldq;
      const bool ok0 = qr < T, ok1 = qr + 8 < T;
#pragma unroll
      for (int kk = 0; kk < HQ / 16; ++kk) {
        qa[kk][0] = ok0 ? __ldg(reinterpret_cast<const unsigned int*>(q0 + kk * 16)) : 0u;
        qa[kk][1] = ok1 ? __ldg(reinterpret_cast<const unsigned int*>(q1 + kk * 16)) : 0u;
        qa[kk][2] = ok0 ? __ldg(reinterpret_cast<const unsigned int*>(q0 + kk * 16 + 8)) : 0u;
        qa[kk][3] = ok1 ? __ldg(reinterpret_cast<const unsigned int*>(q1 + kk * 16 + 8)) : 0u;
      }
    }
    cp_async_wait<1>();
    __syncthreads();
    const __nv_bfloat16* Ks = base + st * (tileK + tileV);
    const __nv_bfloat16* Vs = Ks + tileK;

    float oacc[HV / 8][4];
#pragma unroll
    for (int j = 0; j < HV / 8; ++j) oacc[j][0] = oacc[j][1] = oacc[j][2] = oacc[j][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;      // running max of the raw scores, running sums
    // one chunk of NJ*8 keys.  FULL chunks (every key valid) compile without the per-block predicates and the -inf
    // masking; only the last, ragged chunk of a window takes the general path.
    auto do_chunk = [&](const int kb, auto full_tag) {
      constexpr bool FULL = decltype(full_tag)::value;
      const int Tl = T - kb;                            // keys left from this chunk on (may exceed the chunk)
      float s[NJ][4];
#pragma unroll
      for (int j = 0; j < NJ; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
      const __nv_bfloat16* bp = Ks + (kb + (lane & 7)) * LDK + (lane >> 3) * 8;
#pragma unroll
      for (int k2 = 0; k2 < HQ / 32; ++k2) {
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          if (FULL || j * 8 < Tl) {
            uint32_t b[4];
            ldsm_x4(b, bp + j * 8 * LDK + k2 * 32);
            mma16816(s[j], qa[2 * k2], b[0], b[1]);
            mma16816(s[j], qa[2 * k2 + 1], b[2], b[3]);
          }
        }
      }
      if constexpr ((HQ / 16) % 2 == 1) {
        constexpr int kk = HQ / 16 - 1;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          if (FULL || j * 8 < Tl) {
            uint32_t b0, b1;
            ldsm_x2(b0, b1, Ks + (kb + j * 8 + (lane & 7)) * LDK + kk * 16 + ((lane >> 3) & 1) * 8);
            mma16816(s[j], qa[kk], b0, b1);
          }
        }
      }
      // chunk maxima over the valid keys
      float mx0 = m0, mx1 = m1;
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        if (FULL || j * 8 + 8 <= Tl) {
          mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
          mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
        } else if (FULL || j * 8 < Tl) {
          const int key = j * 8 + 2 * t;
#pragma unroll
          for (int e = 0; e < 4; ++e) s[j][e] = (key + (e & 1) < Tl) ? s[j][e] : -INFINITY;
          mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
          mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
        }
      }
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      const float c0 = ex2((m0 - mx0) * scale_log2), c1 = ex2((m1 - mx1) * scale_log2);     // first chunk: ex2(-inf) = 0
      m0 = mx0; m1 = mx1;
      const float o0 = m0 * scale_log2, o1 = m1 * scale_log2;
      float r0 = 0.f, r1 = 0.f;
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        if (FULL || j * 8 < Tl) {
          s[j][0] = ex2(fmaf(s[j][0], scale_log2, -o0)); s[j][1] = ex2(fmaf(s[j][1], scale_log2, -o0));
          s[j][2] = ex2(fmaf(s[j][2], scale_log2, -o1)); s[j][3] = ex2(fmaf(s[j][3], scale_log2, -o1));
          r0 += s[j][0] + s[j][1];
          r1 += s[j][2] + s[j][3];
        } else {
          s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
        }
      }
      l0 = l0 * c0 + r0;
      l1 = l1 * c1 + r1;
#pragma unroll
      for (int j = 0; j < HV / 8; ++j) { oacc[j][0] *= c0; oacc[j][1] *= c0; oacc[j][2] *= c1; oacc[j][3] *= c1; }
#pragma unroll
      for (int kk = 0; kk < NJ / 2; ++kk) {
        if (FULL || kk * 16 < Tl) {
          uint32_t pa[4];
          pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
          pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
          pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
          pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
          if constexpr (HV >= 16) {
            mma_ab16<HV, LDV>(oacc, pa, Vs + (kb + kk * 16) * LDV, lane);
          } else {                                        // 8-wide values (the CoM blend): one n = 8 block
            uint32_t b0, b1;
            ldsm_x2_trans(b0, b1, Vs + (kb + kk * 16 + (lane & 15)) * LDV);
            mma16816(oacc[0], pa, b0, b1);
          }
        }
      }
    };
    {
      int kb = 0;
      for (; kb + NJ * 8 <= T; kb += NJ * 8) do_chunk(kb, std::true_type{});
      if (kb < T) do_chunk(kb, std::false_type{});
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float inv0 = 1.f / l0, inv1 = 1.f / l1;
    __nv_bfloat16* out0 = o + (win * T + qr) * ldo + h * HV + 2 * t;
    __nv_bfloat16* out1 = out0 + 8 * ldo;
#pragma unroll
    for (int j = 0; j < HV / 8; ++j) {
      if (qr < T) *reinterpret_cast<uint32_t*>(out0 + j * 8) = pack_bf16x2(oacc[j][0] * inv0, oacc[j][1] * inv0);
      if (qr + 8 < T) *reinterpret_cast<uint32_t*>(out1 + j * 8) = pack_bf16x2(oacc[j][2] * inv1, oacc[j][3] * inv1);
    }
    __syncthreads();                                    // stage st is free for the load issued next iteration
  }
}

// dV = P^T dO, dP = dO V^T, dS = P o (dP - rowsum(P o dP)), dQ = scale dS K, dK = scale dS^T Q.
// dbias (optional): fp32 [3 * kv_off'] accumulators of the column sums of dqkv — the in-projection bias gradient
// (TransformerBaseline.py:12 in_proj_bias) — kept in registers over all windows of this CTA's head.
template <int HD>
__global__ void __launch_bounds__(kThreads, 3)
attn_bwd_kernel(const __nv_bfloat16* __restrict__ qkv, int64_t ld, int64_t kv_off, const __nv_bfloat16* __restrict__ dout,
                int64_t ldo, __nv_bfloat16* __restrict__ dqkv, int T, int H, int64_t n_win, float scale,
                float* __restrict__ dbias) {
  constexpr int LD = HD + kPad;       // Q / dO tiles [64][LD]
  constexpr int LP = 64 + kPad;       // P / dS tiles [64][LP]
  constexpr int LX = LD > LP ? LD : LP;   // K and V tiles use this stride: P and dS later overwrite them in place
  constexpr int STAGE = 2 * 64 * LD + 2 * 64 * LX;
  extern __shared__ __align__(16) uint8_t smem_attn[];
  __nv_bfloat16* base = reinterpret_cast<__nv_bfloat16*>(smem_attn);          // [2 stages][Q | dO | K | V]
  const int h = blockIdx.x % H;
  const int64_t cta = blockIdx.x / H, ctas = gridDim.x / H;
  for (int i = threadIdx.x; i < 2 * STAGE / 8; i += kThreads) reinterpret_cast<uint4*>(base)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  auto load_item = [&](int64_t win, int stage) {
    const int64_t row0 = win * T;
    __nv_bfloat16* Qs = base + stage * STAGE;
    const __nv_bfloat16* src = qkv + row0 * ld + h * HD;
    load_tile_async<HD, LD>(Qs, src, ld, T);
    load_tile_async<HD, LD>(Qs + 64 * LD, dout + row0 * ldo + h * HD, ldo, T);
    load_tile_async<HD, LX>(Qs + 2 * 64 * LD, src + kv_off, ld, T);
    load_tile_async<HD, LX>(Qs + 2 * 64 * LD + 64 * LX, src + 2 * kv_off, ld, T);
  };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = warp * 16 + g;                      // rows r0, r0+8 (queries in phase 1, keys in phase 2)
  const float scale_log2 = scale * 1.4426950408889634f;
  float cq[HD / 8][2], ck[HD / 8][2], cv[HD / 8][2];  // column sums of dq / dk / dv over this thread's rows, all windows
#pragma unroll
  for (int j = 0; j < HD / 8; ++j) { cq[j][0] = cq[j][1] = ck[j][0] = ck[j][1] = cv[j][0] = cv[j][1] = 0.f; }

  int64_t win = cta;
  if (win < n_win) load_item(win, 0);
  cp_async_commit();
  for (int it = 0; win < n_win; win += ctas, ++it) {
    const int st = it & 1;
    if (win + ctas < n_win) load_item(win + ctas, st ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    __nv_bfloat16* Qs = base + st * STAGE;
    __nv_bfloat16* dOs = Qs + 64 * LD;
    __nv_bfloat16* Ks = dOs + 64 * LD;
    __nv_bfloat16* Vs = Ks + 64 * LX;
    __nv_bfloat16* Ps = Ks;             // valid after the barrier that ends phase 1 (K, V no longer needed)
    __nv_bfloat16* dSs = Vs;
    const int64_t row0 = win * T;

    // ---- phase 1: this warp owns 16 query rows ----
    float s[8][4], dp[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f; dp[j][0] = dp[j][1] = dp[j][2] = dp[j][3] = 0.f; }
    mma_abt<HD, LD, LX>(s, Qs + warp * 16 * LD, Ks, lane, T);
    mma_abt<HD, LD, LX>(dp, dOs + warp * 16 * LD, Vs, lane, T);
    float inv0, inv1;
    softmax_rows(s, t, T, scale_log2, inv0, inv1);
    // padded query rows (>= T) get P = 0 so that the K tile they later alias keeps zero pad rows
    if (r0 >= T) inv0 = 0.f;
    if (r0 + 8 >= T) inv1 = 0.f;
    float d0 = 0.f, d1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[j][0] *= inv0; s[j][1] *= inv0; s[j][2] *= inv1; s[j][3] *= inv1;      // P
      d0 = fmaf(s[j][0], dp[j][0], fmaf(s[j][1], dp[j][1], d0));
      d1 = fmaf(s[j][2], dp[j][2], fmaf(s[j][3], dp[j][3], d1));
    }
    d0 += __shfl_xor_sync(0xffffffffu, d0, 1); d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
    d1 += __shfl_xor_sync(0xffffffffu, d1, 1); d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
    uint32_t dsa[4][4];                                  // scale*dS as A fragments for dQ = dS K
    uint32_t ppk[8][2];                                  // P (bf16 pairs), parked in registers until K/V are dead
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float e0 = s[j][0] * (dp[j][0] - d0) * scale, e1 = s[j][1] * (dp[j][1] - d0) * scale;
      const float e2 = s[j][2] * (dp[j][2] - d1) * scale, e3 = s[j][3] * (dp[j][3] - d1) * scale;
      ppk[j][0] = pack_bf16x2(s[j][0], s[j][1]);
      ppk[j][1] = pack_bf16x2(s[j][2], s[j][3]);
      dsa[j >> 1][(j & 1) * 2] = pack_bf16x2(e0, e1);
      dsa[j >> 1][(j & 1) * 2 + 1] = pack_bf16x2(e2, e3);
    }
    {
      float dq[HD / 8][4];
#pragma unroll
      for (int j = 0; j < HD / 8; ++j) dq[j][0] = dq[j][1] = dq[j][2] = dq[j][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
        if (kk * 16 < T) mma_ab16<HD, LX>(dq, dsa[kk], Ks + kk * 16 * LX, lane);
      __nv_bfloat16* g0 = dqkv + (row0 + r0) * ld + h * HD + 2 * t;
      __nv_bfloat16* g1 = g0 + 8 * ld;
#pragma unroll
      for (int j = 0; j < HD / 8; ++j) {
        if (r0 < T) *reinterpret_cast<uint32_t*>(g0 + j * 8) = pack_bf16x2(dq[j][0], dq[j][1]);
        if (r0 + 8 < T) *reinterpret_cast<uint32_t*>(g1 + j * 8) = pack_bf16x2(dq[j][2], dq[j][3]);
        // bias gradient: fp32 column sums of the unrounded values; rows >= T are exactly 0
        cq[j][0] += dq[j][0] + dq[j][2];
        cq[j][1] += dq[j][1] + dq[j][3];
      }
    }
    __syncthreads();                                     // every warp is done reading K and V
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      *reinterpret_cast<uint32_t*>(Ps + r0 * LP + j * 8 + 2 * t) = ppk[j][0];
      *reinterpret_cast<uint32_t*>(Ps + (r0 + 8) * LP + j * 8 + 2 * t) = ppk[j][1];
      *reinterpret_cast<uint32_t*>(dSs + r0 * LP + j * 8 + 2 * t) = dsa[j >> 1][(j & 1) * 2];
      *reinterpret_cast<uint32_t*>(dSs + (r0 + 8) * LP + j * 8 + 2 * t) = dsa[j >> 1][(j & 1) * 2 + 1];
    }
    __syncthreads();

    // ---- phase 2: this warp owns 16 key rows: dV = P^T dO, dK = (scale dS)^T Q ----
    {
      float dv[HD / 8][4], dk[HD / 8][4];
#pragma unroll
      for (int j = 0; j < HD / 8; ++j) { dv[j][0] = dv[j][1] = dv[j][2] = dv[j][3] = 0.f; dk[j][0] = dk[j][1] = dk[j][2] = dk[j][3] = 0.f; }
      const int kr = warp * 16;
      // x4.trans address pattern: matrices (q-rows 0-7 | keys 0-7), (q 0-7 | keys 8-15), (q 8-15 | keys 0-7), (q 8-15 | keys 8-15)
      const int qoff = (lane & 7) + ((lane >> 4) << 3);
      const int koff = ((lane >> 3) & 1) << 3;
#pragma unroll
      for (int kq = 0; kq < 4; ++kq) {
        if (kq * 16 < T) {                               // P and dS rows of padded queries are zero
          uint32_t pa[4], sa[4];
          ldsm_x4_trans(pa, Ps + (kq * 16 + qoff) * LP + kr + koff);
          ldsm_x4_trans(sa, dSs + (kq * 16 + qoff) * LP + kr + koff);
          mma_ab16<HD, LD>(dv, pa, dOs + kq * 16 * LD, lane);
          mma_ab16<HD, LD>(dk, sa, Qs + kq * 16 * LD, lane);
        }
      }
      __nv_bfloat16* gk0 = dqkv + (row0 + r0) * ld + kv_off + h * HD + 2 * t;
      __nv_bfloat16* gv0 = gk0 + kv_off;
      __nv_bfloat16* gk1 = gk0 + 8 * ld;
      __nv_bfloat16* gv1 = gv0 + 8 * ld;
#pragma unroll
      for (int j = 0; j < HD / 8; ++j) {
        if (r0 < T) {
          *reinterpret_cast<uint32_t*>(gk0 + j * 8) = pack_bf16x2(dk[j][0], dk[j][1]);
          *reinterpret_cast<uint32_t*>(gv0 + j * 8) = pack_bf16x2(dv[j][0], dv[j][1]);
        }
        if (r0 + 8 < T) {
          *reinterpret_cast<uint32_t*>(gk1 + j * 8) = pack_bf16x2(dk[j][2], dk[j][3]);
          *reinterpret_cast<uint32_t*>(gv1 + j * 8) = pack_bf16x2(dv[j][2], dv[j][3]);
        }
        ck[j][0] += dk[j][0] + dk[j][2]; ck[j][1] += dk[j][1] + dk[j][3];
        cv[j][0] += dv[j][0] + dv[j][2]; cv[j][1] += dv[j][1] + dv[j][3];
      }
    }
    __syncthreads();                                     // stage st (incl. the P / dS aliases) is free again
  }

  if (dbias != nullptr) {
    // reduce over the 8 row groups of the warp (lanes that share t), then one atomic per column per warp
#pragma unroll
    for (int j = 0; j < HD / 8; ++j) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        float a = cq[j][e], b = ck[j][e], c = cv[j][e];
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
          a += __shfl_xor_sync(0xffffffffu, a, o);
          b += __shfl_xor_sync(0xffffffffu, b, o);
          c += __shfl_xor_sync(0xffffffffu, c, o);
        }
        if (g == 0) {
          const int col = h * HD + j * 8 + 2 * t + e;
          atomicAdd(dbias + col, a);
          atomicAdd(dbias + kv_off + col, b);
          atomicAdd(dbias + 2 * kv_off + col, c);
        }
      }
    }
  }
}

template <int HQ, int HV>
static int launch_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o, int64_t ldo,
                      int64_t n_win, int T, int H, float scale, cudaStream_t s) {
  const int Tpad = (T + 63) & ~63;
  const size_t smem = (size_t)Tpad * ((HQ + kPad) + (HV + kPad)) * 2;
  auto kern = attn_fwd_kernel<HQ, HV>;
  static size_t smem_set = 0;                    // per instantiation; raise the opt-in limit only when it grows
  if (smem > smem_set) {
    IBM_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  const int q_tiles = Tpad / 64;
  const int64_t grid = n_win * H * q_tiles;
  IBM_CHECK_ARG(grid < (1ll << 31), "attention_fwd: grid too large");
  kern<<<(unsigned)grid, kThreads, smem, s>>>(static_cast<const __nv_bfloat16*>(q), ldq, static_cast<const __nv_bfloat16*>(k), ldk,
                                              static_cast<const __nv_bfloat16*>(v), ldv, static_cast<__nv_bfloat16*>(o), ldo, T, H,
                                              q_tiles, scale * 1.4426950408889634f);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

// persistent grid: as many CTAs as fit on the device, a multiple of H so that a CTA keeps one head
template <typename K>
static int pipe_grid(K kern, size_t smem, int64_t n_win, int H, int* grid) {
  int per_sm = 0;
  IBM_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, smem));
  if (per_sm < 1) per_sm = 1;
  int64_t g = (int64_t)sm_count() * per_sm / H * H;
  if (g < H) g = H;
  if (g > n_win * H) g = n_win * H;
  *grid = (int)g;
  return IBM_OK;
}

template <int HD>
static int launch_fwd_pipe(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o, int64_t ldo,
                           int64_t n_win, int T, int H, float scale, cudaStream_t s) {
  const size_t smem = (size_t)2 * 3 * 64 * (HD + kPad) * 2;
  auto kern = attn_fwd_pipe_kernel<HD>;
  static int grid_cache_key = -1, grid_cached = 0;
  static bool attr_set = false;
  if (!attr_set) {
    IBM_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  (void)grid_cache_key; (void)grid_cached;
  int grid = 0;
  int rc = pipe_grid(kern, smem, n_win, H, &grid);
  if (rc) return rc;
  kern<<<grid, kThreads, smem, s>>>(static_cast<const __nv_bfloat16*>(q), ldq, static_cast<const __nv_bfloat16*>(k), ldk,
                                    static_cast<const __nv_bfloat16*>(v), ldv, static_cast<__nv_bfloat16*>(o), ldo, T, H, n_win,
                                    scale * 1.4426950408889634f, next_walk_reverse(n_win * T * (int64_t)H * HD * 2 * 4));
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

template <int HQ, int HV>
static int launch_fwd_long(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o, int64_t ldo,
                           int64_t n_win, int T, int H, float scale, cudaStream_t s) {
  const int warps = (T + 15) / 16;
  const int threads = warps * 32;
  const size_t smem = (size_t)2 * ((T + 15) & ~15) * ((HQ + kPad) + (HV + kPad)) * 2;
  // <= 208 frames (13 warps): 32-key chunks keep the kernel under 80 registers so that TWO CTAs share an SM (26 warps
  // instead of 13 hide the HMMA / MUFU latencies; ncu: 20 % warps active, 29 % fixed-latency stalls with one);
  // longer windows: one CTA of up to 16 warps, 64-key chunks
  const bool two = warps <= 13 && 2 * smem + 4096 <= 227 * 1024 && getenv("IBM_ATTN_LONG_ONE") == nullptr;
  auto kern = two ? attn_fwd_long_kernel<HQ, HV, 4, 416, 2> : attn_fwd_long_kernel<HQ, HV, 8, 512, 1>;
  static size_t smem_set = 0;
  if (smem > smem_set) {
    IBM_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_long_kernel<HQ, HV, 4, 416, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    IBM_CHECK_CUDA(cudaFuncSetAttribute(attn_fwd_long_kernel<HQ, HV, 8, 512, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  int per_sm = 0;
  IBM_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
  if (per_sm < 1) per_sm = 1;
  int64_t g = (int64_t)sm_count() * per_sm / H * H;
  if (g < H) g = H;
  if (g > n_win * H) g = n_win * H;
  kern<<<(unsigned)g, threads, smem, s>>>(static_cast<const __nv_bfloat16*>(q), ldq, static_cast<const __nv_bfloat16*>(k), ldk,
                                          static_cast<const __nv_bfloat16*>(v), ldv, static_cast<__nv_bfloat16*>(o), ldo, T, H, n_win,
                                          scale * 1.4426950408889634f);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

template <int HD>
static int launch_bwd(const void* qkv, int64_t ld, int64_t kv_off, const void* d_o, int64_t ldo, void* dqkv, int64_t n_win, int T,
                      int H, float scale, float* dbias, cudaStream_t s) {
  constexpr int LD = HD + kPad, LP = 64 + kPad, LX = LD > LP ? LD : LP;
  const size_t smem = (size_t)2 * (2 * 64 * LD + 2 * 64 * LX) * 2;          // 2 stages x (Q, dO, K/P, V/dS)
  auto kern = attn_bwd_kernel<HD>;
  static bool attr_set = false;
  if (!attr_set) {
    IBM_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  int grid = 0;
  int rc = pipe_grid(kern, smem, n_win, H, &grid);
  if (rc) return rc;
  kern<<<grid, kThreads, smem, s>>>(static_cast<const __nv_bfloat16*>(qkv), ld, kv_off, static_cast<const __nv_bfloat16*>(d_o), ldo,
                                    static_cast<__nv_bfloat16*>(dqkv), T, H, n_win, scale, dbias);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

}  // namespace attn
}  // namespace ibm

namespace ibm {
int attention_fwd_tc(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o, int64_t ldo,
                     int64_t n_win, int T, int H, int head_dim, float scale, cudaStream_t s);        // attention_tc.cu
int attention_bwd_tc(const void* qkv, int64_t ld, int64_t kv_off, const void* d_o, int64_t ldo, void* dqkv, int64_t n_win, int T, int H,
                     int head_dim, float scale, float* dbias, cudaStream_t s);      // attention_tc.cu
}

extern "C" int ibm_attention_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o,
                                 int64_t ldo, int64_t n_win, int32_t T, int32_t H, int32_t hd_qk, int32_t hd_v, float scale,
                                 void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(q && k && v && o && n_win > 0 && T > 0 && H > 0, "attention_fwd: bad argument");
  IBM_CHECK_ARG(T <= 256, "attention_fwd: T=%d > 256 unsupported (whole sequence must fit in shared memory)", T);
  IBM_CHECK_ARG(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ldo % 2 == 0 && aligned16(q) && aligned16(k) && aligned16(v),
                "attention_fwd: leading dimensions must be multiples of 8 and pointers 16-byte aligned");
  IBM_CHECK_ARG(aligned4(o), "attention_fwd: o must be 4-byte aligned (outputs are stored as bf16 pairs)");
  IBM_CHECK_ARG(attn_scale_ok(scale), "attention_fwd: scale %g unsupported; it must be finite and > 0", scale);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // short windows, 64-wide heads (the denoiser): a tcgen05 forward kernel exists (attention_tc.cu, same construction as the
  // backward) and is parity-tested, but with half the work per window pair its per-pair latency chain leaves it at
  // 182 us vs 171 us for the mma.sync pipeline below, so it is opt-in: IBM_ATTN_FWD=tc
  if (T <= 64 && hd_qk == 64 && hd_v == 64 && ldo % 8 == 0 && aligned16(o)) {
    static int use_tc = -1;
    if (use_tc < 0) {
      const char* e = getenv("IBM_ATTN_FWD");
      use_tc = (e && e[0] == 't') ? 1 : 0;
    }
    if (use_tc) {
      const int rc = attention_fwd_tc(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, hd_qk, scale, s);
      if (rc != IBM_E_UNSUPPORTED) return rc;
    }
  }
  // short windows (T <= 64), other head sizes: persistent, double-buffered mma.sync kernel
  if (T <= 64 && hd_qk == hd_v && ldo % 8 == 0 && aligned16(o)) {
    if (hd_qk == 64) return attn::launch_fwd_pipe<64>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
    if (hd_qk == 48) return attn::launch_fwd_pipe<48>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
    if (hd_qk == 32) return attn::launch_fwd_pipe<32>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
  }
  // long windows (64 < T <= 256; the T = 200 analysis stream): one CTA per (window, head), K/V fetched once, persistent
  if (T > 64 && ldo % 2 == 0) {
    static int use_long = -1;
    if (use_long < 0) {
      const char* e = getenv("IBM_ATTN_LONG");
      use_long = (e && e[0] == '0') ? 0 : 1;           // IBM_ATTN_LONG=0 keeps the one-shot kernel (A/B measurements)
    }
    if (use_long) {
      if (hd_qk == 64 && hd_v == 64) return attn::launch_fwd_long<64, 64>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
      if (hd_qk == 48 && hd_v == 48) return attn::launch_fwd_long<48, 48>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
      if (hd_qk == 32 && hd_v == 32) return attn::launch_fwd_long<32, 32>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
      // the CoM blend of the TransformerBaseline (SimpleAttention, TransformerBaseline.py:51-70): d-wide q/k (d = 3*dofs + 9 +
      // temporal_embedding_dim padded to a multiple of 16: 112 for the dataset's 23 DOF), 8-wide values
      if (hd_v == 8) {
        if (hd_qk == 112) return attn::launch_fwd_long<112, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
        if (hd_qk == 64) return attn::launch_fwd_long<64, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
        if (hd_qk == 80) return attn::launch_fwd_long<80, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
        if (hd_qk == 96) return attn::launch_fwd_long<96, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
        if (hd_qk == 128) return attn::launch_fwd_long<128, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
      }
    }
  }
  if (hd_qk == 64 && hd_v == 64) return attn::launch_fwd<64, 64>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
  if (hd_qk == 48 && hd_v == 48) return attn::launch_fwd<48, 48>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
  if (hd_qk == 32 && hd_v == 32) return attn::launch_fwd<32, 32>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
  if (hd_v == 8) {
    if (hd_qk == 112) return attn::launch_fwd<112, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
    if (hd_qk == 64) return attn::launch_fwd<64, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
    if (hd_qk == 80) return attn::launch_fwd<80, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
    if (hd_qk == 96) return attn::launch_fwd<96, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
    if (hd_qk == 128) return attn::launch_fwd<128, 8>(q, ldq, k, ldk, v, ldv, o, ldo, n_win, T, H, scale, s);
  }
  set_error("attention_fwd: unsupported head dims (%d, %d); supported (64,64) (48,48) (32,32) and ({64,80,96,112,128},8)", hd_qk, hd_v);
  return IBM_E_UNSUPPORTED;
}

extern "C" int ibm_attention_bwd(const void* qkv, int64_t ld_qkv, int64_t kv_off, const void* d_o, int64_t ld_o, void* dqkv,
                                 int64_t n_win, int32_t T, int32_t H, int32_t head_dim, float scale, float* dbias_qkv,
                                 void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(qkv && d_o && dqkv && n_win > 0 && T > 0 && H > 0, "attention_bwd: bad argument");
  IBM_CHECK_ARG(T <= 64, "attention_bwd: T=%d > 64 unsupported", T);
  IBM_CHECK_ARG(ld_qkv % 8 == 0 && ld_o % 8 == 0 && kv_off % 8 == 0 && aligned16(qkv) && aligned16(d_o) && aligned16(dqkv),
                "attention_bwd: leading dimensions must be multiples of 8 and pointers 16-byte aligned");
  IBM_CHECK_ARG(attn_scale_ok(scale), "attention_bwd: scale %g unsupported; it must be finite and > 0", scale);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  {
    // tcgen05 kernel for the denoiser's heads (head_dim 64); IBM_ATTN_BWD=mma keeps the mma.sync kernel (A/B measurements)
    static int use_tc = -1;
    if (use_tc < 0) {
      const char* e = getenv("IBM_ATTN_BWD");
      use_tc = (e && e[0] == 'm') ? 0 : 1;
    }
    if (use_tc) {
      const int rc = attention_bwd_tc(qkv, ld_qkv, kv_off, d_o, ld_o, dqkv, n_win, T, H, head_dim, scale, dbias_qkv, s);
      if (rc != IBM_E_UNSUPPORTED) return rc;
    }
  }
  if (head_dim == 64) return attn::launch_bwd<64>(qkv, ld_qkv, kv_off, d_o, ld_o, dqkv, n_win, T, H, scale, dbias_qkv, s);
  if (head_dim == 48) return attn::launch_bwd<48>(qkv, ld_qkv, kv_off, d_o, ld_o, dqkv, n_win, T, H, scale, dbias_qkv, s);
  if (head_dim == 32) return attn::launch_bwd<32>(qkv, ld_qkv, kv_off, d_o, ld_o, dqkv, n_win, T, H, scale, dbias_qkv, s);
  set_error("attention_bwd: unsupported head dim %d; supported 32, 48, 64", head_dim);
  return IBM_E_UNSUPPORTED;
}
