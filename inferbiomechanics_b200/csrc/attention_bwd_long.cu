// Softmax-attention backward for whole windows of up to 256 frames, any supported head width.
//
// Replaces the autograd backward of nn.MultiheadAttention's core at the reference's own shape
//   /root/reference/src/models/TransformerBaseline.py:12-13,29  (3 heads x 36 -> 48 padded, T = window_size up to 200)
// and of SimpleAttention (…:51-70: unscaled scores over 108 -> 112-wide q/k, 3 -> 8-wide values, values are an INPUT
// so only dq / dk are produced).  ibm_attention_bwd (attention.cu / attention_tc.cu) covers T <= 64.
//
// One CTA = ceil(T/16) warps holds Q, K, V and dO of one (window, head) in shared memory; CTAs are persistent over
// the windows of one head.  Nothing T x T ever leaves registers, in two phases with swapped roles:
//   phase 1 (a warp owns 16 QUERY rows): pass A over the keys gives the row maximum and sum (log-sum-exp) and
//            D = rowsum(dO o O); pass B recomputes P chunk by chunk, dP = dO V^T, dS = P o (dP - D) * scale, and
//            accumulates dQ = dS K.  (lse, D) per query go to shared memory.
//   phase 2 (a warp owns 16 KEY rows): S^T = K Q^T and dP^T = V dO^T per query chunk, P^T / dS^T from the stored
//            (lse, D), dV = P^T dO and dK = dS^T Q accumulate in registers — the mma.sync C fragment of a
//            [16 keys x 8 queries] tile IS the A fragment of the [16 x 16] x [16 x hd] product that follows.
// The score products are therefore evaluated three times instead of once (3 HQ + ... of T^2 work), the price of keeping the
// T x T matrices out of shared memory (P and dS in bf16 would need 173 KB at T = 208 next to the 93 KB of operands).
// Column sums of dq / dk / dv (the in_proj_bias gradient) are kept in registers over all windows of the CTA's head.
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "mma_sync.cuh"

namespace ibm {
namespace attn {

// s[NJ][4] += A[16 x HD] (fragments a[HD/16]) · B[NJ*8 x HD]^T, B rows at `Brows` with row stride LDB; 8-row blocks
// starting at or after `left` rows are skipped
template <int HD, int LDB, int NJ>
__device__ __forceinline__ void mma_frag_abt(float (&s)[NJ][4], const uint32_t (&a)[HD / 16][4], const __nv_bfloat16* Brows,
                                             int lane, int left) {
  const __nv_bfloat16* bp = Brows + (lane & 7) * LDB + (lane >> 3) * 8;
#pragma unroll
  for (int k2 = 0; k2 < HD / 32; ++k2) {
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      if (j * 8 < left) {
        uint32_t b[4];
        ldsm_x4(b, bp + j * 8 * LDB + k2 * 32);
        mma16816(s[j], a[2 * k2], b[0], b[1]);
        mma16816(s[j], a[2 * k2 + 1], b[2], b[3]);
      }
    }
  }
  if constexpr ((HD / 16) % 2 == 1) {
    constexpr int kk = HD / 16 - 1;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      if (j * 8 < left) {
        uint32_t b0, b1;
        ldsm_x2(b0, b1, Brows + (j * 8 + (lane & 7)) * LDB + kk * 16 + ((lane >> 3) & 1) * 8);
        mma16816(s[j], a[kk], b0, b1);
      }
    }
  }
}

template <int HD, int LDA>
__device__ __forceinline__ void load_a_frags(uint32_t (&a)[HD / 16][4], const __nv_bfloat16* Arows, int lane) {
  const __nv_bfloat16* ap = Arows + (lane & 15) * LDA + (lane >> 4) * 8;
#pragma unroll
  for (int kk = 0; kk < HD / 16; ++kk) ldsm_x4(a[kk], ap + kk * 16);
}

template <int NJ>
__device__ __forceinline__ void zero_acc(float (&s)[NJ][4]) {
#pragma unroll
  for (int j = 0; j < NJ; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
}

// HQ: width of q / k rows; HV: width of v / o / dO rows (8 for the CoM blend, contraction padded to 16 with zero columns);
// NEED_DV: also produce dv (false when the values are an input); DB: accumulate the column sums (bias gradients).
template <int HQ, int HV, bool NEED_DV, bool DB, int MAXT>
__global__ void __launch_bounds__(MAXT, 1)
attn_bwd_long_kernel(const __nv_bfloat16* __restrict__ q, int64_t ldq, const __nv_bfloat16* __restrict__ k, int64_t ldk,
                     const __nv_bfloat16* __restrict__ v, int64_t ldv, const __nv_bfloat16* __restrict__ o, int64_t ldo,
                     const __nv_bfloat16* __restrict__ dO, int64_t lddo, __nv_bfloat16* __restrict__ dq, int64_t lddq,
                     __nv_bfloat16* __restrict__ dk, int64_t lddk, __nv_bfloat16* __restrict__ dv, int64_t lddv, int T, int H,
                     int64_t n_win, float scale, float* __restrict__ dbq, float* __restrict__ dbk, float* __restrict__ dbv) {
  constexpr int NJ = 4;                                 // 32-key (phase 1) / 32-query (phase 2) chunks
  constexpr int HVK = HV < 16 ? 16 : HV;                // contraction width of dO V^T
  constexpr int LDK = HQ + kPad, LDV = HVK + kPad;
  constexpr int CPRK = HQ / 8, CPRV = HV / 8;
  static_assert(!NEED_DV || HV >= 16, "dv needs 16-wide value rows");
  extern __shared__ __align__(16) uint8_t smem_attn[];
  const int nthreads = blockDim.x;
  const int Tp = (nthreads >> 5) * 16;
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(smem_attn);
  __nv_bfloat16* Ks = Qs + Tp * LDK;
  __nv_bfloat16* Vs = Ks + Tp * LDK;
  __nv_bfloat16* dOs = Vs + Tp * LDV;
  float2* stats = reinterpret_cast<float2*>(dOs + Tp * LDV);        // (lse in the log2 domain, D) per query row
  const int h = blockIdx.x % H;
  const int64_t cta = blockIdx.x / H, ctas = gridDim.x / H;
  // rows >= T and the pad columns stay zero for the whole kernel: the loads only touch rows < T, columns < HQ / HV
  for (int i = threadIdx.x; i < (2 * Tp * LDK + 2 * Tp * LDV) / 8; i += nthreads) reinterpret_cast<uint4*>(Qs)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int r0 = warp * 16 + g;                         // this thread's rows r0, r0 + 8 (queries in phase 1, keys in phase 2)
  const bool ok0 = r0 < T, ok1 = r0 + 8 < T;
  const float sl = scale * 1.4426950408889634f;
  float cq[DB ? HQ / 8 : 1][2], ck[DB ? HQ / 8 : 1][2], cv[DB && NEED_DV ? HV / 8 : 1][2];
  if constexpr (DB) {
#pragma unroll
    for (int j = 0; j < HQ / 8; ++j) cq[j][0] = cq[j][1] = ck[j][0] = ck[j][1] = 0.f;
    if constexpr (NEED_DV) {
#pragma unroll
      for (int j = 0; j < HV / 8; ++j) cv[j][0] = cv[j][1] = 0.f;
    }
  }

  for (int64_t win = cta; win < n_win; win += ctas) {
    const int64_t row0 = win * T;
    {
      const __nv_bfloat16* qsrc = q + row0 * ldq + h * HQ;
      const __nv_bfloat16* ksrc = k + row0 * ldk + h * HQ;
      const __nv_bfloat16* vsrc = v + row0 * ldv + h * HV;
      const __nv_bfloat16* gsrc = dO + row0 * lddo + h * HV;
      for (int i = threadIdx.x; i < T * CPRK; i += nthreads) {
        const int r = i / CPRK, c = (i - r * CPRK) * 8;
        cp_async16(Qs + r * LDK + c, qsrc + (int64_t)r * ldq + c);
        cp_async16(Ks + r * LDK + c, ksrc + (int64_t)r * ldk + c);
      }
      for (int i = threadIdx.x; i < T * CPRV; i += nthreads) {
        const int r = i / CPRV, c = (i - r * CPRV) * 8;
        cp_async16(Vs + r * LDV + c, vsrc + (int64_t)r * ldv + c);
        cp_async16(dOs + r * LDV + c, gsrc + (int64_t)r * lddo + c);
      }
      cp_async_commit();
    }
    // D = rowsum(dO o O) for this thread's two query rows, straight from global (each element read once)
    float d0 = 0.f, d1 = 0.f;
    {
      const __nv_bfloat16* o0 = o + (row0 + r0) * ldo + h * HV + 2 * t;
      const __nv_bfloat16* g0 = dO + (row0 + r0) * lddo + h * HV + 2 * t;
#pragma unroll
      for (int j = 0; j < HV / 8; ++j) {
        if (ok0) {
          const float2 a = unpack_bf16x2(__ldg(reinterpret_cast<const unsigned int*>(o0 + j * 8)));
          const float2 b = unpack_bf16x2(__ldg(reinterpret_cast<const unsigned int*>(g0 + j * 8)));
          d0 = fmaf(a.x, b.x, fmaf(a.y, b.y, d0));
        }
        if (ok1) {
          const float2 a = unpack_bf16x2(__ldg(reinterpret_cast<const unsigned int*>(o0 + 8 * ldo + j * 8)));
          const float2 b = unpack_bf16x2(__ldg(reinterpret_cast<const unsigned int*>(g0 + 8 * lddo + j * 8)));
          d1 = fmaf(a.x, b.x, fmaf(a.y, b.y, d1));
        }
      }
      d0 += __shfl_xor_sync(0xffffffffu, d0, 1); d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
      d1 += __shfl_xor_sync(0xffffffffu, d1, 1); d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
    }
    cp_async_wait<0>();
    __syncthreads();

    // ------------------------------ phase 1: 16 query rows per warp ------------------------------
    float lse0, lse1;
    {
      uint32_t qa[HQ / 16][4], ga[HVK / 16][4];
      load_a_frags<HQ, LDK>(qa, Qs + warp * 16 * LDK, lane);
      load_a_frags<HVK, LDV>(ga, dOs + warp * 16 * LDV, lane);
      // pass A: row maximum of the raw scores and the sum of exponentials
      float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
      for (int kb = 0; kb < T; kb += NJ * 8) {
        const int Tl = T - kb;
        float s[NJ][4];
        zero_acc<NJ>(s);
        mma_frag_abt<HQ, LDK, NJ>(s, qa, Ks + kb * LDK, lane, Tl);
        float mx0 = m0, mx1 = m1;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int key = j * 8 + 2 * t;
#pragma unroll
          for (int e = 0; e < 4; ++e) s[j][e] = (key + (e & 1) < Tl) ? s[j][e] : -INFINITY;
          mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
          mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float c0 = ex2((m0 - mx0) * sl), c1 = ex2((m1 - mx1) * sl);       // first chunk: ex2(-inf) = 0
        m0 = mx0; m1 = mx1;
        const float o0 = m0 * sl, o1 = m1 * sl;
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          a0 += ex2(fmaf(s[j][0], sl, -o0)) + ex2(fmaf(s[j][1], sl, -o0));      // masked keys: ex2(-inf) = 0
          a1 += ex2(fmaf(s[j][2], sl, -o1)) + ex2(fmaf(s[j][3], sl, -o1));
        }
        l0 = l0 * c0 + a0;
        l1 = l1 * c1 + a1;
      }
      l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
      lse0 = fmaf(m0, sl, __log2f(l0));
      lse1 = fmaf(m1, sl, __log2f(l1));
      // padded query rows: lse = +inf makes every probability of that row vanish in phase 2
      if (t == 0) {
        stats[r0] = make_float2(ok0 ? lse0 : INFINITY, d0);
        stats[r0 + 8] = make_float2(ok1 ? lse1 : INFINITY, d1);
      }
      // pass B: P, dP, dS per key chunk; dQ = dS K
      float acc[HQ / 8][4];
      zero_acc<HQ / 8>(acc);
      for (int kb = 0; kb < T; kb += NJ * 8) {
        const int Tl = T - kb;
        float s[NJ][4], dp[NJ][4];
        zero_acc<NJ>(s);
        zero_acc<NJ>(dp);
        mma_frag_abt<HQ, LDK, NJ>(s, qa, Ks + kb * LDK, lane, Tl);
        mma_frag_abt<HVK, LDV, NJ>(dp, ga, Vs + kb * LDV, lane, Tl);
        uint32_t dsa[NJ / 2][4];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int key = j * 8 + 2 * t;
          const bool v0 = key < Tl, v1 = key + 1 < Tl;
          const float p0 = v0 ? ex2(fmaf(s[j][0], sl, -lse0)) : 0.f, p1 = v1 ? ex2(fmaf(s[j][1], sl, -lse0)) : 0.f;
          const float p2 = v0 ? ex2(fmaf(s[j][2], sl, -lse1)) : 0.f, p3 = v1 ? ex2(fmaf(s[j][3], sl, -lse1)) : 0.f;
          dsa[j >> 1][(j & 1) * 2] = pack_bf16x2(p0 * (dp[j][0] - d0) * scale, p1 * (dp[j][1] - d0) * scale);
          dsa[j >> 1][(j & 1) * 2 + 1] = pack_bf16x2(p2 * (dp[j][2] - d1) * scale, p3 * (dp[j][3] - d1) * scale);
        }
#pragma unroll
        for (int kk = 0; kk < NJ / 2; ++kk)
          if (kk * 16 < Tl) mma_ab16<HQ, LDK>(acc, dsa[kk], Ks + (kb + kk * 16) * LDK, lane);
      }
      __nv_bfloat16* g0 = dq + (row0 + r0) * lddq + h * HQ + 2 * t;
      __nv_bfloat16* g1 = g0 + 8 * lddq;
#pragma unroll
      for (int j = 0; j < HQ / 8; ++j) {
        if (ok0) *reinterpret_cast<uint32_t*>(g0 + j * 8) = pack_bf16x2(acc[j][0], acc[j][1]);
        if (ok1) *reinterpret_cast<uint32_t*>(g1 + j * 8) = pack_bf16x2(acc[j][2], acc[j][3]);
        if constexpr (DB) {                              // rows >= T are exactly zero (dO rows are zero there)
          cq[j][0] += acc[j][0] + acc[j][2];
          cq[j][1] += acc[j][1] + acc[j][3];
        }
      }
    }
    __syncthreads();                                     // (lse, D) of every query row are in shared memory

    // ------------------------------ phase 2: 16 key rows per warp --------------------------------
    {
      uint32_t ka[HQ / 16][4], va[HVK / 16][4];
      load_a_frags<HQ, LDK>(ka, Ks + warp * 16 * LDK, lane);
      load_a_frags<HVK, LDV>(va, Vs + warp * 16 * LDV, lane);
      float dka[HQ / 8][4];
      float dva[NEED_DV ? HV / 8 : 1][4];
      zero_acc<HQ / 8>(dka);
      zero_acc<NEED_DV ? HV / 8 : 1>(dva);
      for (int qb = 0; qb < T; qb += NJ * 8) {
        const int Tl = T - qb;
        float s[NJ][4], dp[NJ][4];
        zero_acc<NJ>(s);
        zero_acc<NJ>(dp);
        mma_frag_abt<HQ, LDK, NJ>(s, ka, Qs + qb * LDK, lane, Tl);
        mma_frag_abt<HVK, LDV, NJ>(dp, va, dOs + qb * LDV, lane, Tl);
        uint32_t pa[NJ / 2][4], dsa[NJ / 2][4];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          float p[4], e[4];
          if (j * 8 < Tl) {
            const float2 st0 = stats[qb + j * 8 + 2 * t], st1 = stats[qb + j * 8 + 2 * t + 1];   // queries >= T: lse = +inf
            p[0] = ex2(fmaf(s[j][0], sl, -st0.x)); p[1] = ex2(fmaf(s[j][1], sl, -st1.x));
            p[2] = ex2(fmaf(s[j][2], sl, -st0.x)); p[3] = ex2(fmaf(s[j][3], sl, -st1.x));
            e[0] = p[0] * (dp[j][0] - st0.y) * scale; e[1] = p[1] * (dp[j][1] - st1.y) * scale;
            e[2] = p[2] * (dp[j][2] - st0.y) * scale; e[3] = p[3] * (dp[j][3] - st1.y) * scale;
          } else {
            p[0] = p[1] = p[2] = p[3] = 0.f;
            e[0] = e[1] = e[2] = e[3] = 0.f;
          }
          pa[j >> 1][(j & 1) * 2] = pack_bf16x2(p[0], p[1]);
          pa[j >> 1][(j & 1) * 2 + 1] = pack_bf16x2(p[2], p[3]);
          dsa[j >> 1][(j & 1) * 2] = pack_bf16x2(e[0], e[1]);
          dsa[j >> 1][(j & 1) * 2 + 1] = pack_bf16x2(e[2], e[3]);
        }
#pragma unroll
        for (int kk = 0; kk < NJ / 2; ++kk) {
          if (kk * 16 < Tl) {
            if constexpr (NEED_DV) mma_ab16<HV, LDV>(dva, pa[kk], dOs + (qb + kk * 16) * LDV, lane);
            mma_ab16<HQ, LDK>(dka, dsa[kk], Qs + (qb + kk * 16) * LDK, lane);
          }
        }
      }
      __nv_bfloat16* gk0 = dk + (row0 + r0) * lddk + h * HQ + 2 * t;
      __nv_bfloat16* gk1 = gk0 + 8 * lddk;
#pragma unroll
      for (int j = 0; j < HQ / 8; ++j) {
        if (ok0) *reinterpret_cast<uint32_t*>(gk0 + j * 8) = pack_bf16x2(dka[j][0], dka[j][1]);
        if (ok1) *reinterpret_cast<uint32_t*>(gk1 + j * 8) = pack_bf16x2(dka[j][2], dka[j][3]);
        if constexpr (DB) {                              // padded KEY rows hold garbage (their scores are not masked): excluded
          ck[j][0] += (ok0 ? dka[j][0] : 0.f) + (ok1 ? dka[j][2] : 0.f);
          ck[j][1] += (ok0 ? dka[j][1] : 0.f) + (ok1 ? dka[j][3] : 0.f);
        }
      }
      if constexpr (NEED_DV) {
        __nv_bfloat16* gv0 = dv + (row0 + r0) * lddv + h * HV + 2 * t;
        __nv_bfloat16* gv1 = gv0 + 8 * lddv;
#pragma unroll
        for (int j = 0; j < HV / 8; ++j) {
          if (ok0) *reinterpret_cast<uint32_t*>(gv0 + j * 8) = pack_bf16x2(dva[j][0], dva[j][1]);
          if (ok1) *reinterpret_cast<uint32_t*>(gv1 + j * 8) = pack_bf16x2(dva[j][2], dva[j][3]);
          if constexpr (DB) {
            cv[j][0] += (ok0 ? dva[j][0] : 0.f) + (ok1 ? dva[j][2] : 0.f);
            cv[j][1] += (ok0 ? dva[j][1] : 0.f) + (ok1 ? dva[j][3] : 0.f);
          }
        }
      }
    }
    __syncthreads();                                     // the tiles are free for the next window's loads
  }

  if constexpr (DB) {
    // reduce over the 8 row groups of the warp (lanes that share t), then one atomic per column per warp
#pragma unroll
    for (int j = 0; j < HQ / 8; ++j) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        float a = cq[j][e], b = ck[j][e];
#pragma unroll
        for (int x = 4; x < 32; x <<= 1) {
          a += __shfl_xor_sync(0xffffffffu, a, x);
          b += __shfl_xor_sync(0xffffffffu, b, x);
        }
        if (g == 0) {
          const int col = h * HQ + j * 8 + 2 * t + e;
          if (dbq) atomicAdd(dbq + col, a);
          if (dbk) atomicAdd(dbk + col, b);
        }
      }
    }
    if constexpr (NEED_DV) {
#pragma unroll
      for (int j = 0; j < HV / 8; ++j) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          float c = cv[j][e];
#pragma unroll
          for (int x = 4; x < 32; x <<= 1) c += __shfl_xor_sync(0xffffffffu, c, x);
          if (g == 0 && dbv) atomicAdd(dbv + h * HV + j * 8 + 2 * t + e, c);
        }
      }
    }
  }
}

template <int HQ, int HV, bool NEED_DV>
static int launch_bwd_long(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const void* o,
                           int64_t ldo, const void* d_o, int64_t lddo, void* dq, int64_t lddq, void* dk, int64_t lddk, void* dv,
                           int64_t lddv, int64_t n_win, int T, int H, float scale, float* dbq, float* dbk, float* dbv, cudaStream_t s) {
  constexpr int HVK = HV < 16 ? 16 : HV;
  const int warps = (T + 15) / 16;
  const int threads = warps * 32;
  const int Tp = warps * 16;
  const size_t smem = (size_t)2 * Tp * ((HQ + kPad) + (HVK + kPad)) * 2 + (size_t)Tp * sizeof(float2);
  const bool db = dbq || dbk || dbv;
  // <= 13 warps (T <= 208, the reference's window sizes): compiled for 416 threads so the register allocator gets 152
  // registers per thread; up to 16 warps otherwise (128 registers)
  const bool small = warps <= 13;
  auto pick = [&](auto dbtag) {
    constexpr bool DB = decltype(dbtag)::value;
    return small ? attn_bwd_long_kernel<HQ, HV, NEED_DV, DB, 416> : attn_bwd_long_kernel<HQ, HV, NEED_DV, DB, 512>;
  };
  auto kern = db ? pick(std::true_type{}) : pick(std::false_type{});
  IBM_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  IBM_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
  if (per_sm < 1) per_sm = 1;
  int64_t g = (int64_t)sm_count() * per_sm / H * H;
  if (g < H) g = H;
  if (g > n_win * H) g = n_win * H;
  kern<<<(unsigned)g, threads, smem, s>>>(
      static_cast<const __nv_bfloat16*>(q), ldq, static_cast<const __nv_bfloat16*>(k), ldk, static_cast<const __nv_bfloat16*>(v), ldv,
      static_cast<const __nv_bfloat16*>(o), ldo, static_cast<const __nv_bfloat16*>(d_o), lddo, static_cast<__nv_bfloat16*>(dq), lddq,
      static_cast<__nv_bfloat16*>(dk), lddk, static_cast<__nv_bfloat16*>(dv), lddv, T, H, n_win, scale, dbq, dbk, dbv);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

}  // namespace attn
}  // namespace ibm

extern "C" int ibm_attention_bwd_long(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                                      const void* o, int64_t ldo, const void* d_o, int64_t ld_do, void* dq, int64_t lddq, void* dk,
                                      int64_t lddk, void* dv, int64_t lddv, int64_t n_win, int32_t T, int32_t H, int32_t hd_qk,
                                      int32_t hd_v, float scale, float* dbias_q, float* dbias_k, float* dbias_v, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(q && k && v && o && d_o && dq && dk && n_win > 0 && T > 0 && H > 0, "attention_bwd_long: bad argument");
  IBM_CHECK_ARG(T <= 256, "attention_bwd_long: T=%d > 256 unsupported (whole sequence must fit in shared memory)", T);
  IBM_CHECK_ARG(ldq % 8 == 0 && ldk % 8 == 0 && ldv % 8 == 0 && ld_do % 8 == 0 && ldo % 2 == 0 && lddq % 2 == 0 && lddk % 2 == 0 &&
                    (dv == nullptr || lddv % 2 == 0) && aligned16(q) && aligned16(k) && aligned16(v) && aligned16(d_o),
                "attention_bwd_long: q/k/v/d_o need leading dimensions that are multiples of 8 and 16-byte aligned pointers");
  IBM_CHECK_ARG(aligned4(o) && aligned4(dq) && aligned4(dk) && (dv == nullptr || aligned4(dv)),
                "attention_bwd_long: o, dq, dk and dv must be 4-byte aligned (they are read and stored as bf16 pairs)");
  IBM_CHECK_ARG(attn_scale_ok(scale), "attention_bwd_long: scale %g unsupported; it must be finite and > 0", scale);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define IBM_BWD_LONG(HQV, HVV, DV) \
  return attn::launch_bwd_long<HQV, HVV, DV>(q, ldq, k, ldk, v, ldv, o, ldo, d_o, ld_do, dq, lddq, dk, lddk, dv, lddv, n_win, T, H, scale, \
                                             dbias_q, dbias_k, dbias_v, s)
  if (dv != nullptr) {
    if (hd_qk == 64 && hd_v == 64) IBM_BWD_LONG(64, 64, true);
    if (hd_qk == 48 && hd_v == 48) IBM_BWD_LONG(48, 48, true);
    if (hd_qk == 32 && hd_v == 32) IBM_BWD_LONG(32, 32, true);
  } else {
    IBM_CHECK_ARG(dbias_v == nullptr, "attention_bwd_long: dbias_v without dv");
    // the CoM blend of the TransformerBaseline (SimpleAttention, TransformerBaseline.py:51-70): the values are an input
    if (hd_v == 8) {
      if (hd_qk == 112) IBM_BWD_LONG(112, 8, false);
      if (hd_qk == 64) IBM_BWD_LONG(64, 8, false);
      if (hd_qk == 80) IBM_BWD_LONG(80, 8, false);
      if (hd_qk == 96) IBM_BWD_LONG(96, 8, false);
      if (hd_qk == 128) IBM_BWD_LONG(128, 8, false);
    }
  }
#undef IBM_BWD_LONG
  set_error("attention_bwd_long: unsupported (hd_qk, hd_v, dv) = (%d, %d, %s); supported (64,64) (48,48) (32,32) with dv, ({64,80,96,112,128},8) without",
            hd_qk, hd_v, dv ? "yes" : "no");
  return IBM_E_UNSUPPORTED;
}
