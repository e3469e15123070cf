// Persistent, warp-specialised bf16 GEMM for sm_100a: TMA-fed tcgen05.mma with fp32 accumulators
// in TMEM (double-buffered so the epilogue of tile i overlaps the main loop of tile i+1), fused
// bias / activation / residual / activation-gradient epilogue, TMA store (or TMA reduce-add for
// split-K weight gradients).
//
// Replaces the cuBLAS sgemm + separate bias/activation kernels behind
//   nn.Linear  — /root/reference/src/models/FeedForwardRegressionBaseline.py:73,113,
//                /root/reference/src/models/Groundlink.py:51-62,
//                /root/reference/src/models/TransformerBaseline.py:12-18,91 (and their autograd
//                backward: dgrad = dY·W, wgrad = dYᵀ·X)
//   nn.Conv1d  — /root/reference/src/models/Groundlink.py:41 (taps > 1: implicit GEMM over row-shifted A)
//
// Roles (384 threads, 1 CTA/SM): warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane),
// warp 2 = TMEM allocator, warps 4-11 = epilogue.  Each epilogue warp is an independent pipeline over
// its own 32 accumulator rows (TMEM lane quadrant) and every other 128-byte column chunk: TMEM →
// registers → its private swizzled staging rows → its own 32-row TMA store, with its own TMA-fed ring
// of aux (residual / saved-activation) tiles — no block-wide barrier anywhere in the epilogue.
// Tile 128 x BN x 64 per CTA; UMMA 128 x BN x 16 (cta_group::1) or 256 x BN x 16 across a CTA pair
// (cta_group::2); operand tiles in SWIZZLE_128B layout.
#include <cuda.h>

#include <stdlib.h>

#include <mutex>

#include "common.cuh"
#include "sm100_ptx.cuh"
#include "tma_host.cuh"

namespace ibm {
namespace gemm {

using namespace ptx;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;      // 64 bf16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int kThreads = 384;      // 4 control warps (TMA, MMA, TMEM alloc, spare) + 8 epilogue warps
constexpr int kEpiWarps = 8;
constexpr int kEpiWarp0 = 4;
constexpr int kStageA = BLOCK_M * BLOCK_K * 2;          // 16 KB
constexpr int kWarpStage = 32 * 128;                    // one epilogue warp's staging tile: 32 rows x 128 B = 4 KB
constexpr int kSmemCap = 227 * 1024;                    // opt-in dynamic shared memory per CTA on sm_100
constexpr int kOutBufsPerWarp = 1;                      // output staging tiles per epilogue warp

// CG = CTAs per MMA (cta_group): 1 = one 128 x BN tile per CTA; 2 = a CTA pair computes a 256 x BN tile, each CTA
// holding its own 128 rows of A and HALF of the B tile (BN / 2 rows), which halves the B traffic through shared memory
// (at 128 x 256 with cta_group::1 the operand reads + TMA writes exceed the 128 B/clk shared-memory port: 64 % tensor
// pipe, profiles/r01a; the pair brings it under the port limit).
// NT = column tiles per work item (1 or 2).  With NT = 2 a work item is a 256 x 2*BN "supertile": one A tile feeds both
// accumulators, so the operand bytes pulled through the L2 -> SM fabric per FLOP drop by a quarter.  All well-shaped
// launches measured 9.6-9.9 TB/s of L2 -> SM reads at 68-69 % tensor pipe, whatever their K, stage count or epilogue
// (profiles/r01b): that fabric, not the tensor pipe, paces a 256 x 256 tile.  The price: both TMEM accumulators belong to
// one work item, so its epilogue no longer overlaps the next main loop — worth it when the main loop is long (K >= 1024).
// AS = A-stationary (short K): the whole 128 x K operand block of a row block (K <= 512: eight 16 KB slots) stays in shared
// memory while the CTA pair walks ALL column tiles of that row block, so only B streams through the ring — half the
// L2 -> SM bytes of a 256 x 256 tile, with the epilogue still overlapped (both TMEM accumulators alternate as usual).
constexpr int kASlots = 8;
template <int BN, bool AUX, int CG, int NT = 1, bool AS = false>
struct Cfg {
  static constexpr int kStageB = NT * (BN / CG) * BLOCK_K * 2;
  // per epilogue warp: output staging tiles (double-buffered; single when the aux ring also needs room) and a
  // 2-deep ring of aux tiles, each loaded one of the warp's chunks ahead
  static constexpr int kOutBufs = kOutBufsPerWarp;
  // supertiles keep ONE aux tile per warp: it is copied to registers as soon as it lands and the next load is issued
  // into the same tile at once, so the load flies during the chunk's arithmetic and store (an operand stage is worth
  // more than the second aux tile there).  Measured alternatives (profiles/r02b_gemm_experiments.md): two aux tiles paid
  // for by storing the rows straight from registers (390 vs 364 us, FFN-2 forward), per-thread cp.async or plain global
  // loads of the aux rows (393 / 470 us) — all slower.
  static constexpr int kAuxBufs = AUX ? (NT == 2 ? 1 : 2) : 0;
  static constexpr int kEpiBytes = kEpiWarps * (kOutBufs + kAuxBufs) * kWarpStage;
  static constexpr int kFixed = 1024 /*align slack*/ + kEpiBytes + 512 /*mbarriers, tmem slot*/ + (AS ? kASlots * kStageA : 0);
  static constexpr int kFit = (kSmemCap - kFixed) / ((AS ? 0 : kStageA) + kStageB);
  static constexpr int kStages = kFit > 8 ? 8 : kFit;                  // operand ring: whatever is left, at most 8
  static_assert(kStages >= 2, "operand ring needs at least two stages");
  static constexpr uint32_t kTmemCols = (2 * BN < 32) ? 32 : 2 * BN;
  static constexpr int kSmem = kFixed + kStages * ((AS ? 0 : kStageA) + kStageB);
  static constexpr int kSlotsA = AS ? kASlots : kStages;               // A tiles resident in shared memory
};

struct Args {
  int64_t M, N;
  int32_t kb_total;        // number of 64-wide k blocks (all taps)
  int32_t kb_per_tap;      // k blocks per tap (== kb_total when taps == 1)
  int32_t kb_per_split;
  int32_t splits;
  int32_t tiles_m, tiles_n;
  int32_t a_mn, b_mn;
  int32_t act, aux_mode;
  const float* bias;
  const __nv_bfloat16* aux;
  int64_t ldaux;
  float* colsum;           // optional fp32[N]: += column sums of the (bf16-rounded) output — a bias gradient
  uint8_t* mask;           // optional sign bitmask [M][ldmask bytes], bit (c & 7) of byte c >> 3 <-> column c
  int64_t ldmask;
  int32_t mask_mode;       // 1: write (output > 0) after the activation; 2: zero the outputs whose bit is clear
  int32_t fp2;             // bias adds as packed fp32 (FADD2); IBM_GEMM_FP2=0 keeps the scalar adds for A/B runs
  int32_t pf_aux;          // aux tiles are pulled into L2 ahead of the epilogue: 0 no, 1 by TMA prefetches of the producer, 2 by warp 3
  int32_t stagger;         // supertiles: start on accumulator 0 while accumulator 1 is still being drained
  int32_t reverse;         // work items are taken from the last one down (ibm_set_walk_order); never with A-stationary
};

__device__ __forceinline__ void advance(int& stage, uint32_t& phase, int nstages) {
  if (++stage == nstages) { stage = 0; phase ^= 1u; }
}


// ---- epilogue math, specialised at compile time on the activation (no per-element switch) ----------
template <int ACT> __device__ __forceinline__ float act_t(float x) { return act_apply(x, ACT); }
template <int ACT> __device__ __forceinline__ float dact_t(float y) { return act_grad_from_output(y, ACT); }

__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// v holds acc + bias on entry
template <int ACT, int PT>
__device__ __forceinline__ void epi_plain(float (&v)[PT]) {
#pragma unroll
  for (int j = 0; j < PT; ++j) v[j] = act_t<ACT>(v[j]);
}
template <int PT>
__device__ __forceinline__ void epi_dispatch_plain(float (&v)[PT], int act) {
  switch (act) {
    case IBM_ACT_NONE: break;
    case IBM_ACT_RELU: epi_plain<IBM_ACT_RELU, PT>(v); break;
    case IBM_ACT_SIGMOID: epi_plain<IBM_ACT_SIGMOID, PT>(v); break;
    case IBM_ACT_TANH: epi_plain<IBM_ACT_TANH, PT>(v); break;
    case IBM_ACT_ELU: epi_plain<IBM_ACT_ELU, PT>(v); break;
    default: epi_plain<IBM_ACT_SILU, PT>(v); break;
  }
}
// MODE 1: out = act(acc + bias) + aux;  MODE 2: out = (acc + bias) * act'(aux).  aux: bf16, 8 per 16-byte piece of
// this thread's swizzled 128-byte row.
template <int ACT, int MODE, int PT>
__device__ __forceinline__ void epi_aux(float (&v)[PT], uint32_t xrow, int rsw, const uint4* ax) {
#pragma unroll
  for (int jj = 0; jj < PT / 8; ++jj) {
    const uint4 u = ax != nullptr ? ax[jj] : ld_shared_v4(xrow + ((jj ^ rsw) << 4));
    float y[8];
    float2 t;
    t = unpack_bf16x2(u.x); y[0] = t.x; y[1] = t.y;
    t = unpack_bf16x2(u.y); y[2] = t.x; y[3] = t.y;
    t = unpack_bf16x2(u.z); y[4] = t.x; y[5] = t.y;
    t = unpack_bf16x2(u.w); y[6] = t.x; y[7] = t.y;
    if constexpr (MODE == 1 && ACT == IBM_ACT_NONE) {      // residual add: packed fp32 adds
#pragma unroll
      for (int e = 0; e < 8; e += 2) {
        const float2 r = __fadd2_rn(make_float2(v[8 * jj + e], v[8 * jj + e + 1]), make_float2(y[e], y[e + 1]));
        v[8 * jj + e] = r.x; v[8 * jj + e + 1] = r.y;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float x = v[8 * jj + e];
        v[8 * jj + e] = MODE == 1 ? act_t<ACT>(x) + y[e] : x * dact_t<ACT>(y[e]);
      }
    }
  }
}
template <int PT>
__device__ __forceinline__ void epi_dispatch_aux(float (&v)[PT], uint32_t xrow, int rsw, int act, int mode, const uint4* ax) {
  if constexpr (PT % 8 == 0) {
    if (mode == 1) {
      switch (act) {
        case IBM_ACT_NONE: epi_aux<IBM_ACT_NONE, 1, PT>(v, xrow, rsw, ax); break;
        case IBM_ACT_RELU: epi_aux<IBM_ACT_RELU, 1, PT>(v, xrow, rsw, ax); break;
        default: epi_aux<IBM_ACT_ELU, 1, PT>(v, xrow, rsw, ax); break;
      }
    } else {
      switch (act) {
        case IBM_ACT_NONE: epi_aux<IBM_ACT_NONE, 2, PT>(v, xrow, rsw, ax); break;
        case IBM_ACT_RELU: epi_aux<IBM_ACT_RELU, 2, PT>(v, xrow, rsw, ax); break;
        case IBM_ACT_SIGMOID: epi_aux<IBM_ACT_SIGMOID, 2, PT>(v, xrow, rsw, ax); break;
        case IBM_ACT_TANH: epi_aux<IBM_ACT_TANH, 2, PT>(v, xrow, rsw, ax); break;
        default: epi_aux<IBM_ACT_ELU, 2, PT>(v, xrow, rsw, ax); break;
      }
    }
  }
}

// MM: the sign-bitmask mode as a compile-time constant (0 none, 1 write, 2 gate) for the hot bf16 shapes, so that the
// plain epilogue does not carry the registers of the two mask paths (ptxas: every runtime-mask variant sits at the
// 168-register cap with spills); -1 = read args.mask_mode at run time.
template <int BN, bool kOutF32, bool kAccum, bool kAux, int CG, int NT, bool kAS, int MM = -1>
__global__ void __launch_bounds__(kThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmX, const Args args) {
  using C = Cfg<BN, kAux, CG, NT, kAS>;
  static_assert(NT == 1 || (NT == 2 && CG == 2 && BN == 256), "supertiles: CTA pairs, 256-wide tiles");
  static_assert(!kAS || (CG == 2 && NT == 1 && !kAux && !kAccum), "A-stationary: CTA pairs, plain epilogue, no split-K");
  constexpr bool kAuxRegs = NT == 2;                 // aux values reach the arithmetic through registers
  static_assert(CG == 1 || BN >= 128, "a CTA pair splits B into two halves of at least one 64-wide swizzle atom");
  static_assert(!kAux || (!kOutF32 && !kAccum), "TMA-staged aux tiles exist for bf16 outputs only");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem_a + C::kSlotsA * kStageA;
  uint8_t* smem_out = smem_b + C::kStages * C::kStageB;              // [8 warps][kOutBufs] x 4 KB, 1024-aligned
  uint8_t* smem_aux = smem_out + kEpiWarps * C::kOutBufs * kWarpStage;   // [8 warps][kAuxBufs] x 4 KB
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_aux + kEpiWarps * C::kAuxBufs * kWarpStage);
  uint64_t* empty_bar = full_bar + C::kStages;
  uint64_t* tfull_bar = empty_bar + C::kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* aux_bar = tempty_bar + 2;                                // [8 warps][2]
  uint64_t* afull_bar = aux_bar + kEpiWarps * 2;                     // [kASlots] A-stationary: slot filled / slot free
  uint64_t* aempty_bar = afull_bar + kASlots;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty_bar + kASlots);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mask_mode = MM >= 0 ? MM : args.mask_mode;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmD);
    prefetch_tmap(&tmX);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < C::kStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    // the leader's MMA thread waits for the epilogue warps of BOTH CTAs of a pair before reusing an accumulator
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], CG * kEpiWarps); }
    for (int i = 0; i < kEpiWarps * 2; ++i) mbar_init(&aux_bar[i], 1);
    for (int i = 0; i < kASlots; ++i) { mbar_init(&afull_bar[i], 1); mbar_init(&aempty_bar[i], 1); }
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (CG == 2) tmem_alloc_pair<C::kTmemCols>(tmem_slot);
    else tmem_alloc<C::kTmemCols>(tmem_slot);
  }
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all();      // peer barriers are initialised before any remote arrive / TMA completion
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // work item = (row block of CG*128 rows, column tile, k split); a pair walks the same list, CTA `rank` owning
  // rows [rank*128, +128) of the row block and B rows [rank*BN/2, +BN/2) of the column tile
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
  const int worker = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int n_workers = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  // work w = split * n_tiles + tile: the work items in flight together are the tiles of ONE k split, so they stream the
  // same rows of both operands at the same pace and share them through L2 (split-K weight gradients)
  const int n_tiles = args.tiles_m * args.tiles_n;                       // tiles_m counts CG*128-row blocks
  const int total_work = n_tiles * args.splits;
  constexpr int BN_LOAD = BN / CG;
  // position in the worker's round-robin sequence -> work item: descending when args.reverse (the consumer of a tensor
  // then starts on the rows its producer wrote last, which are still in L2)
  auto item_of = [&](int w) { return args.reverse ? total_work - 1 - w : w; };

  if (warp == 0) {
    // ===================================== TMA producer ======================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t tx_bytes = CG * (kStageA + C::kStageB);     // the pair's loads all complete on the leader's barrier
      const bool prefetch_aux = kAux && args.pf_aux == 1;
      if constexpr (kAS) {
        // row block by row block: refill the A slots (each as soon as the previous block's last column tile has consumed
        // it), then stream B for every column tile
        uint32_t gen = 0;
        for (int rb = worker; rb < args.tiles_m; rb += n_workers, ++gen) {
          const int m0 = (rb * CG + rank) * BLOCK_M;
          for (int kb = 0; kb < args.kb_total; ++kb) {
            mbar_wait(&aempty_bar[kb], (gen & 1u) ^ 1u);
            if (rank == 0) mbar_arrive_expect_tx(&afull_bar[kb], CG * kStageA);
            uint8_t* sa = smem_a + kb * kStageA;
            if (!args.a_mn) {
              tma_load_2d_pair(sa, &tmA, &afull_bar[kb], kb * BLOCK_K, m0);
            } else {
#pragma unroll
              for (int i = 0; i < BLOCK_M / 64; ++i) tma_load_2d_pair(sa + i * (BLOCK_K * 128), &tmA, &afull_bar[kb], m0 + 64 * i, kb * BLOCK_K);
            }
          }
          for (int ti = 0; ti < args.tiles_n; ++ti) {
            // pairs start at different column tiles: all of them streaming the same B tile in lockstep would hammer
            // the same L2 lines
            const int tn = (ti + worker) % args.tiles_n;
            const int nb0 = tn * BN + rank * BN_LOAD;
            for (int kb = 0; kb < args.kb_total; ++kb) {
              mbar_wait(&empty_bar[stage], phase ^ 1u);
              if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], CG * C::kStageB);
              uint8_t* sb = smem_b + stage * C::kStageB;
              if (!args.b_mn) {
                tma_load_2d_pair(sb, &tmB, &full_bar[stage], kb * BLOCK_K, nb0);
              } else {
#pragma unroll
                for (int i = 0; i < BN_LOAD / 64; ++i) tma_load_2d_pair(sb + i * (BLOCK_K * 128), &tmB, &full_bar[stage], nb0 + 64 * i, kb * BLOCK_K);
              }
              advance(stage, phase, C::kStages);
            }
          }
        }
      } else
      for (int w = worker; w < total_work; w += n_workers) {
        const int split = item_of(w) / n_tiles;
        const int tile = item_of(w) - split * n_tiles;
        const int tn = tile % args.tiles_n, tm = tile / args.tiles_n;
        const int m0 = (tm * CG + rank) * BLOCK_M, n0 = tn * NT * BN;
        const int nb0 = n0 + rank * BN_LOAD;                      // first B row this CTA loads (per column tile: + t*BN)
        const int kb0 = split * args.kb_per_split;
        const int kb1 = min(args.kb_total, kb0 + args.kb_per_split);
        if (prefetch_aux) {
          // round-1 behaviour (IBM_GEMM_PFAUX=1, off by default: measured 4 % slower): the epilogue of this tile runs ~1.5
          // tile-times from now, pull its aux tile into L2 so the epilogue's one-chunk-ahead TMA loads see L2 latency
          for (int c = 0; c < NT * BN && n0 + c < args.N; c += 64)
            for (int r = 0; r < BLOCK_M; r += 32) tma_prefetch_l2_2d(&tmX, n0 + c, m0 + r);
        }
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], tx_bytes);
          uint8_t* sa = smem_a + stage * kStageA;
          uint8_t* sb = smem_b + stage * C::kStageB;
          const int tap = kb / args.kb_per_tap;
          const int k0a = (kb - tap * args.kb_per_tap) * BLOCK_K;      // k coordinate inside A
          const int k0b = kb * BLOCK_K;                                 // k coordinate inside B
          auto load = [&](void* dst, const CUtensorMap* tm_, int c0, int c1) {
            if constexpr (CG == 2) tma_load_2d_pair(dst, tm_, &full_bar[stage], c0, c1);
            else tma_load_2d(dst, tm_, &full_bar[stage], c0, c1);
          };
          if (!args.a_mn) {
            load(sa, &tmA, k0a, m0 + tap);
          } else {
#pragma unroll
            for (int i = 0; i < BLOCK_M / 64; ++i) load(sa + i * (BLOCK_K * 128), &tmA, m0 + 64 * i, k0a);
          }
#pragma unroll
          for (int t = 0; t < NT; ++t) {
            uint8_t* sbt = sb + t * (C::kStageB / NT);
            if (!args.b_mn) {
              load(sbt, &tmB, k0b, nb0 + t * BN);
            } else {
#pragma unroll
              for (int i = 0; i < BN_LOAD / 64; ++i) load(sbt + i * (BLOCK_K * 128), &tmB, nb0 + t * BN + 64 * i, k0b);
            }
          }
          advance(stage, phase, C::kStages);
        }
      }
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer =======================================
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc_bf16(CG * BLOCK_M, BN, args.a_mn, args.b_mn);
      // K-major: 8-row groups are 1024 B apart (SBO); LBO unused.  MN-major: 64-wide MN atoms are
      // BLOCK_K*128 B apart (LBO), 8-k-row groups 1024 B apart (SBO).
      const uint32_t a_lbo = args.a_mn ? BLOCK_K * 128 : 0, b_lbo = args.b_mn ? BLOCK_K * 128 : 0;
      const uint32_t a_kstep = args.a_mn ? UMMA_K * 128 : UMMA_K * 2;
      const uint32_t b_kstep = args.b_mn ? UMMA_K * 128 : UMMA_K * 2;
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      if constexpr (kAS) {
        uint32_t gen = 0;
        for (int rb = worker; rb < args.tiles_m; rb += n_workers, ++gen) {
          for (int tn = 0; tn < args.tiles_n; ++tn) {
            mbar_wait(&tempty_bar[as], aphase ^ 1u);
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
            for (int kb = 0; kb < args.kb_total; ++kb) {
              if (tn == 0) mbar_wait(&afull_bar[kb], gen & 1u);
              mbar_wait(&full_bar[stage], phase);
              tc_fence_after();
              const uint32_t sa = smem_u32(smem_a + kb * kStageA);
              const uint32_t sb = smem_u32(smem_b + stage * C::kStageB);
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k)
                umma_bf16_pair(tmem_d, make_smem_desc_sw128(sa + k * a_kstep, a_lbo, 1024),
                               make_smem_desc_sw128(sb + k * b_kstep, b_lbo, 1024), idesc, (kb > 0 || k > 0) ? 1u : 0u);
              umma_commit_pair(&empty_bar[stage]);
              if (tn == args.tiles_n - 1) umma_commit_pair(&aempty_bar[kb]);   // last use of this A slot for the row block
              advance(stage, phase, C::kStages);
            }
            umma_commit_pair(&tfull_bar[as]);
            if (++as == 2) { as = 0; aphase ^= 1u; }
          }
        }
      } else
      for (int w = worker; w < total_work; w += n_workers) {
        const int split = item_of(w) / n_tiles;
        const int kb0 = split * args.kb_per_split;
        const int kb1 = min(args.kb_total, kb0 + args.kb_per_split);
        // NT == 1: accumulator `as` (the other one is being drained).  NT == 2: both accumulators, one per column tile.
        mbar_wait(&tempty_bar[as], aphase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
        auto issue_kblock = [&](int st, int t, bool first) {        // the four k steps of one 64-wide k block into accumulator t
          const uint32_t sa = smem_u32(smem_a + st * kStageA);
          const uint32_t sb = smem_u32(smem_b + st * C::kStageB) + t * (C::kStageB / NT);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t adesc = make_smem_desc_sw128(sa + k * a_kstep, a_lbo, 1024);
            const uint64_t bdesc = make_smem_desc_sw128(sb + k * b_kstep, b_lbo, 1024);
            if constexpr (CG == 2) umma_bf16_pair(tmem_d + t * BN, adesc, bdesc, idesc, (!first || k > 0) ? 1u : 0u);
            else umma_bf16(tmem_d + t * BN, adesc, bdesc, idesc, (!first || k > 0) ? 1u : 0u);
          }
        };
        int kb = kb0;
        if constexpr (NT == 2) {
          // Staggered start: the epilogue drains accumulator 0 first, then accumulator 1.  As soon as accumulator 0 is free
          // the first k blocks of THIS item are multiplied into it (their operand stages are kept), and when accumulator 1
          // follows, the same stages feed it and are released — up to kStages k blocks of tensor work hide the second half
          // of the previous item's epilogue, which a supertile otherwise exposes completely.
          const int pre = args.stagger ? min(C::kStages, kb1 - kb0) : 0;
          int st = stage;
          uint32_t ph = phase;
          for (int j = 0; j < pre; ++j) {
            mbar_wait(&full_bar[st], ph);
            tc_fence_after();
            issue_kblock(st, 0, j == 0);
            advance(st, ph, C::kStages);
          }
          mbar_wait(&tempty_bar[1], aphase ^ 1u);
          tc_fence_after();
          for (int j = 0; j < pre; ++j) {
            issue_kblock(stage, 1, j == 0);
            umma_commit_pair(&empty_bar[stage]);
            advance(stage, phase, C::kStages);
          }
          kb += pre;
        }
        for (; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem_a + stage * kStageA);
          const uint32_t sb = smem_u32(smem_b + stage * C::kStageB);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t adesc = make_smem_desc_sw128(sa + k * a_kstep, a_lbo, 1024);
#pragma unroll
            for (int t = 0; t < NT; ++t) {
              const uint64_t bdesc = make_smem_desc_sw128(sb + t * (C::kStageB / NT) + k * b_kstep, b_lbo, 1024);
              if constexpr (CG == 2) umma_bf16_pair(tmem_d + t * BN, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
              else umma_bf16(tmem_d + t * BN, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            }
          }
          // frees the smem slot (in both CTAs of a pair) when these MMAs retire
          if constexpr (CG == 2) umma_commit_pair(&empty_bar[stage]);
          else umma_commit(&empty_bar[stage]);
          advance(stage, phase, C::kStages);
        }
        // accumulator(s) complete → epilogue (of both CTAs)
        if constexpr (CG == 2) umma_commit_pair(&tfull_bar[as]);
        else umma_commit(&tfull_bar[as]);
        if constexpr (NT == 2) {
          umma_commit_pair(&tfull_bar[1]);
          aphase ^= 1u;                             // `as` stays 0: every work item uses both accumulators
        } else {
          if (++as == 2) { as = 0; aphase ^= 1u; }
        }
      }
    }
  } else if (warp == 3) {
    // ================================== aux prefetcher (optional) =============================
    // pulls the aux tile of work item i into L2 with plain prefetches (LSU path: nothing is queued in the TMA unit ahead of
    // the operand loads) when the accumulators of item i-1 complete, i.e. one main loop before the epilogue reads it
    if constexpr (kAux && !kAS) {
      if (args.pf_aux == 2) {
        int as = 0;
        uint32_t aphase = 0;
        constexpr int kLinesPerRow = NT * BN * 2 / 128;
        for (int w = worker; w < total_work; w += n_workers) {
          const int tile = item_of(w) % n_tiles;
          const int tn = tile % args.tiles_n, tm = tile / args.tiles_n;
          const int64_t m0 = (int64_t)(tm * CG + rank) * BLOCK_M;
          const int n0 = tn * NT * BN;
          for (int i = lane; i < BLOCK_M * kLinesPerRow; i += 32) {
            const int64_t row = m0 + i / kLinesPerRow;
            const int col = n0 + (i % kLinesPerRow) * 64;
            if (row < args.M && col < args.N) asm volatile("prefetch.global.L2 [%0];" ::"l"(args.aux + row * args.ldaux + col));
          }
          mbar_wait(&tfull_bar[as], aphase);          // item w's main loop is over: the next item's starts now
          if (NT == 2) { aphase ^= 1u; } else if (++as == 2) { as = 0; aphase ^= 1u; }
        }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ======================================= epilogue ========================================
    // warp (q, half): TMEM lanes [32q, +32) = tile rows [32q, +32); column chunks half, half+2, … of the tile.
    // A chunk is one 128-byte staging row per thread: 64 bf16 or 32 fp32 columns.
    constexpr int CW = kOutF32 ? 32 : 64;           // columns per chunk == columns per thread per chunk
    constexpr int PT = CW;
    static_assert(BN >= CW, "an epilogue chunk must not be wider than the accumulator tile");
    const int ew = warp - kEpiWarp0;                // 0..7
    const int q = warp & 3;                         // TMEM lane quadrant this warp may access
    const int half = ew >> 2;
    const int rsw = lane & 7;                       // SWIZZLE_128B: 16-byte piece j of row r lives at piece j ^ (r & 7)
    uint8_t* my_out = smem_out + ew * (C::kOutBufs * kWarpStage);
    uint8_t* my_aux = smem_aux + ew * (C::kAuxBufs * kWarpStage);
    uint64_t* my_aux_bar = aux_bar + ew * 2;
    int as = 0, ob = 0;
    uint32_t aphase = 0;
    int xg = 0;                                     // chunks consumed so far by this warp (aux ring position)
    int pw = worker, pts = 0, pch = half;           // prefetch cursor: (work item, column tile, chunk) of this warp's next aux load
    auto chunks_of = [&](int w, int ts) {
      const int n0w = (((item_of(w) % n_tiles) % args.tiles_n) * NT + ts) * BN;
      return ((int)max((int64_t)0, min((int64_t)BN, args.N - n0w)) + CW - 1) / CW;
    };
    auto issue_aux = [&](int buf) {                 // lane 0 only
      while (pw < total_work && pch >= chunks_of(pw, pts)) {
        pch = half;
        if (++pts == NT) { pts = 0; pw += n_workers; }
      }
      if (pw >= total_work) return;
      const int t2 = item_of(pw) % n_tiles;
      mbar_arrive_expect_tx(&my_aux_bar[buf], kWarpStage);
      tma_load_2d(my_aux + buf * kWarpStage, &tmX, &my_aux_bar[buf], ((t2 % args.tiles_n) * NT + pts) * BN + pch * CW,
                  ((t2 / args.tiles_n) * CG + rank) * BLOCK_M + q * 32);
      pch += 2;
    };
    if (kAux && lane == 0) {
      issue_aux(0);
      if (C::kAuxBufs == 2) issue_aux(1);
    }
    auto release_tmem = [&]() {                     // this warp has read everything it needs from accumulator `as`
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CG == 2) mbar_arrive_cluster(&tempty_bar[as], 0);
        else mbar_arrive(&tempty_bar[as]);
      }
    };
    // the tile sequence of this worker: round-robin work items (and their NT column tiles), or — A-stationary — every
    // column tile of its round-robin row blocks (w1 steps through one row block's tiles, w0 from row block to row block)
    const int w_step0 = kAS ? n_workers * args.tiles_n : n_workers;
    const int w_inner = kAS ? args.tiles_n : 1;
    for (int w0 = kAS ? worker * args.tiles_n : worker; w0 < total_work; w0 += w_step0)
    for (int wi = w0; wi < w0 + w_inner; ++wi)
    for (int tsub = 0; tsub < NT; ++tsub) {           // column tile inside the supertile: accumulator `as` == tsub when NT == 2
      const int w = kAS ? w0 + (wi - w0 + worker) % args.tiles_n : item_of(wi);      // A-stationary: rotated column order (see producer)
      const int tile = w % n_tiles;
      const int tn = tile % args.tiles_n, tm = tile / args.tiles_n;
      const int m0 = (tm * CG + rank) * BLOCK_M + q * 32, n0 = (tn * NT + tsub) * BN;       // this warp's first row
      const int n_valid = (int)max((int64_t)0, min((int64_t)BN, args.N - n0));              // 0: the tile lies beyond N
      const int n_chunks = (n_valid + CW - 1) / CW;

      // ReLU-derivative bitmask of this thread's row (mask_mode 2): 8 bytes per chunk, fetched before the accumulator wait
      // so that the (uncoalesced, tiny) loads fly under the main loop
      uint2 mbits[(BN / CW + 1) / 2];
      if constexpr (!kOutF32 && !kAux) {
        if (mask_mode == 2) {
          const int64_t row = (int64_t)m0 + lane;
#pragma unroll
          for (int i = 0; i < (BN / CW + 1) / 2; ++i) {
            const int ch = half + 2 * i;
            mbits[i] = make_uint2(0u, 0u);
            if (ch < n_chunks && row < args.M) mbits[i] = __ldg(reinterpret_cast<const uint2*>(args.mask + row * args.ldmask + ((n0 + ch * CW) >> 3)));
          }
        }
      }
      mbar_wait(&tfull_bar[as], aphase);
      tc_fence_after();
      const uint32_t tmem_acc = tmem_base + (uint32_t)(as * BN) + ((uint32_t)(q * 32) << 16);
      if (half >= n_chunks) release_tmem();         // narrow tile: nothing for this warp, but the MMA warp counts it

      for (int ch = half; ch < n_chunks; ch += 2) {
        float v[PT];
#pragma unroll
        for (int i = 0; i < PT / 32; ++i) tmem_ld_32x32(tmem_acc + ch * CW + i * 32, reinterpret_cast<uint32_t*>(v) + i * 32);
        const int c0 = n0 + ch * CW;               // global column of the chunk
        const int xb = C::kAuxBufs == 2 ? (xg & 1) : 0;
        const uint32_t xph = C::kAuxBufs == 2 ? (uint32_t)((xg >> 1) & 1) : (uint32_t)(xg & 1);
        uint4 ax[PT / 8];                          // this thread's aux row piece when it travels through registers
        if (kAux) {
          mbar_wait(&my_aux_bar[xb], xph);         // this chunk's aux tile has landed
          if constexpr (NT == 2) {
            // single aux tile: move it to registers and put the next load in flight right away
            const uint32_t xr = smem_u32(my_aux + lane * 128);
#pragma unroll
            for (int j = 0; j < PT / 8; ++j) ax[j] = ld_shared_v4(xr + ((j ^ rsw) << 4));
            __syncwarp();
            if (lane == 0) issue_aux(0);
          }
        }
        tmem_ld_wait();
        if (ch + 2 >= n_chunks) release_tmem();

        if (!kAccum) {
          if (args.bias != nullptr) {
            if (c0 + PT <= args.N) {
              const float4* b4 = reinterpret_cast<const float4*>(args.bias + c0);
#pragma unroll
              for (int j = 0; j < PT / 4; ++j) {       // packed fp32 adds (FADD2): half the issue slots of the bias add
                const float4 b = __ldg(b4 + j);
                if (args.fp2) {
                  const float2 lo = __fadd2_rn(make_float2(v[4 * j], v[4 * j + 1]), make_float2(b.x, b.y));
                  const float2 hi = __fadd2_rn(make_float2(v[4 * j + 2], v[4 * j + 3]), make_float2(b.z, b.w));
                  v[4 * j] = lo.x; v[4 * j + 1] = lo.y; v[4 * j + 2] = hi.x; v[4 * j + 3] = hi.y;
                } else {
                  v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < PT; ++j) v[j] += (c0 + j < args.N) ? __ldg(args.bias + c0 + j) : 0.f;
            }
          }
          if (kAux) {
            epi_dispatch_aux<PT>(v, smem_u32(my_aux + xb * kWarpStage + lane * 128), rsw, args.act, args.aux_mode, kAuxRegs ? ax : nullptr);
          } else {
            // fp32 aux_mode 2 (below): (acc + bias) * act'(aux), no act; bf16 kernels without kAux never see aux
            if (!kOutF32 || args.aux_mode != 2) epi_dispatch_plain<PT>(v, args.act);
            if constexpr (!kOutF32) {
              if (mask_mode == 1) {
                // the sign pattern of the (post-activation) outputs: what the dgrad of this layer needs instead of the
                // whole activation matrix (1 bit instead of 16 per element)
                // outputs are >= 0 here (ReLU): x > 0  <=>  the sign bit of -bits(x) is set; a funnel shift pushes that
                // bit into the word, two instructions per element
                uint32_t lo = 0, hi = 0;
#pragma unroll
                for (int j = 31; j >= 0; --j) {
                  lo = __funnelshift_l((uint32_t)(-(int32_t)__float_as_uint(fmaxf(v[j], 0.f))), lo, 1);
                  hi = __funnelshift_l((uint32_t)(-(int32_t)__float_as_uint(fmaxf(v[32 + j], 0.f))), hi, 1);
                }
                const int64_t row = (int64_t)m0 + lane;
                if (row < args.M && c0 + PT <= args.N) *reinterpret_cast<uint2*>(args.mask + row * args.ldmask + (c0 >> 3)) = make_uint2(lo, hi);
              } else if (mask_mode == 2) {
                const uint2 mb = mbits[(ch - half) >> 1];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  if (!((mb.x >> j) & 1u)) v[j] = 0.f;
                  if (!((mb.y >> j) & 1u)) v[32 + j] = 0.f;
                }
              }
            }
            if (args.aux_mode != 0) {
              // fp32-output fallback: aux read straight from global memory (not on the training path)
              const int64_t row = (int64_t)m0 + lane;
              const __nv_bfloat16* ap = args.aux + row * args.ldaux + c0;
#pragma unroll
              for (int j = 0; j < PT; ++j) {
                const float y = (row < args.M && c0 + j < args.N) ? __bfloat162float(ap[j]) : 0.f;
                v[j] = args.aux_mode == 1 ? v[j] + y : v[j] * act_grad_from_output(y, args.act);
              }
            }
          }
        }
        // the staging tile `ob` must no longer be read by the store issued kOutBufs chunks ago
        if (lane == 0) tma_wait_group_read<C::kOutBufs - 1>();
        __syncwarp();
        const uint32_t srow = smem_u32(my_out + ob * kWarpStage + lane * 128);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          uint4 pk;
          if (kOutF32) {
            pk = make_uint4(__float_as_uint(v[4 * jj]), __float_as_uint(v[4 * jj + 1]), __float_as_uint(v[4 * jj + 2]),
                            __float_as_uint(v[4 * jj + 3]));
          } else {
            pk = make_uint4(pack_bf16x2(v[8 * jj], v[8 * jj + 1]), pack_bf16x2(v[8 * jj + 2], v[8 * jj + 3]),
                            pack_bf16x2(v[8 * jj + 4], v[8 * jj + 5]), pack_bf16x2(v[8 * jj + 6], v[8 * jj + 7]));
          }
          st_shared_v4(srow + ((jj ^ rsw) << 4), pk);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (kAccum) tma_reduce_add_2d(&tmD, my_out + ob * kWarpStage, c0, m0);
          else tma_store_2d(&tmD, my_out + ob * kWarpStage, c0, m0);
          tma_commit_group();
          if (kAux && NT == 1) issue_aux(xb);   // every lane is past its reads of aux tile xb
        }
        if constexpr (!kOutF32) {
          if (args.colsum != nullptr) {
            // bias gradient of the layer that produced this tensor: lane l sums columns 2l, 2l+1 of the staged
            // (rounded) 32 x 64 tile — conflict-free 4-byte reads of the swizzled rows — then two coalesced REDs
            const int rows = (int)min((int64_t)32, args.M - m0);
            const uint32_t sbase = smem_u32(my_out + ob * kWarpStage) + (lane & 3) * 4;
            float a0 = 0.f, a1 = 0.f;
#pragma unroll 8
            for (int r = 0; r < rows; ++r) {
              uint32_t u;
              asm volatile("ld.shared.u32 %0, [%1];" : "=r"(u) : "r"(sbase + r * 128 + (((lane >> 2) ^ (r & 7)) << 4)));
              a0 += __uint_as_float(u << 16);
              a1 += __uint_as_float(u & 0xffff0000u);
            }
            const int col = c0 + 2 * lane;
            if (col < args.N) atomicAdd(args.colsum + col, a0);
            if (col + 1 < args.N) atomicAdd(args.colsum + col + 1, a1);
          }
        }
        if (++ob == C::kOutBufs) ob = 0;
        ++xg;
      }
      if (++as == 2) { as = 0; aphase ^= 1u; }
    }
    if (lane == 0) tma_wait_group<0>();   // all global writes issued by this warp are complete
  }

  // ---- teardown ----
  tc_fence_before();
  if constexpr (CG == 2) cluster_sync_all();      // no CTA retires while its peer can still signal into it
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CG == 2) tmem_dealloc_pair<C::kTmemCols>(tmem_base);
    else tmem_dealloc<C::kTmemCols>(tmem_base);
  }
}

// ------------------------------------------- host side -------------------------------------------

template <int BN, bool F32, bool ACC, bool AUX, int CG, int NT = 1, bool AS = false, int MM = -1>
static int launch(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& d, const CUtensorMap& x, const Args& args, int grid,
                  cudaStream_t s) {
  static bool attr_set = false;     // per instantiation
  auto kern = gemm_kernel<BN, F32, ACC, AUX, CG, NT, AS, MM>;
  if (!attr_set) {
    IBM_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<BN, AUX, CG, NT, AS>::kSmem));
    attr_set = true;
  }
  if constexpr (CG == 1) {
    kern<<<grid, kThreads, Cfg<BN, AUX, CG, NT, AS>::kSmem, s>>>(a, b, d, x, args);
  } else {
    // CTA pairs: clusters of 2 along x so both CTAs of a pair sit on the two SMs of one TPC
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = Cfg<BN, AUX, CG, NT, AS>::kSmem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    IBM_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, a, b, d, x, args));
  }
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

// IBM_GEMM_CG=1 forces single-CTA MMAs everywhere (A/B measurements, tools/gemm_probe.py)
// IBM_GEMM_NT=1 disables the two-tile supertiles
static int forced_nt() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IBM_GEMM_NT");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v;
}
static int forced_cg() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IBM_GEMM_CG");
    v = (e && e[0] == '1') ? 1 : ((e && e[0] == '2') ? 2 : 0);
  }
  return v;
}

static int pick_bn(int64_t N) {
  const int cands[4] = {256, 128, 64, 32};
  for (int i = 0; i < 4; ++i) {
    const int bn = cands[i];
    const double eff = (double)N / (double)(ceil_div(N, bn) * bn);
    if (eff >= 0.75) return bn;
  }
  return 32;
}

}  // namespace gemm
}  // namespace ibm

// Diagnostic: how many clusters of `cluster_size` CTAs of the 256 x 256 bf16 kernel can be resident at once (the answer
// bounds the persistent grid; GPCs whose SM count is not a multiple of the cluster size leave SMs idle).
extern "C" int ibm_debug_gemm_max_clusters(int32_t cluster_size) {
  using namespace ibm::gemm;
  auto kern = gemm_kernel<256, false, false, false, 2, 1, false>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<256, false, 2>::kSmem);
  if (cluster_size > 8) cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(148 / cluster_size * cluster_size);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = Cfg<256, false, 2>::kSmem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster_size;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = -1;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return -1; }
  return n;
}

extern "C" int ibm_gemm_bf16(const void* A, int64_t lda, int32_t a_mn_major, const void* B, int64_t ldb, int32_t b_mn_major,
                             int64_t M, int64_t N, int64_t K, const float* bias, int32_t act, const void* aux, int64_t ldaux,
                             int32_t aux_mode, void* D, int64_t ldd, int32_t out_dtype, int32_t accumulate, int32_t split_k,
                             int32_t taps, float* colsum_out, void* mask, int64_t ldmask, int32_t mask_mode, void* stream) {
  using namespace ibm;
  using namespace ibm::gemm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(A && B && D, "gemm: null operand");
  IBM_CHECK_ARG(M > 0 && N > 0 && K > 0, "gemm: empty problem (M=%lld N=%lld K=%lld)", (long long)M, (long long)N, (long long)K);
  IBM_CHECK_ARG(M < (1ll << 31) && N < (1ll << 31) && K < (1ll << 31), "gemm: dimension too large");
  IBM_CHECK_ARG(lda % 8 == 0 && ldb % 8 == 0 && aligned16(A) && aligned16(B) && aligned16(D),
                "gemm: lda/ldb must be multiples of 8 elements and pointers 16-byte aligned");
  IBM_CHECK_ARG(out_dtype == IBM_BF16 || out_dtype == IBM_F32, "gemm: bad out dtype");
  IBM_CHECK_ARG((out_dtype == IBM_BF16 && ldd % 8 == 0) || (out_dtype == IBM_F32 && ldd % 4 == 0), "gemm: ldd not 16-byte aligned");
  IBM_CHECK_ARG(act >= 0 && act <= IBM_ACT_SILU, "gemm: bad activation %d", act);
  IBM_CHECK_ARG(aux_mode >= 0 && aux_mode <= 2 && (aux_mode == 0 || aux != nullptr), "gemm: bad aux mode");
  IBM_CHECK_ARG(aux_mode == 0 || (ldaux % 8 == 0 && aligned16(aux)), "gemm: aux must be 16-byte aligned with ld %% 8 == 0");
  // the epilogues instantiated for aux: the residual add after none / relu / elu, and every derivative that follows from
  // the activation's output (SiLU's does not)
  IBM_CHECK_ARG(aux_mode != 1 || act == IBM_ACT_NONE || act == IBM_ACT_RELU || act == IBM_ACT_ELU,
                "gemm: aux_mode 1 (residual) supports act none, relu or elu, got %d", act);
  IBM_CHECK_ARG(aux_mode != 2 || act != IBM_ACT_SILU, "gemm: aux_mode 2 needs act' from the activation output: not silu");
  IBM_CHECK_ARG(bias == nullptr || aligned16(bias), "gemm: bias must be 16-byte aligned");
  IBM_CHECK_ARG(!accumulate || (out_dtype == IBM_F32 && act == IBM_ACT_NONE && aux_mode == 0 && bias == nullptr),
                "gemm: accumulate mode needs fp32 output and a plain epilogue");
  IBM_CHECK_ARG(colsum_out == nullptr || (out_dtype == IBM_BF16 && !accumulate), "gemm: colsum_out needs a bf16 output");
  IBM_CHECK_ARG(mask_mode >= 0 && mask_mode <= 2, "gemm: bad mask mode");
  IBM_CHECK_ARG(mask_mode == 0 || (mask != nullptr && out_dtype == IBM_BF16 && !accumulate && aux_mode == 0 && N % 64 == 0 &&
                                   ldmask % 8 == 0 && ldmask * 8 >= N && (reinterpret_cast<uintptr_t>(mask) & 7) == 0),
                "gemm: sign bitmask needs a bf16 output without aux, N %% 64 == 0 and an 8-byte aligned mask with ldmask %% 8 == 0");
  IBM_CHECK_ARG(mask_mode != 2 || act == IBM_ACT_NONE, "gemm: mask_mode 2 gates acc + bias: act must be none");
  if (taps < 1) taps = 1;
  IBM_CHECK_ARG(taps == 1 || (!a_mn_major && K % taps == 0 && (K / taps) % 8 == 0), "gemm: taps needs K-major A and K/taps %% 8 == 0");

  int bn = pick_bn(N);
  if (b_mn_major && bn < 64) bn = 64;     // an MN-major SWIZZLE_128B atom is 64 elements wide
  if (out_dtype == IBM_BF16 && bn < 64) bn = 64;   // bf16 epilogue chunks are 64 columns (one 128-byte staging row)
  const int64_t k_tap = K / taps;
  Args args;
  args.M = M; args.N = N;
  args.kb_per_tap = (int32_t)ceil_div(k_tap, BLOCK_K);
  args.kb_total = args.kb_per_tap * taps;
  // CTA pairs (256-row blocks) whenever there are at least two 128-row blocks and B splits into whole swizzle atoms
  int cg = (ceil_div(M, BLOCK_M) >= 2 && bn >= 128) ? 2 : 1;
  if (forced_cg() == 1) cg = 1;
  args.tiles_m = (int32_t)ceil_div(M, (int64_t)cg * BLOCK_M);
  // two column tiles per work item when the main loop is long enough to pay for the un-overlapped epilogue, the plain
  // (non-aux) epilogue is in use and the tile count is even
  int nt = 1;
  static int64_t min_k = -1;
  if (min_k < 0) {
    const char* e = getenv("IBM_GEMM_NT_MINK");
    min_k = e ? atoll(e) : 1024;
  }
  // (small problems keep single tiles: fewer, fatter work items would leave pairs idle in the last round —
  //  split-K launches are exempt, their split count restores the balance)
  if (cg == 2 && bn == 256 && K >= min_k && ceil_div(N, bn) % 2 == 0 && forced_nt() != 1 &&
      (aux_mode == 0 || (out_dtype == IBM_BF16 && !accumulate)) &&
      (accumulate || (int64_t)args.tiles_m * (ceil_div(N, bn) / 2) >= 2 * (sm_count() / cg)))
    nt = 2;
  args.tiles_n = (int32_t)ceil_div(N, (int64_t)nt * bn);
  const int sms = sm_count();
  int splits = 1;
  if (accumulate) {
    const int64_t tiles = (int64_t)args.tiles_m * args.tiles_n;
    if (split_k > 0) {
      splits = split_k;
    } else {
      // fill whole rounds of the persistent grid: most work per round among 1..4 rounds, fewest splits on a tie
      const int workers = sms / cg;
      double best = 0.0;
      for (int rounds = 1; rounds <= 4; ++rounds) {
        const int sp = (int)((int64_t)rounds * workers / tiles) > 0 ? (int)((int64_t)rounds * workers / tiles) : 1;
        const int64_t wk = tiles * sp;
        const double eff = (double)wk / (double)(ceil_div(wk, workers) * workers);
        if (eff > best + 0.02) { best = eff; splits = sp; }
      }
    }
    int max_splits = args.kb_total / 8 > 0 ? args.kb_total / 8 : 1;
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
  }
  args.kb_per_split = (int32_t)ceil_div(args.kb_total, splits);
  args.splits = (int32_t)ceil_div(args.kb_total, args.kb_per_split);
  args.a_mn = a_mn_major ? 1 : 0;
  args.b_mn = b_mn_major ? 1 : 0;
  args.act = act; args.aux_mode = aux_mode;
  args.bias = bias;
  args.aux = static_cast<const __nv_bfloat16*>(aux);
  args.ldaux = ldaux;
  args.colsum = colsum_out;
  args.mask = static_cast<uint8_t*>(mask);
  args.ldmask = ldmask;
  args.mask_mode = mask_mode;
  args.reverse = 0;
  static int stagger_on = -1;
  if (stagger_on < 0) {
    const char* e = getenv("IBM_GEMM_STAGGER");
    stagger_on = (e && e[0] == '0') ? 0 : 1;
  }
  args.stagger = stagger_on;
  static int fp2_on = -1;
  if (fp2_on < 0) {
    const char* e = getenv("IBM_GEMM_FP2");
    fp2_on = (e && e[0] == '0') ? 0 : 1;
  }
  args.fp2 = fp2_on;
  // L2 prefetch of the aux tiles a main loop ahead of the epilogue: OFF.  Measured on one box (profiles/r02b_gemm_experiments.md):
  // both ways of doing it — 32 TMA prefetch ops per item in the producer, or plain prefetch.global.L2 from the spare warp —
  // cost 4 % on every aux shape (FFN-2 forward 364 -> 378 us, QKV dgrad 284 -> 298); IBM_GEMM_PFAUX=1/2 re-enables them.
  static int pf_aux = -1;
  if (pf_aux < 0) {
    const char* e = getenv("IBM_GEMM_PFAUX");
    pf_aux = (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 0;
  }
  args.pf_aux = pf_aux;
  // With taps the B operand is [N, taps * kb_per_tap * 64] (each tap's K padded to whole k blocks; [taps * kb_per_tap * 64, N]
  // when MN-major).
  const int64_t Kb = taps == 1 ? K : (int64_t)args.kb_total * BLOCK_K;

  CUtensorMap ta, tb, td;
  int rc;
  if (!args.a_mn) rc = make_map(&ta, A, false, k_tap, M + (taps - 1), lda, BLOCK_K, BLOCK_M);
  else rc = make_map(&ta, A, false, M, K, lda, 64, BLOCK_K);
  if (rc) return rc;
  if (!args.b_mn) rc = make_map(&tb, B, false, Kb, N, ldb, BLOCK_K, (uint32_t)(bn / cg));
  else rc = make_map(&tb, B, false, N, Kb, ldb, 64, BLOCK_K);
  if (rc) return rc;
  const bool f32 = out_dtype == IBM_F32;
  rc = make_map(&td, D, f32, N, M, ldd, f32 ? 32 : 64, 32);           // one epilogue warp's 32-row tile
  if (rc) return rc;
  CUtensorMap tx = td;                       // aux tile map (bf16 [M,N], same 64 x 32 box as the bf16 store)
  if (aux_mode != 0 && !f32 && !accumulate) {
    rc = make_map(&tx, aux, false, N, M, ldaux, 64, 32);
    if (rc) return rc;
  }

  const int64_t work = (int64_t)args.tiles_m * args.tiles_n * args.splits;
  const int workers = sms / cg;
  int grid = (int)(work < workers ? work : workers) * cg;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // A-stationary: short K (the row block's A fits eight 16 KB slots), several column tiles to amortise it over, enough
  // row blocks to balance the pairs.  OFF by default: it cuts the L2 -> SM reads of the K = 512 layers by 44 % (ncu, r01c)
  // but measured 4-7 % slower than the plain 256 x 256 tiles (290 vs 272 us QKV, 379 vs 361 us FFN-1; 60 % vs 68 % tensor
  // pipe) — the short main loops are not fabric-bound.  IBM_GEMM_AS=1 enables it for experiments; parity-tested either way.
  static int as_on = -1;
  if (as_on < 0) {
    const char* e = getenv("IBM_GEMM_AS");
    as_on = (e && e[0] == '1') ? 1 : 0;
  }
  const bool use_as = as_on && cg == 2 && bn == 256 && nt == 1 && aux_mode == 0 && !accumulate && taps == 1 && args.kb_total <= kASlots &&
      args.tiles_n >= 2 && args.tiles_m >= 2 * workers;
  // bytes this launch streams: both operands once plus the output (the walk order only matters, and only alternates, for
  // launches that cannot live in L2)
  if (!use_as) args.reverse = next_walk_reverse((M * K + N * K) * 2 + M * N * (f32 ? 4 : 2));
  if (as_on && cg == 2 && bn == 256 && nt == 1 && aux_mode == 0 && !accumulate && taps == 1 && args.kb_total <= kASlots &&
      args.tiles_n >= 2 && args.tiles_m >= 2 * workers) {
    grid = workers * cg;
    if (f32) return launch<256, true, false, false, 2, 1, true>(ta, tb, td, tx, args, grid, s);
    return launch<256, false, false, false, 2, 1, true>(ta, tb, td, tx, args, grid, s);
  }
#define IBM_GEMM_DISPATCH(BNV, CGV)                                                        \
  do {                                                                                     \
    if (accumulate) return launch<BNV, true, true, false, CGV>(ta, tb, td, tx, args, grid, s);   \
    if (f32) return launch<BNV, true, false, false, CGV>(ta, tb, td, tx, args, grid, s);         \
    if (aux_mode != 0) return launch<BNV, false, false, true, CGV>(ta, tb, td, tx, args, grid, s); \
    return launch<BNV, false, false, false, CGV>(ta, tb, td, tx, args, grid, s);                 \
  } while (0)
  if (nt == 2) {
    if (accumulate) return launch<256, true, true, false, 2, 2>(ta, tb, td, tx, args, grid, s);
    if (f32) return launch<256, true, false, false, 2, 2>(ta, tb, td, tx, args, grid, s);
    if (aux_mode != 0) return launch<256, false, false, true, 2, 2>(ta, tb, td, tx, args, grid, s);
    return launch<256, false, false, false, 2, 2>(ta, tb, td, tx, args, grid, s);
  }
  if (cg == 2) {
    if (bn == 256 && !accumulate && !f32 && aux_mode == 0) {      // the hot bf16 shapes: mask mode compiled in
      if (mask_mode == 0) return launch<256, false, false, false, 2, 1, false, 0>(ta, tb, td, tx, args, grid, s);
      if (mask_mode == 1) return launch<256, false, false, false, 2, 1, false, 1>(ta, tb, td, tx, args, grid, s);
      return launch<256, false, false, false, 2, 1, false, 2>(ta, tb, td, tx, args, grid, s);
    }
    if (bn == 256) IBM_GEMM_DISPATCH(256, 2);
    IBM_GEMM_DISPATCH(128, 2);
  }
  switch (bn) {
    case 256: IBM_GEMM_DISPATCH(256, 1);
    case 128: IBM_GEMM_DISPATCH(128, 1);
    case 64: IBM_GEMM_DISPATCH(64, 1);
    default:                          // BN = 32 exists for fp32 outputs only (bf16 chunks are 64 columns wide)
      if (accumulate) return launch<32, true, true, false, 1>(ta, tb, td, tx, args, grid, s);
      return launch<32, true, false, false, 1>(ta, tb, td, tx, args, grid, s);
  }
#undef IBM_GEMM_DISPATCH
}
