// Ensemble scoring of K sampled trajectories per window (ibm_ensemble_score, DESIGN.md §3): the ensemble mean, and per channel
// the fair CRPS, the spread, the squared error of the mean and the mean pairwise distance, summed into a caller-owned fp64
// accumulator.  One read of the K draws, HBM/L2-streaming: each thread owns one output channel of one row at a time and holds
// its K values in registers (KMAX of them, a compile-time power of two >= K), so the mean, the two-pass variance, the label
// distances and the sorted-form pair sum are arithmetic on values already on chip.  Per-thread fp64 sums -> per-block
// partials -> the last-arriving block reduces them in a fixed order (deterministic, no float atomics) and adds the batch's
// totals into the accumulator.
#include "common.cuh"

namespace ibm {

constexpr int kEnsChannels = 30;
constexpr int kEnsRows = 8;                       // rows per block and trip: 8 x 30 = 240 active threads of 256
constexpr int kEnsThreads = 256;
constexpr int kEnsQ = 5;                          // accumulator rows: crps, s2, sqerr, pair, count
constexpr int kEnsVals = kEnsQ * kEnsChannels;
constexpr int kEnsMaxBlocks = 1024;               // size of the caller's partials buffer (ibm_b200.h)
constexpr int kEnsSlices = 8;                     // last block: each value summed in 8 interleaved slices, then in order

// Bitonic sorting network on N registers, ascending; every index is a compile-time constant after unrolling, so v stays in
// registers.  fminf / fmaxf are exact.
template <int N>
__device__ __forceinline__ void sort_network(float (&v)[N]) {
#pragma unroll
  for (int size = 2; size <= N; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const int j = i ^ stride;
        if (j > i) {
          const float lo = fminf(v[i], v[j]), hi = fmaxf(v[i], v[j]);
          const bool up = (i & size) == 0;
          v[i] = up ? lo : hi;
          v[j] = up ? hi : lo;
        }
      }
    }
  }
}

// Two blocks per SM up to KMAX = 32 (<= 128 registers); KMAX = 64 needs ~250 registers for its 64 values and runs one block
// per SM, which still keeps 64 loads per thread in flight.  No instantiation spills (-Xptxas -v).
template <int KMAX>
__global__ void __launch_bounds__(kEnsThreads, KMAX > 32 ? 1 : 2)
ensemble_score_kernel(const float* __restrict__ draws, int K, long long rows, int F, int Fo, const float* __restrict__ labels,
                      float thr2, float* __restrict__ mean_out, double* __restrict__ acc, double* __restrict__ partials,
                      unsigned int* __restrict__ counter) {
  __shared__ double red[kEnsQ][kEnsRows][kEnsChannels];
  __shared__ double slice[kEnsVals][kEnsSlices];
  __shared__ bool is_last;
  const int t = threadIdx.x;
  const bool active = t < kEnsRows * kEnsChannels;
  const int c = active ? t % kEnsChannels : 0, rs = active ? t / kEnsChannels : 0;
  // CoP channels 0-2 (3-5) are scored on the rows where the label force of the same foot, channels 6-8 (9-11), is a contact
  const int fc = c < 3 ? 6 : 9;
  const long long draw_stride = rows * (Fo == 1 ? (long long)F : 1ll) * kEnsChannels;    // floats per draw (B * F * 30)
  const double invK = 1.0 / (double)K, invKK1 = 1.0 / ((double)K * (double)(K - 1));
  double s_crps = 0.0, s_var = 0.0, s_se = 0.0, s_pair = 0.0, s_n = 0.0;
  if (active) {
    for (long long r = (long long)blockIdx.x * kEnsRows + rs; r < rows; r += (long long)gridDim.x * kEnsRows) {
      // scored row r = (b, fo); its draws sit at row b*F + f of each draw, f = fo (Fo == F) or F - 1 (Fo == 1)
      const long long dr = Fo == 1 ? r * F + (F - 1) : r;
      const float* xp = draws + dr * kEnsChannels + c;
      float v[KMAX];
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        v[k] = k < K ? __ldcs(xp) : INFINITY;
        xp += draw_stride;
      }
      const float* __restrict__ lrow = labels + r * kEnsChannels;
      const float y = __ldg(lrow + c);
      double sx = 0.0;
#pragma unroll
      for (int k = 0; k < KMAX; ++k)
        if (k < K) sx += (double)v[k];
      const double m = sx * invK;
      const float mf = (float)m;
      mean_out[r * kEnsChannels + c] = mf;
      if (c < 6 && !norm3_gt2(__ldg(lrow + fc), __ldg(lrow + fc + 1), __ldg(lrow + fc + 2), thr2)) continue;
      // deviations and distances are single fp32 subtractions (one rounding each, relative to their own size), summed in
      // fp64; the K values stay fp32 so that only K registers are live per element
      double sd = 0.0, ss = 0.0, sa = 0.0;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) {
        if (k < K) {
          const double d = (double)(v[k] - mf);
          sd += d;
          ss = fma(d, d, ss);
          sa += (double)fabsf(v[k] - y);
        }
      }
      // sum_{i<j} |x_i - x_j| = sum_k (2k - K - 1) x_(k), k 1-based over the ascending order, evaluated on the deviations d
      // (the weights sum to 0) as sum_k (2k - 1) d_(k) - K sum_k d_k: compile-time weights, and the large weights multiply
      // deviations, not the values.  The +inf padding sorts behind the K draws.
      sort_network<KMAX>(v);
      double sp = 0.0;
#pragma unroll
      for (int k = 0; k < KMAX; ++k)
        if (k < K) sp = fma((double)(2 * k + 1), (double)(v[k] - mf), sp);
      sp -= (double)K * sd;
      const double e = m - (double)y;
      s_crps += sa * invK - sp * invKK1;
      s_var += ss / (double)(K - 1);
      s_se = fma(e, e, s_se);
      s_pair += 2.0 * sp * invKK1;
      s_n += 1.0;
    }
  }
  if (active) {
    red[0][rs][c] = s_crps;
    red[1][rs][c] = s_var;
    red[2][rs][c] = s_se;
    red[3][rs][c] = s_pair;
    red[4][rs][c] = s_n;
  }
  __syncthreads();
  if (t < kEnsVals) {
    const int q = t / kEnsChannels, ch = t % kEnsChannels;
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < kEnsRows; ++i) s += red[q][i][ch];
    partials[(size_t)blockIdx.x * kEnsVals + t] = s;
  }
  __threadfence();
  __syncthreads();
  if (t == 0) is_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int i = t; i < kEnsVals * kEnsSlices; i += kEnsThreads) {
    const int k = i / kEnsSlices, sl = i % kEnsSlices;
    double s = 0.0;
    for (unsigned int j = sl; j < gridDim.x; j += kEnsSlices) s += __ldcg(partials + (size_t)j * kEnsVals + k);
    slice[k][sl] = s;
  }
  __syncthreads();
  if (t == 0) {
    // one thread adds the batch's totals, in a fixed order, into the accumulator successive batches share
    for (int k = 0; k < kEnsVals; ++k) {
      double s = 0.0;
#pragma unroll
      for (int sl = 0; sl < kEnsSlices; ++sl) s += slice[k][sl];
      acc[k] += s;
    }
    *counter = 0u;
  }
}

template <int KMAX>
static int launch_ensemble(const float* draws, int K, long long rows, int F, int Fo, const float* labels, float thr2,
                           float* mean_out, double* acc, double* partials, unsigned int* counter, cudaStream_t s) {
  static int per_sm = 0;
  if (per_sm == 0) {
    IBM_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ensemble_score_kernel<KMAX>, kEnsThreads, 0));
    if (per_sm < 1) per_sm = 1;
  }
  long long need = ceil_div(rows, kEnsRows);
  long long cap = (long long)sm_count() * per_sm;
  if (cap > kEnsMaxBlocks) cap = kEnsMaxBlocks;
  const int grid = (int)(need < cap ? need : cap);
  ensemble_score_kernel<KMAX><<<grid, kEnsThreads, 0, s>>>(draws, K, rows, F, Fo, labels, thr2, mean_out, acc, partials, counter);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

}  // namespace ibm

extern "C" int ibm_ensemble_score(const float* draws, int32_t K, int64_t B, int32_t F, const float* labels, int32_t Fo,
                                  float threshold, float* mean_out, double* acc, double* partials, uint32_t* counter,
                                  void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(draws && labels && mean_out && acc && partials && counter, "ensemble_score: null pointer");
  IBM_CHECK_ARG(K >= 2 && K <= 64, "ensemble_score: K must lie in [2, 64] (the kernel holds the K draws of an element in "
                "registers), got %d", (int)K);
  IBM_CHECK_ARG(B > 0 && F > 0, "ensemble_score: empty batch (B=%lld F=%d)", (long long)B, (int)F);
  IBM_CHECK_ARG(Fo == 1 || Fo == F, "ensemble_score: Fo must be 1 (last frame) or F=%d, got %d", (int)F, (int)Fo);
  IBM_CHECK_ARG((reinterpret_cast<uintptr_t>(draws) | reinterpret_cast<uintptr_t>(labels) | reinterpret_cast<uintptr_t>(mean_out)) % 4 == 0 &&
                (reinterpret_cast<uintptr_t>(acc) | reinterpret_cast<uintptr_t>(partials)) % 8 == 0 &&
                reinterpret_cast<uintptr_t>(counter) % 4 == 0,
                "ensemble_score: misaligned buffer");
  const long long rows = B * (long long)Fo;
  const float thr2 = norm3_threshold_sq(threshold);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  unsigned int* ctr = reinterpret_cast<unsigned int*>(counter);
  if (K <= 4) return launch_ensemble<4>(draws, K, rows, F, Fo, labels, thr2, mean_out, acc, partials, ctr, s);
  if (K <= 8) return launch_ensemble<8>(draws, K, rows, F, Fo, labels, thr2, mean_out, acc, partials, ctr, s);
  if (K <= 16) return launch_ensemble<16>(draws, K, rows, F, Fo, labels, thr2, mean_out, acc, partials, ctr, s);
  if (K <= 32) return launch_ensemble<32>(draws, K, rows, F, Fo, labels, thr2, mean_out, acc, partials, ctr, s);
  return launch_ensemble<64>(draws, K, rows, F, Fo, labels, thr2, mean_out, acc, partials, ctr, s);
}
