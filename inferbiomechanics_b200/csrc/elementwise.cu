// Small HBM-bound helpers around the GEMMs: bias-gradient column sums, dtype casts, standalone
// activation forward/backward, Conv1d weight re-layout.
#include "common.cuh"

namespace ibm {

constexpr int kThreads = 256;

// ---- column sums (bias gradients: torch autograd's sum over rows for nn.Linear bias) -----------
constexpr int kColsumRows = 512;
__global__ void __launch_bounds__(kThreads)
colsum_kernel(const __nv_bfloat16* __restrict__ X, long long ld, long long M, long long N, float* __restrict__ out) {
  __shared__ float sm[8][256 + 8];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long c = (long long)blockIdx.y * 256 + tx * 8;
  const long long r0 = (long long)blockIdx.x * kColsumRows;
  const long long r1 = r0 + kColsumRows < M ? r0 + kColsumRows : M;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (c < N) {
    const bool full = c + 8 <= N;
#pragma unroll 4
    for (long long r = r0 + ty; r < r1; r += 8) {
      if (full) {
        uint4 u = ld_stream16(X + r * ld + c);
        float2 a;
        a = unpack_bf16x2(u.x); acc[0] += a.x; acc[1] += a.y;
        a = unpack_bf16x2(u.y); acc[2] += a.x; acc[3] += a.y;
        a = unpack_bf16x2(u.z); acc[4] += a.x; acc[5] += a.y;
        a = unpack_bf16x2(u.w); acc[6] += a.x; acc[7] += a.y;
      } else {
        for (int j = 0; j < 8 && c + j < N; ++j) acc[j] += __bfloat162float(X[r * ld + c + j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sm[ty][tx * 8 + j] = acc[j];
  __syncthreads();
  const long long col = (long long)blockIdx.y * 256 + threadIdx.x;
  if (col < N) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += sm[w][threadIdx.x];
    atomicAdd(out + col, s);
  }
}

// ---- casts ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
cast_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long n8 = n >> 3;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
    float4 a = ld_stream_f4(src + i * 8), b = ld_stream_f4(src + i * 8 + 4);
    st_stream16(dst + i * 8, make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y), pack_bf16x2(b.z, b.w)));
  }
  for (long long i = (n8 << 3) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = __float2bfloat16_rn(src[i]);
}
__global__ void __launch_bounds__(kThreads)
cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dst[i] = __bfloat162float(src[i]);
}
__global__ void __launch_bounds__(kThreads)
cast_pad_kernel(const float* __restrict__ src, long long ld_src, __nv_bfloat16* __restrict__ dst, long long ld_dst,
                long long rows, long long cols) {
  const long long n = rows * ld_dst;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / ld_dst, c = i - r * ld_dst;
    dst[i] = c < cols ? __float2bfloat16_rn(__ldg(src + r * ld_src + c)) : __float2bfloat16_rn(0.f);
  }
}

// ---- standalone activation (time-embedding MLP's SiLU) ----------------------------------------
__global__ void __launch_bounds__(kThreads)
act_fwd_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n, int act) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = __float2bfloat16_rn(act_apply(__bfloat162float(x[i]), act));
}
__global__ void __launch_bounds__(kThreads)
act_bwd_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ dx,
               long long n, int act) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dx[i] = __float2bfloat16_rn(__bfloat162float(dy[i]) * act_grad_from_input(__bfloat162float(x[i]), act));
}

// ---- Conv1d weight (Cout,Cin,Kt) <-> GEMM layout [Cout, Kt*cin_pad] ((tap, ci) order) -----------
__global__ void __launch_bounds__(kThreads)
conv_w_to_gemm_kernel(const float* __restrict__ w, int cout, int cin, int kt, int cin_pad, __nv_bfloat16* __restrict__ dst) {
  const long long n = (long long)cout * kt * cin_pad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int ci = (int)(i % cin_pad);
    const long long r = i / cin_pad;
    const int j = (int)(r % kt);
    const int co = (int)(r / kt);
    dst[i] = __float2bfloat16_rn(ci < cin ? __ldg(w + ((long long)co * cin + ci) * kt + j) : 0.f);
  }
}
__global__ void __launch_bounds__(kThreads)
conv_wgrad_from_gemm_kernel(const float* __restrict__ g, int cout, int cin, int kt, int cin_pad, float* __restrict__ dw,
                            int accumulate) {
  const long long n = (long long)cout * cin * kt;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % kt);
    const long long r = i / kt;
    const int ci = (int)(r % cin);
    const int co = (int)(r / cin);
    const float v = __ldg(g + ((long long)co * kt + j) * cin_pad + ci);
    dw[i] = accumulate ? dw[i] + v : v;
  }
}

static int ew_grid(long long n_items) {
  long long need = ceil_div(n_items, kThreads);
  long long cap = (long long)sm_count() * 16;
  return (int)(need < 1 ? 1 : (need < cap ? need : cap));
}

}  // namespace ibm

extern "C" int ibm_colsum_bf16(const void* X, int64_t ld, int64_t M, int64_t N, float* out, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(X && out && M > 0 && N > 0 && ld >= N, "colsum: bad argument");
  IBM_CHECK_ARG(ld % 8 == 0 && aligned16(X), "colsum: ld must be a multiple of 8 and X 16-byte aligned");
  dim3 grid((unsigned)ceil_div(M, kColsumRows), (unsigned)ceil_div(N, 256));
  colsum_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(X), ld, M, N, out);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_act_fwd(const void* x, void* y, int64_t n, int32_t act, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x && y && n > 0 && act >= 0 && act <= IBM_ACT_SILU, "act_fwd: bad argument");
  act_fwd_kernel<<<ew_grid(n), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(y), n, act);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_act_bwd(const void* dy, const void* x, void* dx, int64_t n, int32_t act, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(dy && x && dx && n > 0 && act >= 0 && act <= IBM_ACT_SILU, "act_bwd: bad argument");
  act_bwd_kernel<<<ew_grid(n), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(dx), n, act);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(src && dst && n > 0, "cast_f32_bf16: bad argument");
  IBM_CHECK_ARG(aligned16(src) && aligned16(dst), "cast_f32_bf16: pointers must be 16-byte aligned");
  cast_f32_bf16_kernel<<<ew_grid(n / 8 + 1), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      src, static_cast<__nv_bfloat16*>(dst), n);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_cast_bf16_f32(const void* src, float* dst, int64_t n, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(src && dst && n > 0, "cast_bf16_f32: bad argument");
  cast_bf16_f32_kernel<<<ew_grid(n), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(src), dst, n);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_cast_pad_f32_bf16(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int64_t rows,
                                     int64_t cols, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(src && dst && rows > 0 && cols > 0 && ld_src >= cols && ld_dst >= cols, "cast_pad: bad argument");
  cast_pad_kernel<<<ew_grid(rows * ld_dst), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      src, ld_src, static_cast<__nv_bfloat16*>(dst), ld_dst, rows, cols);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_conv_weight_to_gemm(const float* w, int32_t cout, int32_t cin, int32_t kt, int32_t cin_pad,
                                       void* dst_bf16, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(w && dst_bf16 && cout > 0 && cin > 0 && kt > 0 && cin_pad >= cin, "conv_weight_to_gemm: bad argument");
  conv_w_to_gemm_kernel<<<ew_grid((long long)cout * kt * cin_pad), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      w, cout, cin, kt, cin_pad, static_cast<__nv_bfloat16*>(dst_bf16));
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_conv_wgrad_from_gemm(const float* g, int32_t cout, int32_t cin, int32_t kt, int32_t cin_pad, float* dw,
                                        int32_t accumulate, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(g && dw && cout > 0 && cin > 0 && kt > 0 && cin_pad >= cin, "conv_wgrad_from_gemm: bad argument");
  conv_wgrad_from_gemm_kernel<<<ew_grid((long long)cout * cin * kt), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      g, cout, cin, kt, cin_pad, dw, accumulate);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

// ---- temporal replicate padding for the implicit-GEMM convolution (Groundlink.py:41, padding_mode="replicate") ----
// Activations live in a padded row layout: window b owns rows [b*Tp, (b+1)*Tp), Tp = T + 2*pad, frame t at row
// b*Tp + pad + t.  replicate_pad copies the first/last frame rows into the pad rows; fold_pad is its adjoint
// (pad-row gradients are added into the edge frames, then the pad rows are zeroed so they cannot leak into the
// shifted dgrad/wgrad GEMMs).  With T == 1 both edges are the same row, so the side-0 thread folds both sides' pad
// rows into it and the side-1 thread does nothing (two threads storing one row would drop one side's sum).
namespace ibm {
__global__ void __launch_bounds__(kThreads)
replicate_pad_kernel(__nv_bfloat16* __restrict__ X, long long ld, long long n_win, int T, int pad, int cols8) {
  const long long n = n_win * 2 * pad * cols8;
  const int Tp = T + 2 * pad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cols8) * 8;
    const long long r = i / cols8;
    const int k = (int)(r % (2 * pad));
    const long long b = r / (2 * pad);
    const int dst = k < pad ? k : T + k;                       // pad rows 0..pad-1 and T+pad..Tp-1
    const int src = k < pad ? pad : T + pad - 1;
    *reinterpret_cast<uint4*>(X + (b * Tp + dst) * ld + c) = *reinterpret_cast<const uint4*>(X + (b * Tp + src) * ld + c);
  }
}
__global__ void __launch_bounds__(kThreads)
fold_pad_kernel(__nv_bfloat16* __restrict__ G, long long ld, long long n_win, int T, int pad, int cols8) {
  const long long n = n_win * 2 * cols8;
  const int Tp = T + 2 * pad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cols8) * 8;
    const long long r = i / cols8;
    const int side = (int)(r & 1);
    if (side && T == 1) continue;
    const long long b = r >> 1;
    const int edge = side ? T + pad - 1 : pad;
    const int last_side = T == 1 ? 1 : side;
    float acc[8];
    {
      uint4 u = *reinterpret_cast<const uint4*>(G + (b * Tp + edge) * ld + c);
      float2 t;
      t = unpack_bf16x2(u.x); acc[0] = t.x; acc[1] = t.y;
      t = unpack_bf16x2(u.y); acc[2] = t.x; acc[3] = t.y;
      t = unpack_bf16x2(u.z); acc[4] = t.x; acc[5] = t.y;
      t = unpack_bf16x2(u.w); acc[6] = t.x; acc[7] = t.y;
    }
    for (int s = side; s <= last_side; ++s) {
      for (int k = 0; k < pad; ++k) {
        const int prow = s ? T + pad + k : k;
        __nv_bfloat16* pp = G + (b * Tp + prow) * ld + c;
        uint4 u = *reinterpret_cast<const uint4*>(pp);
        float2 t;
        t = unpack_bf16x2(u.x); acc[0] += t.x; acc[1] += t.y;
        t = unpack_bf16x2(u.y); acc[2] += t.x; acc[3] += t.y;
        t = unpack_bf16x2(u.z); acc[4] += t.x; acc[5] += t.y;
        t = unpack_bf16x2(u.w); acc[6] += t.x; acc[7] += t.y;
        *reinterpret_cast<uint4*>(pp) = make_uint4(0, 0, 0, 0);
      }
    }
    *reinterpret_cast<uint4*>(G + (b * Tp + edge) * ld + c) =
        make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]), pack_bf16x2(acc[4], acc[5]), pack_bf16x2(acc[6], acc[7]));
  }
}

// inverted dropout with a counter-based mask: element i is kept iff Philox(seed, offset)[i] >= p; kept values are
// scaled by 1/(1-p).  Forward and backward call the same kernel with the same (seed, offset), so the mask is never stored.
__global__ void __launch_bounds__(kThreads)
dropout_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, long long n, float p, float scale,
               uint64_t seed, uint64_t offset, const long long* __restrict__ step_dev, long long step_mul) {
  // device-resident step counter (CUDA-graph replays cannot change a by-value argument): offset += step_mul * *step_dev
  if (step_dev != nullptr) offset += (uint64_t)(step_mul * __ldg(step_dev));
  const long long n4 = n >> 2;
  const uint32_t thresh = (uint32_t)(p * 4294967296.0);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint2 u = *reinterpret_cast<const uint2*>(x + 4 * i);
    float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
    a.x = r.x >= thresh ? a.x * scale : 0.f;
    a.y = r.y >= thresh ? a.y * scale : 0.f;
    b.x = r.z >= thresh ? b.x * scale : 0.f;
    b.y = r.w >= thresh ? b.y * scale : 0.f;
    *reinterpret_cast<uint2*>(y + 4 * i) = make_uint2(pack_bf16x2(a.x, a.y), pack_bf16x2(b.x, b.y));
  }
}

__global__ void counter_add_kernel(long long* ctr, long long inc) { *ctr += inc; }

// Conv1d weight (Cout,Cin,Kt) fp32 → bf16 dgrad-GEMM layout [Cin, Kt*cout_pad]: B[ci, j'*cout_pad + co] = W[co, ci, Kt-1-j']
__global__ void __launch_bounds__(kThreads)
conv_w_to_dgrad_kernel(const float* __restrict__ w, int cout, int cin, int kt, int cout_pad, __nv_bfloat16* __restrict__ dst) {
  const long long n = (long long)cin * kt * cout_pad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i % cout_pad);
    const long long r = i / cout_pad;
    const int jp = (int)(r % kt);
    const int ci = (int)(r / kt);
    dst[i] = __float2bfloat16_rn(co < cout ? __ldg(w + ((long long)co * cin + ci) * kt + (kt - 1 - jp)) : 0.f);
  }
}
}  // namespace ibm

extern "C" int ibm_replicate_pad_rows(void* X, int64_t ld, int64_t n_win, int32_t T, int32_t pad, int32_t cols, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(X && n_win > 0 && T > 0 && pad >= 0 && cols > 0 && cols % 8 == 0 && ld % 8 == 0 && ld >= cols && aligned16(X),
                "replicate_pad_rows: bad argument (cols and ld must be multiples of 8)");
  if (pad == 0) return IBM_OK;                                  // kernel size 1: no pad rows
  replicate_pad_kernel<<<ew_grid(n_win * 2 * pad * (cols / 8)), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<__nv_bfloat16*>(X), ld, n_win, T, pad, cols / 8);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_fold_pad_rows(void* G, int64_t ld, int64_t n_win, int32_t T, int32_t pad, int32_t cols, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(G && n_win > 0 && T > 0 && pad >= 0 && cols > 0 && cols % 8 == 0 && ld % 8 == 0 && ld >= cols && aligned16(G),
                "fold_pad_rows: bad argument (cols and ld must be multiples of 8)");
  if (pad == 0) return IBM_OK;                                  // kernel size 1: no pad rows
  fold_pad_kernel<<<ew_grid(n_win * 2 * (cols / 8)), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<__nv_bfloat16*>(G), ld, n_win, T, pad, cols / 8);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_dropout_bf16(const void* x, void* y, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x && y && n > 0 && n % 4 == 0 && p >= 0.f && p < 1.f, "dropout: bad argument (n %% 4 == 0, 0 <= p < 1)");
  dropout_kernel<<<ew_grid(n / 4), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(y), n, p, 1.f / (1.f - p), seed, offset, nullptr, 0);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_dropout_bf16_dev(const void* x, void* y, int64_t n, float p, uint64_t seed, uint64_t offset, const int64_t* step_dev,
                                    int64_t step_mul, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(x && y && step_dev && n > 0 && n % 4 == 0 && p >= 0.f && p < 1.f, "dropout_dev: bad argument (n %% 4 == 0, 0 <= p < 1)");
  dropout_kernel<<<ew_grid(n / 4), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), static_cast<__nv_bfloat16*>(y), n, p, 1.f / (1.f - p), seed, offset,
      reinterpret_cast<const long long*>(step_dev), (long long)step_mul);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_counter_add(int64_t* counter_dev, int64_t inc, void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(counter_dev != nullptr, "counter_add: null counter");
  counter_add_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<long long*>(counter_dev), (long long)inc);
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}

extern "C" int ibm_conv_weight_to_dgrad(const float* w, int32_t cout, int32_t cin, int32_t kt, int32_t cout_pad, void* dst_bf16,
                                        void* stream) {
  using namespace ibm;
  IBM_CHECK_ARCH();
  IBM_CHECK_ARG(w && dst_bf16 && cout > 0 && cin > 0 && kt > 0 && cout_pad >= cout, "conv_weight_to_dgrad: bad argument");
  conv_w_to_dgrad_kernel<<<ew_grid((long long)cin * kt * cout_pad), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      w, cout, cin, kt, cout_pad, static_cast<__nv_bfloat16*>(dst_bf16));
  IBM_LAUNCH_CHECK();
  return IBM_OK;
}
