// Per-column min / max of a row-major n x c float32 or float64 table in one streaming pass.
//
// Replaces data_processing.find_minmax (reference baler/modules/data_processing.py:113-130), which
// walks the table column by column in Python.  HBM-bound: 4*c bytes read per row, nothing written.
//
// Every thread reads 128-bit vectors (VEC = 4 floats or 2 doubles) at a grid stride G chosen so that VEC*G is a
// multiple of c: a thread then always sees the same VEC columns and keeps their running min/max in registers.
// Block results are merged with shared-memory atomics on an order-preserving integer encoding of
// the floats, blocks are merged with global atomics on the same encoding, and the last block to
// finish decodes the result.  NaNs propagate (numpy's min/max semantics): a per-column flag.
#include "bb_common.cuh"

namespace {

// Order-preserving unsigned keys (-0 < +0), 128-bit streaming loads and the quiet NaN of each element type.
template <typename T> struct MM;
template <> struct MM<float> {
  using K = unsigned;
  static constexpr int VEC = 4;  // elements per 16-byte load
  static __device__ __forceinline__ K enc(float f) {
    const unsigned b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  }
  static __device__ __forceinline__ float dec(K u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }
  static __device__ __forceinline__ float qnan() { return __int_as_float(0x7fc00000); }
  static __device__ __forceinline__ float lo(float a, float b) { return fminf(a, b); }
  static __device__ __forceinline__ float hi(float a, float b) { return fmaxf(a, b); }
  static __device__ __forceinline__ void ld_stream(const float* p, float (&e)[4]) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(e[0]), "=f"(e[1]), "=f"(e[2]), "=f"(e[3]) : "l"(p));
  }
};
template <> struct MM<double> {
  using K = unsigned long long;
  static constexpr int VEC = 2;
  static __device__ __forceinline__ K enc(double f) {
    const K b = (K)__double_as_longlong(f);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
  }
  static __device__ __forceinline__ double dec(K u) {
    return __longlong_as_double((long long)((u & 0x8000000000000000ull) ? (u & 0x7fffffffffffffffull) : ~u));
  }
  static __device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000ll); }
  static __device__ __forceinline__ double lo(double a, double b) { return fmin(a, b); }
  static __device__ __forceinline__ double hi(double a, double b) { return fmax(a, b); }
  static __device__ __forceinline__ void ld_stream(const double* p, double (&e)[2]) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(e[0]), "=d"(e[1]) : "l"(p));
  }
};

// acc layout (keys, global): [min c][max c][nan c][counter]
template <typename T, bool VECTOR>
__global__ void __launch_bounds__(1024)
colminmax_kernel(const T* __restrict__ x, const int64_t n_elems, const int c,
                 typename MM<T>::K* __restrict__ acc, T* __restrict__ min_out, T* __restrict__ max_out) {
  using K = typename MM<T>::K;
  constexpr int VEC = VECTOR ? MM<T>::VEC : 1;
  extern __shared__ __align__(8) unsigned char sm_raw[];
  K* sm = reinterpret_cast<K*>(sm_raw);  // [min c][max c][nan c]
  for (int i = threadIdx.x; i < 3 * c; i += blockDim.x) sm[i] = (i < c) ? ~(K)0 : (K)0;
  __syncthreads();

  const int64_t G = (int64_t)gridDim.x * blockDim.x;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  T mn[VEC], mx[VEC];
  bool nan[VEC];  // per lane: a NaN makes its own column's min / max NaN, and only that column's
#pragma unroll
  for (int q = 0; q < VEC; ++q) { mn[q] = (T)INFINITY; mx[q] = -(T)INFINITY; nan[q] = false; }
  const int64_t n_vec = n_elems / VEC;
  if constexpr (VECTOR) {
    int64_t v = g;
    for (; v + 3 * G < n_vec; v += 4 * G) {  // 4 independent 16-byte loads in flight per thread
      T e[4][VEC];
#pragma unroll
      for (int u = 0; u < 4; ++u) MM<T>::ld_stream(x + (v + u * G) * VEC, e[u]);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int q = 0; q < VEC; ++q) {
          mn[q] = MM<T>::lo(mn[q], e[u][q]); mx[q] = MM<T>::hi(mx[q], e[u][q]); nan[q] |= (e[u][q] != e[u][q]);
        }
    }
    for (; v < n_vec; v += G) {
      T e[VEC];
      MM<T>::ld_stream(x + v * VEC, e);
#pragma unroll
      for (int q = 0; q < VEC; ++q) { mn[q] = MM<T>::lo(mn[q], e[q]); mx[q] = MM<T>::hi(mx[q], e[q]); nan[q] |= (e[q] != e[q]); }
    }
  } else {
    for (int64_t v = g; v < n_vec; v += G) {
      const T e = __ldg(x + v);
      mn[0] = MM<T>::lo(mn[0], e); mx[0] = MM<T>::hi(mx[0], e); nan[0] |= (e != e);
    }
  }
  const int col0 = (int)((g * VEC) % c);
#pragma unroll
  for (int q = 0; q < VEC; ++q) {
    const int col = (col0 + q) % c;
    if (mn[q] <= mx[q]) { atomicMin(&sm[col], MM<T>::enc(mn[q])); atomicMax(&sm[c + col], MM<T>::enc(mx[q])); }
    if (nan[q]) sm[2 * c + col] = 1u;
  }
  if (VECTOR && g == 0) {  // scalar tail (n_elems % VEC elements)
    for (int64_t e = n_vec * VEC; e < n_elems; ++e) {
      const T f = x[e];
      const int col = (int)(e % c);
      if (f != f) sm[2 * c + col] = 1u;
      else { atomicMin(&sm[col], MM<T>::enc(f)); atomicMax(&sm[c + col], MM<T>::enc(f)); }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < c; i += blockDim.x) {
    atomicMin(&acc[i], sm[i]);
    atomicMax(&acc[c + i], sm[c + i]);
    if (sm[2 * c + i]) atomicOr(&acc[2 * c + i], (K)1);
  }
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(&acc[3 * c], (K)1) == (K)(gridDim.x - 1));
  __syncthreads();
  if (last) {
    __threadfence();
    for (int i = threadIdx.x; i < c; i += blockDim.x) {
      const bool isnan = __ldcg(&acc[2 * c + i]) != (K)0;
      min_out[i] = isnan ? MM<T>::qnan() : MM<T>::dec(__ldcg(&acc[i]));
      max_out[i] = isnan ? MM<T>::qnan() : MM<T>::dec(__ldcg(&acc[c + i]));
    }
    if (threadIdx.x == 0) acc[3 * c] = (K)0;  // ready for an accumulating follow-up call
  }
}

// Wide tables (c > 1024: flattened 2-D snapshots, e.g. 50 x 50 = 2500 per-pixel columns of CFD_dense_AE): one thread per
// column, blockIdx.y strides over rows; consecutive threads read consecutive columns (coalesced), same accumulator layout.
template <typename T>
__global__ void __launch_bounds__(256)
colminmax_wide_kernel(const T* __restrict__ x, const int64_t n_rows, const int c, typename MM<T>::K* __restrict__ acc,
                      T* __restrict__ min_out, T* __restrict__ max_out) {
  using K = typename MM<T>::K;
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col < c) {
    T mn = (T)INFINITY, mx = -(T)INFINITY;
    bool nan = false;
    for (int64_t r = blockIdx.y; r < n_rows; r += gridDim.y) {
      const T e = __ldg(x + r * c + col);
      mn = MM<T>::lo(mn, e); mx = MM<T>::hi(mx, e); nan |= (e != e);
    }
    if (mn <= mx) { atomicMin(&acc[col], MM<T>::enc(mn)); atomicMax(&acc[c + col], MM<T>::enc(mx)); }
    if (nan) atomicOr(&acc[2 * c + col], (K)1);
  }
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(&acc[3 * c], (K)1) == (K)(gridDim.x * gridDim.y - 1));
  __syncthreads();
  if (last) {
    __threadfence();
    for (int i = threadIdx.x; i < c; i += blockDim.x) {
      const bool isnan = __ldcg(&acc[2 * c + i]) != (K)0;
      min_out[i] = isnan ? MM<T>::qnan() : MM<T>::dec(__ldcg(&acc[i]));
      max_out[i] = isnan ? MM<T>::qnan() : MM<T>::dec(__ldcg(&acc[c + i]));
    }
    if (threadIdx.x == 0) acc[3 * c] = (K)0;
  }
}

int gcd(int a, int b) { return b ? gcd(b, a % b) : a; }

template <typename T>
int colminmax_launch(bb_ctx* ctx, const T* x, int64_t n_rows, int n_cols, T* min_dev, T* max_dev, int reset,
                     cudaStream_t stream) {
  using K = typename MM<T>::K;
  const size_t need = (size_t)(3 * n_cols + 1) * sizeof(K);
  if (ctx->minmax_scratch_bytes < need) {
    if (ctx->minmax_scratch) cudaFree(ctx->minmax_scratch);
    ctx->minmax_scratch = nullptr;
    ctx->minmax_scratch_bytes = 0;
    BB_CUDA(cudaMalloc(&ctx->minmax_scratch, need));
    ctx->minmax_scratch_bytes = need;
    reset = 1;
  }
  K* acc = reinterpret_cast<K*>(ctx->minmax_scratch);
  if (reset) {
    BB_CUDA(cudaMemsetAsync(acc, 0xff, (size_t)n_cols * sizeof(K), stream));
    BB_CUDA(cudaMemsetAsync(acc + n_cols, 0, (size_t)(2 * n_cols + 1) * sizeof(K), stream));
  }
  if (n_rows == 0) return BB_OK;
  if (n_cols > 1024) {
    const int gx = (n_cols + 255) / 256;
    int64_t gy = (int64_t)ctx->sm_count * 8 / gx;
    gy = gy < 1 ? 1 : (gy > n_rows ? n_rows : gy);
    colminmax_wide_kernel<T><<<dim3(gx, (unsigned)gy), 256, 0, stream>>>(x, n_rows, n_cols, acc, min_dev, max_dev);
    return (int)cudaGetLastError();
  }
  constexpr int VEC = MM<T>::VEC;
  const int64_t n_elems = n_rows * n_cols;
  const bool vec = (reinterpret_cast<uintptr_t>(x) & 15u) == 0;
  const int lanes = vec ? n_cols / gcd(n_cols, VEC) : n_cols;  // thread period that keeps columns fixed
  int threads = lanes * (384 / lanes > 0 ? 384 / lanes : 1);
  if (threads > 1024) return BB_ERR_UNSUPPORTED;
  int64_t want = (n_elems / (vec ? VEC : 1) + threads - 1) / threads;
  int grid = (int)(want < (int64_t)ctx->sm_count * 4 ? (want > 0 ? want : 1) : ctx->sm_count * 4);
  const size_t smem = (size_t)3 * n_cols * sizeof(K);
  if (vec) colminmax_kernel<T, true><<<grid, threads, smem, stream>>>(x, n_elems, n_cols, acc, min_dev, max_dev);
  else colminmax_kernel<T, false><<<grid, threads, smem, stream>>>(x, n_elems, n_cols, acc, min_dev, max_dev);
  return (int)cudaGetLastError();
}

}  // namespace

// reset != 0: start a new reduction; reset == 0: fold this table into the running min/max (chunked input)
int bb_colminmax_launch(bb_ctx* ctx, const void* x, int dtype, int64_t n_rows, int n_cols, void* min_dev,
                        void* max_dev, int reset, cudaStream_t stream) {
  if (n_cols <= 0 || n_rows < 0) return BB_ERR_INVALID;
  if (dtype == BB_F32)
    return colminmax_launch(ctx, (const float*)x, n_rows, n_cols, (float*)min_dev, (float*)max_dev, reset, stream);
  if (dtype == BB_F64)
    return colminmax_launch(ctx, (const double*)x, n_rows, n_cols, (double*)min_dev, (double*)max_dev, reset, stream);
  return BB_ERR_INVALID;
}

namespace {
// elementwise (x - min) / range or y * range + min; 8 bytes of HBM traffic per element
template <bool INVERSE>
__global__ void __launch_bounds__(256) colscale_kernel(const float* __restrict__ x, const int64_t n_elems, const int c,
                                                       const float* __restrict__ mn, const float* __restrict__ rg,
                                                       float* __restrict__ out) {
  const int64_t G = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_elems; e += G) {
    const int col = (int)(e % c);
    const float v = x[e];
    out[e] = INVERSE ? fmaf(v, __ldg(rg + col), __ldg(mn + col)) : __fdiv_rn(__fsub_rn(v, __ldg(mn + col)), __ldg(rg + col));
  }
}

// (x - min) / range in float64, one rounding per operation like numpy
__global__ void __launch_bounds__(256) normalize_f64_kernel(const double* __restrict__ x, const int64_t n_elems, const int c,
                                                            const double* __restrict__ mn, const double* __restrict__ rg,
                                                            double* __restrict__ out) {
  const int64_t G = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_elems; e += G) {
    const int col = (int)(e % c);
    out[e] = __ddiv_rn(__dsub_rn(x[e], __ldg(mn + col)), __ldg(rg + col));
  }
}
}  // namespace

extern "C" {
int bb_normalize_f64(bb_ctx* ctx, const double* x_dev, int64_t n_rows, int n_cols, const double* min_dev,
                     const double* range_dev, double* out_dev, bb_stream_t stream) {
  if (!ctx || n_cols <= 0 || n_rows < 0 || !min_dev || !range_dev || ((!x_dev || !out_dev) && n_rows)) return BB_ERR_INVALID;
  if (n_rows == 0) return BB_OK;
  const int64_t n = n_rows * n_cols;
  const int grid = (int)((n + 255) / 256 < (int64_t)ctx->sm_count * 8 ? (n + 255) / 256 : ctx->sm_count * 8);
  normalize_f64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, n, n_cols, min_dev, range_dev, out_dev);
  return (int)cudaGetLastError();
}
int bb_normalize_f32(bb_ctx* ctx, const float* x_dev, int64_t n_rows, int n_cols, const float* min_dev,
                     const float* range_dev, float* out_dev, bb_stream_t stream) {
  if (!ctx || n_cols <= 0 || n_rows < 0 || !min_dev || !range_dev || ((!x_dev || !out_dev) && n_rows)) return BB_ERR_INVALID;
  if (n_rows == 0) return BB_OK;
  const int64_t n = n_rows * n_cols;
  const int grid = (int)((n + 255) / 256 < (int64_t)ctx->sm_count * 8 ? (n + 255) / 256 : ctx->sm_count * 8);
  colscale_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, n, n_cols, min_dev, range_dev, out_dev);
  return (int)cudaGetLastError();
}
int bb_renormalize_f32(bb_ctx* ctx, const float* y_dev, int64_t n_rows, int n_cols, const float* min_dev,
                       const float* range_dev, float* out_dev, bb_stream_t stream) {
  if (!ctx || n_cols <= 0 || n_rows < 0 || !min_dev || !range_dev || ((!y_dev || !out_dev) && n_rows)) return BB_ERR_INVALID;
  if (n_rows == 0) return BB_OK;
  const int64_t n = n_rows * n_cols;
  const int grid = (int)((n + 255) / 256 < (int64_t)ctx->sm_count * 8 ? (n + 255) / 256 : ctx->sm_count * 8);
  colscale_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(y_dev, n, n_cols, min_dev, range_dev, out_dev);
  return (int)cudaGetLastError();
}
}
