// Per-column reconstruction error of a chunk of rows (error_report = True): one streaming pass over the raw rows x and
// what decompress writes for them, y.  baler_b200/error_report.py is the one definition of the record; tests/error_report_ref.py
// its numpy mirror.  For each column j, over the rows where x and y are both finite, e = y - x in float64:
//   count, nonfinite_x, nonfinite_y, x_min / x_max (over finite x), sum e, sum e^2, max |e| with the smallest global row
//   attaining it, Baler's response r = 100 e / x over x != 0 (count, sum r, sum r^2), the histogram of |e| against
//   edge_k * range_j (edges 1e-9 ... 1e-1, 1), and for integer columns the count of trunc(y) != x.
// y is first un-normalised when post_min / post_range are given (y * range + min, two IEEE float64 operations: the host
// arithmetic of helper.decompress for tables beyond F32_OFFSET_LIMIT), then truncated toward zero in integer columns.
//
// Access pattern (colminmax_kernel's): a CTA covers a tile of TC = min(C, 256) columns and RL = 256 / TC row lanes; thread t
// owns column c0 + t % TC for the whole pass and walks rows rl, rl + S, rl + 2 S, ... with S = gridDim.y * RL, so a warp reads
// consecutive elements.  Every accumulator lives in registers (the histogram as 10 cumulative integer counters).
// Determinism: no floating-point atomics.  The RL lanes of a column meet in shared memory in a fixed pairwise tree; each CTA
// writes its partial record; a second kernel folds the gridDim.y partials of a column with one warp in a fixed order (lane l
// takes partials l, l + 32, ... in order, then a fixed xor-butterfly).  A re-run on the same device gives the same bits.
#include "bb_common.cuh"

namespace {

constexpr int ES_THREADS = 256;
constexpr int ES_FIELDS = BB_ERROR_STATS_FIELDS;  // 24 words of 8 bytes per column
constexpr int ES_EDGES = 10;                      // histogram edges; 11 bins
constexpr int ES_UNROLL = 4;                      // rows in flight per thread

// record field indices (error_report.FIELDS); hist bins are fields F_HIST .. F_HIST + 10.  In the partials the same slots hold
// the cumulative counts #(|e| > edge_k * range), k = 0..9, converted to bins by the fold kernel.
enum {
  F_COUNT = 0, F_NFX = 1, F_NFY = 2, F_RCOUNT = 3, F_INTMM = 4, F_MAXROW = 5, F_HIST = 6,
  F_XMIN = 17, F_XMAX = 18, F_SE = 19, F_SE2 = 20, F_MAXABS = 21, F_SR = 22, F_SR2 = 23,
};

__device__ __constant__ double kEdges[ES_EDGES] = {1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1, 1.0};

struct Acc {
  unsigned long long cnt, nfx, nfy, rc, imm;
  long long mrow;
  unsigned long long cum[ES_EDGES];
  double xmin, xmax, se, se2, mabs, sr, sr2;

  __device__ void init() {
    cnt = nfx = nfy = rc = imm = 0ull;
#pragma unroll
    for (int k = 0; k < ES_EDGES; ++k) cum[k] = 0ull;
    mrow = -1;
    xmin = INFINITY; xmax = -INFINITY;
    se = se2 = sr = sr2 = 0.0;
    mabs = -1.0;  // below every |e|: "no row yet"
  }
  // fold b into this (this = the earlier part in the fixed order)
  __device__ void fold(const Acc& b) {
    cnt += b.cnt; nfx += b.nfx; nfy += b.nfy; rc += b.rc; imm += b.imm;
#pragma unroll
    for (int k = 0; k < ES_EDGES; ++k) cum[k] += b.cum[k];
    if (b.xmin < xmin) xmin = b.xmin;
    if (b.xmax > xmax) xmax = b.xmax;
    se = __dadd_rn(se, b.se); se2 = __dadd_rn(se2, b.se2);
    sr = __dadd_rn(sr, b.sr); sr2 = __dadd_rn(sr2, b.sr2);
    if (b.mabs > mabs || (b.mabs == mabs && b.mrow >= 0 && (mrow < 0 || b.mrow < mrow))) { mabs = b.mabs; mrow = b.mrow; }
  }
  // words: field f of this column at w[f * stride]
  __device__ void store(unsigned long long* w, int64_t stride) const {
    w[F_COUNT * stride] = cnt; w[F_NFX * stride] = nfx; w[F_NFY * stride] = nfy; w[F_RCOUNT * stride] = rc;
    w[F_INTMM * stride] = imm; w[F_MAXROW * stride] = (unsigned long long)mrow;
#pragma unroll
    for (int k = 0; k < ES_EDGES; ++k) w[(F_HIST + k) * stride] = cum[k];
    w[(F_HIST + ES_EDGES) * stride] = 0ull;
    w[F_XMIN * stride] = (unsigned long long)__double_as_longlong(xmin);
    w[F_XMAX * stride] = (unsigned long long)__double_as_longlong(xmax);
    w[F_SE * stride] = (unsigned long long)__double_as_longlong(se);
    w[F_SE2 * stride] = (unsigned long long)__double_as_longlong(se2);
    w[F_MAXABS * stride] = (unsigned long long)__double_as_longlong(mabs);
    w[F_SR * stride] = (unsigned long long)__double_as_longlong(sr);
    w[F_SR2 * stride] = (unsigned long long)__double_as_longlong(sr2);
  }
  __device__ void load(const unsigned long long* w, int64_t stride) {
    cnt = w[F_COUNT * stride]; nfx = w[F_NFX * stride]; nfy = w[F_NFY * stride]; rc = w[F_RCOUNT * stride];
    imm = w[F_INTMM * stride]; mrow = (long long)w[F_MAXROW * stride];
#pragma unroll
    for (int k = 0; k < ES_EDGES; ++k) cum[k] = w[(F_HIST + k) * stride];
    xmin = __longlong_as_double((long long)w[F_XMIN * stride]);
    xmax = __longlong_as_double((long long)w[F_XMAX * stride]);
    se = __longlong_as_double((long long)w[F_SE * stride]);
    se2 = __longlong_as_double((long long)w[F_SE2 * stride]);
    mabs = __longlong_as_double((long long)w[F_MAXABS * stride]);
    sr = __longlong_as_double((long long)w[F_SR * stride]);
    sr2 = __longlong_as_double((long long)w[F_SR2 * stride]);
  }
};

__device__ __forceinline__ bool finite64(double v) { return fabs(v) <= 1.7976931348623157e308; }

// grid (tiles, gy); block ES_THREADS; dynamic shared memory ES_FIELDS * ES_THREADS words.  partial: [gy][ES_FIELDS][C] words.
template <typename TX, typename TY>
__global__ void __launch_bounds__(ES_THREADS)
error_stats_kernel(const TX* __restrict__ x, const TY* __restrict__ y, const int64_t n_rows, const int C, const int TC,
                   const int RL, const int64_t row0, const double* __restrict__ post_min, const double* __restrict__ post_range,
                   const double* __restrict__ scale_range, const uint8_t* __restrict__ int_mask,
                   unsigned long long* __restrict__ partial) {
  extern __shared__ __align__(16) unsigned long long s_w[];  // [ES_FIELDS][ES_THREADS]
  const int t = threadIdx.x;
  const int rl = t / TC, cl = t - rl * TC;
  const int col = blockIdx.x * TC + cl;
  const bool active = rl < RL && col < C;
  Acc a;
  a.init();
  if (active) {
    const bool post = post_min != nullptr;
    const double pmn = post ? __ldg(post_min + col) : 0.0, prg = post ? __ldg(post_range + col) : 1.0;
    double rng = scale_range != nullptr ? __ldg(scale_range + col) : 1.0;
    if (!(rng > 0.0 && finite64(rng))) rng = 1.0;
    double thr[ES_EDGES];
#pragma unroll
    for (int k = 0; k < ES_EDGES; ++k) thr[k] = __dmul_rn(kEdges[k], rng);
    const bool is_int = int_mask != nullptr && int_mask[col] != 0;
    const int64_t S = (int64_t)gridDim.y * RL;
    int64_t r = (int64_t)blockIdx.y * RL + rl;
    while (r < n_rows) {
      double xv[ES_UNROLL], yv[ES_UNROLL];
      bool in[ES_UNROLL];
#pragma unroll
      for (int u = 0; u < ES_UNROLL; ++u) {  // loads first: ES_UNROLL rows of x and y in flight
        const int64_t ru = r + u * S;
        in[u] = ru < n_rows;
        const int64_t e = (in[u] ? ru : r) * C + col;
        xv[u] = (double)__ldg(x + e);
        yv[u] = (double)__ldg(y + e);
      }
#pragma unroll
      for (int u = 0; u < ES_UNROLL; ++u) {
        if (!in[u]) continue;
        double yy = yv[u];
        const double xx = xv[u];
        if (post) yy = __dadd_rn(__dmul_rn(yy, prg), pmn);
        if (is_int) yy = trunc(yy);
        const bool fx = finite64(xx), fy = finite64(yy);
        a.nfx += !fx;
        a.nfy += !fy;
        if (fx) {
          a.xmin = xx < a.xmin ? xx : a.xmin;
          a.xmax = xx > a.xmax ? xx : a.xmax;
        }
        if (fx && fy) {
          const double e = __dsub_rn(yy, xx);
          const double ae = fabs(e);
          a.cnt += 1;
          a.se = __dadd_rn(a.se, e);
          a.se2 = __dadd_rn(a.se2, __dmul_rn(e, e));
          if (ae > a.mabs) { a.mabs = ae; a.mrow = row0 + r + u * S; }  // rows only grow along a thread: ties keep the first
          if (xx != 0.0) {
            const double resp = __ddiv_rn(__dmul_rn(100.0, e), xx);
            a.rc += 1;
            a.sr = __dadd_rn(a.sr, resp);
            a.sr2 = __dadd_rn(a.sr2, __dmul_rn(resp, resp));
          }
          if (is_int) a.imm += (yy != xx);
#pragma unroll
          for (int k = 0; k < ES_EDGES; ++k) a.cum[k] += (ae > thr[k]);
        }
      }
      r += ES_UNROLL * S;
    }
  }
  // the RL lanes of each column: fixed pairwise tree in shared memory (lane rl takes rl + s when rl % 2s == 0)
  a.store(s_w + t, ES_THREADS);
  __syncthreads();
  for (int s = 1; s < RL; s <<= 1) {
    if (rl < RL && rl % (2 * s) == 0 && rl + s < RL) {
      Acc b;
      b.load(s_w + t + s * TC, ES_THREADS);
      a.fold(b);
      a.store(s_w + t, ES_THREADS);
    }
    __syncthreads();
  }
  if (rl == 0 && col < C) a.store(partial + (int64_t)blockIdx.y * ES_FIELDS * C + col, C);
}

// one warp per column: fold the gy partials in a fixed order, convert the cumulative counts to bins, write the record
__global__ void __launch_bounds__(256)
error_stats_fold_kernel(const unsigned long long* __restrict__ partial, const int gy, const int C,
                        unsigned long long* __restrict__ record) {
  const int lane = threadIdx.x & 31;
  const int col = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  if (col >= C) return;
  Acc a;
  a.init();
  for (int p = lane; p < gy; p += 32) {
    Acc b;
    b.load(partial + (int64_t)p * ES_FIELDS * C + col, C);
    a.fold(b);
  }
  for (int off = 1; off < 32; off <<= 1) {  // lane l meets l ^ off: the lower lane's part first
    Acc b;
    b.cnt = __shfl_xor_sync(0xffffffffu, a.cnt, off);
    b.nfx = __shfl_xor_sync(0xffffffffu, a.nfx, off);
    b.nfy = __shfl_xor_sync(0xffffffffu, a.nfy, off);
    b.rc = __shfl_xor_sync(0xffffffffu, a.rc, off);
    b.imm = __shfl_xor_sync(0xffffffffu, a.imm, off);
    b.mrow = __shfl_xor_sync(0xffffffffu, a.mrow, off);
#pragma unroll
    for (int k = 0; k < ES_EDGES; ++k) b.cum[k] = __shfl_xor_sync(0xffffffffu, a.cum[k], off);
    b.xmin = __shfl_xor_sync(0xffffffffu, a.xmin, off);
    b.xmax = __shfl_xor_sync(0xffffffffu, a.xmax, off);
    b.se = __shfl_xor_sync(0xffffffffu, a.se, off);
    b.se2 = __shfl_xor_sync(0xffffffffu, a.se2, off);
    b.mabs = __shfl_xor_sync(0xffffffffu, a.mabs, off);
    b.sr = __shfl_xor_sync(0xffffffffu, a.sr, off);
    b.sr2 = __shfl_xor_sync(0xffffffffu, a.sr2, off);
    if (lane & off) {  // keep the order (lower lane, higher lane) on both sides: the two lanes compute the same bits
      Acc lo = b;
      lo.fold(a);
      a = lo;
    } else {
      a.fold(b);
    }
  }
  if (lane != 0) return;
  a.store(record + col, C);
  // cumulative counts -> bins: [0, t0], (t0, t1], ..., (t9, inf)
  record[F_HIST * C + col] = a.cnt - a.cum[0];
  for (int k = 1; k < ES_EDGES; ++k) record[(F_HIST + k) * C + col] = a.cum[k - 1] - a.cum[k];
  record[(F_HIST + ES_EDGES) * C + col] = a.cum[ES_EDGES - 1];
  if (a.cnt == 0) record[F_MAXABS * C + col] = (unsigned long long)__double_as_longlong(0.0);
}

template <typename TX, typename TY>
int error_stats_launch(bb_ctx* ctx, const void* x, const void* y, int64_t n_rows, int C, int64_t row0, const double* post_min,
                       const double* post_range, const double* scale_range, const uint8_t* int_mask,
                       unsigned long long* record, cudaStream_t stream) {
  const int TC = C < ES_THREADS ? C : ES_THREADS;
  const int RL = ES_THREADS / TC;
  const int tiles = (C + TC - 1) / TC;
  const int64_t row_groups = (n_rows + RL - 1) / RL;
  int64_t gy = ((int64_t)ctx->sm_count * 4 + tiles - 1) / tiles;
  gy = gy > row_groups ? row_groups : gy;
  const size_t need = (size_t)(gy > 0 ? gy : 1) * ES_FIELDS * C * sizeof(unsigned long long);
  if (ctx->err_scratch_bytes < need) {  // grown once per context for the widest table (see the header)
    if (ctx->err_scratch) BB_CUDA(cudaFree(ctx->err_scratch));
    ctx->err_scratch = nullptr;
    ctx->err_scratch_bytes = 0;
    BB_CUDA(cudaMalloc(&ctx->err_scratch, need));
    ctx->err_scratch_bytes = need;
  }
  unsigned long long* partial = reinterpret_cast<unsigned long long*>(ctx->err_scratch);
  const size_t smem = (size_t)ES_FIELDS * ES_THREADS * sizeof(unsigned long long);
  if (gy > 0) {
    BB_CUDA(cudaFuncSetAttribute(error_stats_kernel<TX, TY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    error_stats_kernel<TX, TY><<<dim3(tiles, (unsigned)gy), ES_THREADS, smem, stream>>>(
        (const TX*)x, (const TY*)y, n_rows, C, TC, RL, row0, post_min, post_range, scale_range, int_mask, partial);
    BB_CUDA(cudaGetLastError());
  }
  error_stats_fold_kernel<<<(C + 7) / 8, 256, 0, stream>>>(partial, (int)gy, C, record);
  return (int)cudaGetLastError();
}

}  // namespace

extern "C" int bb_error_stats(bb_ctx* ctx, const void* x_dev, int x_dtype, const void* y_dev, int y_dtype, int64_t n_rows,
                              int n_cols, int64_t row0, const double* post_min_dev, const double* post_range_dev,
                              const double* scale_range_dev, const uint8_t* int_mask_dev, void* record_dev,
                              bb_stream_t stream) {
  if (!ctx || n_rows < 0 || n_cols < 1 || row0 < 0 || !record_dev || ((!x_dev || !y_dev) && n_rows)) return BB_ERR_INVALID;
  if ((x_dtype != BB_F32 && x_dtype != BB_F64) || (y_dtype != BB_F32 && y_dtype != BB_F64)) return BB_ERR_INVALID;
  if ((post_min_dev == nullptr) != (post_range_dev == nullptr)) return BB_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(record_dev) & 7u) != 0) return BB_ERR_INVALID;
  const uintptr_t x_align = x_dtype == BB_F64 ? 7u : 3u, y_align = y_dtype == BB_F64 ? 7u : 3u;
  if ((reinterpret_cast<uintptr_t>(x_dev) & x_align) || (reinterpret_cast<uintptr_t>(y_dev) & y_align)) return BB_ERR_INVALID;
  if ((reinterpret_cast<uintptr_t>(post_min_dev) | reinterpret_cast<uintptr_t>(post_range_dev) |
       reinterpret_cast<uintptr_t>(scale_range_dev)) & 7u)
    return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t s = (cudaStream_t)stream;
  unsigned long long* rec = reinterpret_cast<unsigned long long*>(record_dev);
  if (x_dtype == BB_F32 && y_dtype == BB_F32)
    return error_stats_launch<float, float>(ctx, x_dev, y_dev, n_rows, n_cols, row0, post_min_dev, post_range_dev,
                                            scale_range_dev, int_mask_dev, rec, s);
  if (x_dtype == BB_F32)
    return error_stats_launch<float, double>(ctx, x_dev, y_dev, n_rows, n_cols, row0, post_min_dev, post_range_dev,
                                             scale_range_dev, int_mask_dev, rec, s);
  if (y_dtype == BB_F32)
    return error_stats_launch<double, float>(ctx, x_dev, y_dev, n_rows, n_cols, row0, post_min_dev, post_range_dev,
                                             scale_range_dev, int_mask_dev, rec, s);
  return error_stats_launch<double, double>(ctx, x_dev, y_dev, n_rows, n_cols, row0, post_min_dev, post_range_dev,
                                            scale_range_dev, int_mask_dev, rec, s);
}
