// Fused dense chain in float64 (DFMA on CUDA cores): [normalise ->] L dense layers [-> un-normalise].
//
// The reference's AE / AE_Dropout_BN are float64 models: helper.compress / helper.decompress run them in float64 and
// write float64 files (reference baler/modules/helper.py:565, 653; baler.py:410-456).  This kernel computes what they
// compute, in the same arithmetic, for every dense chain of at most 8 layers whose widths are all <= 256.
//
// Normalisation on the way in is a true IEEE subtract + divide in the INPUT's dtype (data_processing.py:133-153): a
// float32 table is normalised in float32, bit-equal to numpy, and then widened (the reference converts to a float64
// tensor only after normalising); a float64 table is normalised in float64.  Un-normalisation on the way out is
// y * range + min in float64 with the features widened exactly, one rounding per operation like numpy (no FMA
// contraction; data_processing.py:188-203).  Each output is a sequential sum over k in layer order, so a row's bits do not
// depend on the tile, the chunk or the rank it went through.
//
// Layout.  One persistent CTA per SM, 256 threads.  A tile of TR rows (64, or 32 when shared memory does not hold two
// 64-row activation buffers of the chain's widths) goes through all layers on chip; activations are kept TRANSPOSED in
// shared memory, act[feature][TRP] (TRP = TR + 2: 16-byte aligned rows, fewer bank conflicts on the transposing loads).
// The weights do not fit: the CMS encoder alone is 30,915 doubles = 247 KB.  Each layer's Wt[Kpad][Npad] (k-major, K
// zero-padded to whole chunks) is streamed from L2 in chunks of KC = 16 k-rows through a two-stage cp.async ring, the
// next chunk (of this layer, of the next layer, or of the next tile) landing while the current one is multiplied.
// Each thread owns a (TR / 8) x TN block of a layer's output: rows {16 q + 2 rt, 16 q + 2 rt + 1} for q < TR / 16,
// TN consecutive features, with TN (8, 4, 2 or 1) the smallest that lets 8 * ceil(N / TN) <= 256 threads cover N.
//
// Budget (per CTA).  Shared memory: ring 2 x KC x max_npad x 8 B + activations (buf_rows[0] + buf_rows[1]) x TRP x 8 B.
// CMS AE (24-200-100-50-15): 51 KB + 300 x 66 x 8 B = 209 KB at TR = 64; the widest chain (256 everywhere) 64 KB +
// 512 x 34 x 8 B = 203 KB at TR = 32.  Registers: TR = 64, TN = 8 holds 64 double accumulators (128 registers) plus
// 8 + 8 operands; the build is checked for spills with -Xptxas -v.
//
// FLOP: 2 x 30,550 per CMS row and direction (61,100).  DFMA rather than DMMA: on this card both pipes have the same
// datasheet FP64 rate (tools/fp64_rate_bench.cu measures both; profiles/r03_fp64_rate.txt), and DFMA keeps the
// summation order of the reference-order numpy chain with no fragment shuffles.
#include "bb_common.cuh"

namespace {

constexpr int NT = 256;
constexpr int KC = 16;     // k-rows of a weight chunk
constexpr int MAXW = 256;  // widest layer the kernel takes

__device__ __forceinline__ double act_f64(double v, int act) {
  if (act == BB_ACT_LEAKY) return v > 0.0 ? v : __dmul_rn(0.01, v);  // F.leaky_relu: slope 0.01 in the model's dtype
  if (act == BB_ACT_RELU) return v > 0.0 ? v : (v == v ? 0.0 : v);   // torch relu: max(v, 0), NaN stays NaN
  return v;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// The weight chunk after (layer l, first k-row k0) in the stream the CTA walks: the rest of this layer, then the next
// layer, then (next tile) layer 0 again.
struct ChunkPos {
  int l, k0;
};
__device__ __forceinline__ ChunkPos next_chunk(const F64Desc& d, ChunkPos p) {
  p.k0 += KC;
  if (p.k0 >= d.layer[p.l].Kpad) {
    p.k0 = 0;
    p.l = (p.l + 1 == d.n_layers) ? 0 : p.l + 1;
  }
  return p;
}
__device__ __forceinline__ void issue_chunk(const F64Desc& d, const double* __restrict__ blob, ChunkPos p, double* ring_stage) {
  const F64Layer& L = d.layer[p.l];
  const double* src = blob + L.w_off + (size_t)p.k0 * L.Npad;
  const int n16 = KC * L.Npad / 2;
  for (int i = threadIdx.x; i < n16; i += NT) cp_async16(ring_stage + 2 * i, src + 2 * i);
  cp_async_commit();
}

// One layer: O[c][r] = act(sum_k A[k][r] * W[k][c] + bias[c]), W streamed chunk by chunk through the ring.
// On entry the chunk (l, 0) is in flight into ring stage `stage`; on exit the chunk after this layer's last is in flight.
template <int TR, int TN>
__device__ __forceinline__ void dense_layer(const F64Desc& d, const double* __restrict__ blob, int l,
                                            const double* __restrict__ A, double* __restrict__ O, double* ring,
                                            int& stage) {
  constexpr int TRP = TR + 2, RT = 8, Q = TR / 16;  // 8 row groups; Q row pairs per thread
  const F64Layer& L = d.layer[l];
  const int stage_elems = KC * d.max_npad;
  const int n_ct = L.Npad / TN;
  const int idx = threadIdx.x;
  const bool active = idx < n_ct * RT;
  const int ct = idx / RT, rt = idx - (idx / RT) * RT;
  double acc[2 * Q][TN];
#pragma unroll
  for (int i = 0; i < 2 * Q; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.0;
  ChunkPos pos{l, 0};
  for (int k0 = 0; k0 < L.Kpad; k0 += KC) {
    cp_async_wait_all();
    __syncthreads();  // chunk k0 landed for every thread; the other stage (previous chunk) is no longer read
    issue_chunk(d, blob, next_chunk(d, pos), ring + (stage ^ 1) * stage_elems);
    pos = next_chunk(d, pos);
    if (active) {
      const double* w = ring + stage * stage_elems + ct * TN;
      const double* a = A + (size_t)k0 * TRP + 2 * rt;
      const int kn = min(KC, L.K - k0);  // rows past K: zero weights, but the activation rows there are not defined
      for (int kk = 0; kk < kn; ++kk) {
        double av[2 * Q];
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          const double2 v = *reinterpret_cast<const double2*>(a + 16 * q);
          av[2 * q] = v.x;
          av[2 * q + 1] = v.y;
        }
        double wv[TN];
        if constexpr (TN == 1) {
          wv[0] = w[0];
        } else {
#pragma unroll
          for (int j = 0; j < TN; j += 2) {
            const double2 v = *reinterpret_cast<const double2*>(w + j);
            wv[j] = v.x;
            wv[j + 1] = v.y;
          }
        }
#pragma unroll
        for (int i = 0; i < 2 * Q; ++i)
#pragma unroll
          for (int j = 0; j < TN; ++j) acc[i][j] = fma(av[i], wv[j], acc[i][j]);
        a += TRP;
        w += L.Npad;
      }
    }
    stage ^= 1;
  }
  if (active) {
    const double* bias = blob + L.b_off;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int c = ct * TN + j;
      const double b = __ldg(bias + c);
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        double2 o;
        o.x = act_f64(__dadd_rn(acc[2 * q][j], b), L.act);
        o.y = act_f64(__dadd_rn(acc[2 * q + 1][j], b), L.act);
        *reinterpret_cast<double2*>(O + (size_t)c * TRP + 16 * q + 2 * rt) = o;
      }
    }
  }
}

template <int TR>
__device__ __forceinline__ void run_layer(const F64Desc& d, const double* __restrict__ blob, int l, const double* A,
                                          double* O, double* ring, int& stage) {
  switch (d.layer[l].tn) {
    case 8: dense_layer<TR, 8>(d, blob, l, A, O, ring, stage); break;
    case 4: dense_layer<TR, 4>(d, blob, l, A, O, ring, stage); break;
    case 2: dense_layer<TR, 2>(d, blob, l, A, O, ring, stage); break;
    default: dense_layer<TR, 1>(d, blob, l, A, O, ring, stage); break;
  }
}

__device__ __forceinline__ double feat(const void* p, int dtype, int c) {
  return dtype == BB_F64 ? __ldg(reinterpret_cast<const double*>(p) + c) : (double)__ldg(reinterpret_cast<const float*>(p) + c);
}

template <int TR>
__global__ void __launch_bounds__(NT, 1)
chain_f64_kernel(const __grid_constant__ F64Desc d, const double* __restrict__ blob, const void* __restrict__ in,
                 const int in_dtype, const int64_t n_rows, const void* __restrict__ pre_min,
                 const void* __restrict__ pre_range, const void* __restrict__ post_min,
                 const void* __restrict__ post_range, const int feat_dtype, void* __restrict__ out, const int out_dtype) {
  constexpr int TRP = TR + 2;
  extern __shared__ __align__(16) double smem[];
  double* ring = smem;
  double* buf0 = ring + 2 * KC * d.max_npad;
  double* buf1 = buf0 + d.buf_rows[0] * TRP;
  int stage = 0;
  issue_chunk(d, blob, ChunkPos{0, 0}, ring);

  const int in_dim = d.in_dim, out_dim = d.out_dim;
  const int64_t n_tiles = (n_rows + TR - 1) / TR;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int rows = (int)min((int64_t)TR, n_rows - tile * TR);
    {  // load pass: row-major global tile -> buf0[feature][row], normalised in the input's dtype, widened
      const int64_t base = tile * TR * (int64_t)in_dim;
      const int n_el = rows * in_dim;
      for (int e = threadIdx.x; e < TR * in_dim; e += NT) {
        const int r = e / in_dim, c = e - r * in_dim;
        double v = 0.0;
        if (e < n_el) {
          if (in_dtype == BB_F64) {
            v = __ldg(reinterpret_cast<const double*>(in) + base + e);
            if (pre_min != nullptr) v = __ddiv_rn(__dsub_rn(v, feat(pre_min, feat_dtype, c)), feat(pre_range, feat_dtype, c));
          } else {
            float f = (in_dtype == BB_F16) ? __half2float(reinterpret_cast<const __half*>(in)[base + e])
                                           : __ldg(reinterpret_cast<const float*>(in) + base + e);
            if (pre_min != nullptr && feat_dtype == BB_F32) {  // numpy float32: (x - min) / range (data_processing.py:151)
              f = __fdiv_rn(__fsub_rn(f, __ldg(reinterpret_cast<const float*>(pre_min) + c)),
                            __ldg(reinterpret_cast<const float*>(pre_range) + c));
              v = (double)f;
            } else {
              v = (double)f;
              if (pre_min != nullptr) v = __ddiv_rn(__dsub_rn(v, feat(pre_min, feat_dtype, c)), feat(pre_range, feat_dtype, c));
            }
          }
        }
        buf0[c * TRP + r] = v;
      }
    }
    double* cur = buf0;
    double* nxt = buf1;
    for (int l = 0; l < d.n_layers; ++l) {  // (the first chunk's barrier publishes the load pass / the previous layer)
      run_layer<TR>(d, blob, l, cur, nxt, ring, stage);
      double* t = cur; cur = nxt; nxt = t;
    }
    __syncthreads();
    {  // store pass: cur[feature][row] -> row-major global tile, un-normalised in float64
      const int64_t base = tile * TR * (int64_t)out_dim;
      const int n_el = rows * out_dim;
      for (int e = threadIdx.x; e < n_el; e += NT) {
        const int r = e / out_dim, c = e - r * out_dim;
        double v = cur[c * TRP + r];
        // reference: y * range + min (data_processing.py:203)
        if (post_min != nullptr) v = __dadd_rn(__dmul_rn(v, feat(post_range, feat_dtype, c)), feat(post_min, feat_dtype, c));
        if (out_dtype == BB_F64) reinterpret_cast<double*>(out)[base + e] = v;
        else if (out_dtype == BB_F16) reinterpret_cast<__half*>(out)[base + e] = __double2half(v);
        else reinterpret_cast<float*>(out)[base + e] = __double2float_rn(v);
      }
    }
    __syncthreads();
  }
  cp_async_wait_all();  // the prefetch of a tile that does not come
}

size_t f64_smem_bytes(const F64Desc& d, int tr) {
  return ((size_t)2 * KC * d.max_npad + (size_t)(d.buf_rows[0] + d.buf_rows[1]) * (tr + 2)) * sizeof(double);
}

}  // namespace

// Plans the layers, packs Wt[Kpad][Npad] + bias in float64 from the host copies and uploads them (first fp64 call only).
int bb_chain_f64_prepare(bb_ctx* ctx, const Chain* c) {
  if (c->f64_blob_dev) return BB_OK;
  const ChainDesc& cd = c->desc;
  F64Desc d = {};
  d.n_layers = cd.n_layers;
  d.in_dim = cd.in_dim;
  d.out_dim = cd.out_dim;
  if (d.in_dim > MAXW) return BB_ERR_UNSUPPORTED;
  int off = 0;
  d.max_npad = 2;
  d.buf_rows[0] = d.in_dim;
  d.buf_rows[1] = 0;
  for (int l = 0; l < d.n_layers; ++l) {
    F64Layer& L = d.layer[l];
    L.K = cd.layer[l].K;
    L.N = cd.layer[l].N;
    L.act = cd.layer[l].act;
    if (L.K > MAXW || L.N > MAXW) return BB_ERR_UNSUPPORTED;
    int tn = 8;
    for (int cand = 1; cand <= 8; cand *= 2)
      if (((L.N + cand - 1) / cand) * 8 <= NT) { tn = cand; break; }
    L.tn = tn;
    const int step = tn < 2 ? 2 : tn;  // even row length: 16-byte cp.async of the chunks
    L.Npad = ((L.N + step - 1) / step) * step;
    L.Kpad = ((L.K + KC - 1) / KC) * KC;
    L.w_off = off;
    off += L.Kpad * L.Npad;
    L.b_off = off;
    off += L.Npad;
    if (L.Npad > d.max_npad) d.max_npad = L.Npad;
    int& b = d.buf_rows[(l + 1) & 1];  // buf0 holds the input and the outputs of odd layers, buf1 the others
    if (L.Npad > b) b = L.Npad;
  }
  d.tr = f64_smem_bytes(d, 64) <= ctx->smem_optin ? 64 : 32;
  if (f64_smem_bytes(d, d.tr) > ctx->smem_optin) return BB_ERR_UNSUPPORTED;

  std::vector<double> blob((size_t)off, 0.0);
  for (int l = 0; l < d.n_layers; ++l) {
    const F64Layer& L = d.layer[l];
    const std::vector<double>& w = c->w_host[l];
    const std::vector<double>& b = c->b_host[l];
    for (int n = 0; n < L.N; ++n) {
      for (int k = 0; k < L.K; ++k) blob[(size_t)L.w_off + (size_t)k * L.Npad + n] = w[(size_t)n * L.K + k];
      blob[(size_t)L.b_off + n] = b[n];
    }
  }
  double* dev = nullptr;
  BB_CUDA(cudaMalloc(&dev, blob.size() * sizeof(double)));
  const cudaError_t e = cudaMemcpy(dev, blob.data(), blob.size() * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cudaFree(dev);
    return (int)e;
  }
  const int max_dyn = (int)ctx->smem_optin;
  BB_CUDA(cudaFuncSetAttribute(chain_f64_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  BB_CUDA(cudaFuncSetAttribute(chain_f64_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  c->f64 = d;
  c->f64_smem = f64_smem_bytes(d, d.tr);
  c->f64_blob_dev = dev;
  return BB_OK;
}

void bb_chain_f64_release(const Chain* c) {
  if (c->f64_blob_dev) cudaFree(c->f64_blob_dev);
  c->f64_blob_dev = nullptr;
  c->f64_smem = 0;
}

int bb_chain_f64_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows, const void* pre_min,
                        const void* pre_range, const void* post_min, const void* post_range, int feat_dtype, void* out,
                        int out_dtype, cudaStream_t stream) {
  if ((in_dtype != BB_F32 && in_dtype != BB_F16 && in_dtype != BB_F64) ||
      (out_dtype != BB_F32 && out_dtype != BB_F16 && out_dtype != BB_F64) || (feat_dtype != BB_F32 && feat_dtype != BB_F64))
    return BB_ERR_INVALID;
  const int rc = bb_chain_f64_prepare(ctx, c);
  if (rc != BB_OK) return rc;
  if (n_rows == 0) return BB_OK;
  const int tr = c->f64.tr;
  const int64_t n_tiles = (n_rows + tr - 1) / tr;
  const int grid = (int)(n_tiles < ctx->sm_count ? n_tiles : ctx->sm_count);
  c->last_route = BB_ROUTE_F64;
  c->last_tile_rows = tr;
  if (tr == 64)
    chain_f64_kernel<64><<<grid, NT, c->f64_smem, stream>>>(c->f64, c->f64_blob_dev, in, in_dtype, n_rows, pre_min, pre_range,
                                                            post_min, post_range, feat_dtype, out, out_dtype);
  else
    chain_f64_kernel<32><<<grid, NT, c->f64_smem, stream>>>(c->f64, c->f64_blob_dev, in, in_dtype, n_rows, pre_min, pre_range,
                                                            post_min, post_range, feat_dtype, out, out_dtype);
  return (int)cudaGetLastError();
}
