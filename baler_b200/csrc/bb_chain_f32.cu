// Fused dense chain on CUDA cores (fp32 FFMA): [normalise ->] L dense layers [-> un-normalise].
//
// Replaces the per-batch `model.encode` / `model.decode` calls of helper.compress / helper.decompress
// (reference baler/modules/helper.py:583-611, 701-723) together with the column normalisation
// (data_processing.py:133-153) and its inverse (data_processing.py:188-203).
//
// Layout.  One persistent CTA per SM, 256 threads.  All layer weights of one direction live in
// shared memory for the whole kernel as Wt[K][Npad] (k-major) + bias[Npad].  A tile of TR rows
// of the table is processed at a time; activations are kept TRANSPOSED in shared memory,
// act[feature][TRP] (TRP = TR + 4), so that both operands of the outer-product FMA loop are read
// with 128-bit LDS along the fast axis.  Each thread owns an 8 x TN block of the layer output
// (rows {4rt..4rt+3} and {TR/2+4rt..}, TN consecutive features), with TN picked per layer on the
// host so that (TR/8) * ceil(N/TN) just fills the 256 threads (hidden widths 200/100/50 and
// TR = 80 give 250 active threads: TN = 8/4/2).
//
// HBM traffic per row is exactly one read of the input row and one write of the output row; this
// kernel is bound by the fp32 FMA pipe (2 * 30,550 FLOP per row for the CMS AE), not by HBM.  It is
// the reference-accuracy path (max-norm error ~2e-7 against the float64 reference) and the fallback
// of the tcgen05 split-fp16 kernel (bb_chain_tc.cu) for shapes / value ranges that kernel rejects.
#include "bb_common.cuh"

namespace {

constexpr int NT = 256;

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == BB_ACT_LEAKY) return v > 0.f ? v : BB_LEAKY * v;
  if (act == BB_ACT_RELU) return fmaxf(v, 0.f);
  return v;
}

template <int TN>
__device__ __forceinline__ void load_w(const float* w, float (&wv)[TN]) {
  if constexpr (TN == 8) {
    const float4 w0 = *reinterpret_cast<const float4*>(w);
    const float4 w1 = *reinterpret_cast<const float4*>(w + 4);
    wv[0] = w0.x; wv[1] = w0.y; wv[2] = w0.z; wv[3] = w0.w;
    wv[4] = w1.x; wv[5] = w1.y; wv[6] = w1.z; wv[7] = w1.w;
  } else if constexpr (TN == 4) {
    const float4 w0 = *reinterpret_cast<const float4*>(w);
    wv[0] = w0.x; wv[1] = w0.y; wv[2] = w0.z; wv[3] = w0.w;
  } else if constexpr (TN == 2) {
    const float2 w0 = *reinterpret_cast<const float2*>(w);
    wv[0] = w0.x; wv[1] = w0.y;
  } else {
    wv[0] = *w;
  }
}

// out[c][r] = act(sum_k A[k][r] * W[k][c] + bias[c]) for an 8 x TN block per thread.
template <int TR, int TN>
__device__ __forceinline__ void dense_tile(const float* __restrict__ A, const float* __restrict__ W,
                                           const float* __restrict__ bias, float* __restrict__ O,
                                           const int K, const int Npad, const int act) {
  constexpr int TRP = TR + 4, RT = TR / 8, H = TR / 2;
  const int n_ct = Npad / TN;
  for (int idx = threadIdx.x; idx < n_ct * RT; idx += NT) {
    const int ct = idx / RT, rt = idx - ct * RT;
    float acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
    const float* a = A + 4 * rt;
    const float* w = W + ct * TN;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(a);
      const float4 a1 = *reinterpret_cast<const float4*>(a + H);
      float wv[TN];
      load_w<TN>(w, wv);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
      a += TRP;
      w += Npad;
    }
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int c = ct * TN + j;
      const float b = bias[c];
      float4 o0, o1;
      o0.x = apply_act(acc[0][j] + b, act); o0.y = apply_act(acc[1][j] + b, act);
      o0.z = apply_act(acc[2][j] + b, act); o0.w = apply_act(acc[3][j] + b, act);
      o1.x = apply_act(acc[4][j] + b, act); o1.y = apply_act(acc[5][j] + b, act);
      o1.z = apply_act(acc[6][j] + b, act); o1.w = apply_act(acc[7][j] + b, act);
      *reinterpret_cast<float4*>(O + c * TRP + 4 * rt) = o0;
      *reinterpret_cast<float4*>(O + c * TRP + H + 4 * rt) = o1;
    }
  }
}

template <int TR>
__global__ void __launch_bounds__(NT, 1)
chain_f32_kernel(const __grid_constant__ ChainDesc d, const float* __restrict__ blob,
                 const void* __restrict__ in, const int in_dtype, const int64_t n_rows,
                 const float* __restrict__ pre_min, const float* __restrict__ pre_range,
                 const float* __restrict__ post_min, const float* __restrict__ post_range,
                 void* __restrict__ out, const int out_dtype) {
  constexpr int TRP = TR + 4;
  extern __shared__ __align__(16) float smem[];
  float* wsm = smem;
  float* buf0 = wsm + ((d.blob_floats + 3) & ~3);
  float* buf1 = buf0 + d.buf_rows[0] * TRP;

  {  // weights: global (L2) -> shared, once per CTA
    const float4* src = reinterpret_cast<const float4*>(blob);
    float4* dst = reinterpret_cast<float4*>(wsm);
    const int n4 = (d.blob_floats + 3) >> 2;
    for (int i = threadIdx.x; i < n4; i += NT) dst[i] = __ldg(src + i);
  }
  __syncthreads();

  const int in_dim = d.in_dim, out_dim = d.out_dim;
  const int64_t n_tiles = (n_rows + TR - 1) / TR;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int rows = (int)min((int64_t)TR, n_rows - tile * TR);
    {  // load pass: row-major global tile -> buf0[feature][row], normalised
      const int64_t base = tile * TR * (int64_t)in_dim;
      const int n_el = rows * in_dim;
      for (int e = threadIdx.x; e < TR * in_dim; e += NT) {
        const int r = e / in_dim, c = e - r * in_dim;
        float v = 0.f;
        if (e < n_el) {
          v = (in_dtype == BB_F16) ? __half2float(reinterpret_cast<const __half*>(in)[base + e])
                                   : __ldg(reinterpret_cast<const float*>(in) + base + e);
          // numpy float32: (x - min) / range with IEEE division (data_processing.py:151)
          if (pre_min != nullptr) v = __fdiv_rn(__fsub_rn(v, __ldg(pre_min + c)), __ldg(pre_range + c));
        }
        buf0[c * TRP + r] = v;
      }
    }
    __syncthreads();
    float* cur = buf0;
    float* nxt = buf1;
    for (int l = 0; l < d.n_layers; ++l) {
      const ChainLayer& L = d.layer[l];
      const float* W = wsm + L.w_off;
      const float* B = wsm + L.b_off;
      switch (L.tn) {
        case 8: dense_tile<TR, 8>(cur, W, B, nxt, L.K, L.Npad, L.act); break;
        case 4: dense_tile<TR, 4>(cur, W, B, nxt, L.K, L.Npad, L.act); break;
        case 2: dense_tile<TR, 2>(cur, W, B, nxt, L.K, L.Npad, L.act); break;
        default: dense_tile<TR, 1>(cur, W, B, nxt, L.K, L.Npad, L.act); break;
      }
      __syncthreads();
      float* t = cur; cur = nxt; nxt = t;
    }
    {  // store pass: cur[feature][row] -> row-major global tile, un-normalised
      const int64_t base = tile * TR * (int64_t)out_dim;
      const int n_el = rows * out_dim;
      for (int e = threadIdx.x; e < n_el; e += NT) {
        const int r = e / out_dim, c = e - r * out_dim;
        float v = cur[c * TRP + r];
        // reference: y * range + min (data_processing.py:203)
        if (post_min != nullptr) v = fmaf(v, __ldg(post_range + c), __ldg(post_min + c));
        if (out_dtype == BB_F16) reinterpret_cast<__half*>(out)[base + e] = __float2half_rn(v);
        else reinterpret_cast<float*>(out)[base + e] = v;
      }
    }
    __syncthreads();
  }
}

size_t f32_smem_bytes(const ChainDesc& d, int tr) {
  return (size_t)(((d.blob_floats + 3) & ~3) + (d.buf_rows[0] + d.buf_rows[1]) * (tr + 4)) * sizeof(float);
}

}  // namespace

// Picks the thread tile per layer, packs Wt[K][Npad] + bias and uploads the blob.
int bb_chain_f32_prepare(bb_ctx* ctx, Chain* c) {
  ChainDesc& d = c->desc;
  // the tile height is fixed first (it decides TN); try the tallest tile whose smem fits
  const int trs[3] = {80, 64, 32};
  int chosen = -1;
  for (int t = 0; t < 3 && chosen < 0; ++t) {
    const int tr = trs[t], rt = tr / 8;
    int off = 0;
    for (int l = 0; l < d.n_layers; ++l) {
      ChainLayer& L = d.layer[l];
      int tn = 8;
      for (int cand = 1; cand <= 8; cand *= 2)
        if (((L.N + cand - 1) / cand) * rt <= NT) { tn = cand; break; }
      L.tn = tn;
      L.Npad = ((L.N + tn - 1) / tn) * tn;
      off = (off + 3) & ~3;
      L.w_off = off;
      off += L.K * L.Npad;
      off = (off + 3) & ~3;
      L.b_off = off;
      off += L.Npad;
    }
    d.blob_floats = off;
    // ping-pong buffers: buf0 holds the input and the outputs of odd layers, buf1 the others
    d.buf_rows[0] = d.in_dim;
    d.buf_rows[1] = 0;
    for (int l = 0; l < d.n_layers; ++l) {
      int& b = d.buf_rows[(l + 1) & 1];
      if (d.layer[l].Npad > b) b = d.layer[l].Npad;
    }
    if (f32_smem_bytes(d, tr) <= ctx->smem_optin) chosen = tr;
  }
  if (chosen < 0) return BB_ERR_UNSUPPORTED;
  c->f32_tr = chosen;
  c->smem_bytes = f32_smem_bytes(d, chosen);

  // whole float4s: the kernel copies the blob to shared memory with (blob_floats + 3) / 4 float4 loads (zero tail)
  std::vector<float> blob(((size_t)d.blob_floats + 3) & ~(size_t)3, 0.f);
  for (int l = 0; l < d.n_layers; ++l) {
    const ChainLayer& L = d.layer[l];
    const std::vector<double>& w = c->w_host[l];
    const std::vector<double>& b = c->b_host[l];
    for (int n = 0; n < L.N; ++n) {
      for (int k = 0; k < L.K; ++k) blob[(size_t)L.w_off + (size_t)k * L.Npad + n] = (float)w[(size_t)n * L.K + k];
      blob[(size_t)L.b_off + n] = (float)b[n];
    }
  }
  if (c->blob_dev) cudaFree(c->blob_dev);
  BB_CUDA(cudaMalloc(&c->blob_dev, blob.size() * sizeof(float)));
  BB_CUDA(cudaMemcpy(c->blob_dev, blob.data(), blob.size() * sizeof(float), cudaMemcpyHostToDevice));
  // the attribute belongs to the kernel, not to this chain (encoder and decoder share it): allow the device maximum
  const int max_dyn = (int)ctx->smem_optin;
  BB_CUDA(cudaFuncSetAttribute(chain_f32_kernel<80>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  BB_CUDA(cudaFuncSetAttribute(chain_f32_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  BB_CUDA(cudaFuncSetAttribute(chain_f32_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  return BB_OK;
}

int bb_chain_f32_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows,
                        const float* pre_min, const float* pre_range, const float* post_min,
                        const float* post_range, void* out, int out_dtype, cudaStream_t stream) {
  if (n_rows == 0) return BB_OK;
  const int tr = c->f32_tr;
  const int64_t n_tiles = (n_rows + tr - 1) / tr;
  const int grid = (int)(n_tiles < ctx->sm_count ? n_tiles : ctx->sm_count);
  c->last_route = BB_ROUTE_F32;
  c->last_tile_rows = tr;
  switch (tr) {
    case 80:
      chain_f32_kernel<80><<<grid, NT, c->smem_bytes, stream>>>(c->desc, c->blob_dev, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out, out_dtype);
      break;
    case 64:
      chain_f32_kernel<64><<<grid, NT, c->smem_bytes, stream>>>(c->desc, c->blob_dev, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out, out_dtype);
      break;
    default:
      chain_f32_kernel<32><<<grid, NT, c->smem_bytes, stream>>>(c->desc, c->blob_dev, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out, out_dtype);
      break;
  }
  return (int)cudaGetLastError();
}
