// Layer-by-layer fp32 trainer for dense autoencoders whose weight matrices do not fit the fused training kernels'
// shared memory: `CFD_dense_AE` on 2500-feature snapshots (models.py:186-226; W1 and W8 are 200 x 2500), or any dense
// chain of up to BB_MAX_LAYERS Linears.  Same arithmetic contract as bb_train.cu (training.py:31-101: forward,
// sum-MSE / n_columns, backward, Adam with the reference's defaults, loss accumulated on the device), one GEMM launch
// per matrix product instead of one fused kernel:
//     forward   A_{l+1} = act(A_l W_l^T + b_l)                       gemm<NT> + bias + activation epilogue
//     loss      sum((A_L - x)^2) / C,   dA_L = 2 (A_L - x) / C       elementwise + block reduction
//     backward  dZ_l = dA_{l+1} * act'(A_{l+1});  dW_l = dZ_l^T A_l;  db_l = colsum(dZ_l);  dA_l = dZ_l W_l
//     Adam      torch.optim.Adam single-tensor update (training.py:266)
// Shapes here are small-batch x wide (60 x 2500): the GEMMs are latency-bound either way, so the kernel is a plain
// 64 x 64 x 16 shared-memory tile with arbitrary strides (one kernel serves NT, NN and TN), not a tuned one.
//
// `Conv_AE` (models.py:316-407) trains through the same chain (bb_ltrainer_create_ex): on a fixed block shape every
// (transposed) convolution is a linear map of the flattened tensor, i.e. a dense matrix whose entries are shared kernel
// weights or structural zeros.  Such a layer keeps its TRAINABLE parameters (kernel, per-channel bias) apart from the
// dense matrix the GEMMs read:
//     expand    Wd[i] = w[map[i]] (0 where map[i] < 0),  bd[n] = b[n / S]         after every Adam step
//     reduce    dw[j] = sum of dWd over the entries that share kernel weight j      (CSR lists, fixed order)
// BatchNorm2d between the affine map and the activation (train mode: batch statistics over rows x positions of a
// channel, biased variance, eps 1e-5, running statistics with momentum 0.1 and the unbiased variance; eval mode: the
// running statistics), one block per channel:
//     forward   xhat = (z - mean) * rstd,  y = gamma * xhat + beta
//     backward  dgamma = sum(dy * xhat),  dbeta = sum(dy),  dz = gamma * rstd * (dy - dbeta / M - xhat * dgamma / M)
//
// `AE_Dropout_BN` (models.py:256-313) trains through the same chain (bb_ltrainer_create_dbn) at any batch size; the fused
// dbn steps need every CTA of a batch resident.  Its two extra layer kinds:
//     dropout   encoder: Linear -> Dropout(p) -> LeakyReLU; keep-bits from bb_philox_keep(seed, step, layer, row, column)
//               (the stream of the fused fp32 / tensor-core dbn steps) or injected masks, kept values x fp32(1 / (1 - p))
//     BN after  decoder layers 0-2: Linear -> LeakyReLU -> BatchNorm1d (the last one keeps Linear -> BatchNorm1d -> ReLU);
//               the pre-BatchNorm activation is kept for LeakyReLU' in the backward pass
#include <cmath>
#include <cstdlib>
#include <vector>

#include "bb_common.cuh"
#include "bb_train_f64.cuh"  // bb_philox_keep

namespace {

constexpr int TM = 64, TN = 64, TK = 16, GT = 256;

__device__ __forceinline__ float act_fwd(float v, int act) {
  if (act == BB_ACT_LEAKY) return v > 0.f ? v : BB_LEAKY * v;
  if (act == BB_ACT_RELU) return fmaxf(v, 0.f);
  return v;
}

// C[m][n] = sum_k A(m, k) * B(k, n) with A(m, k) = A[m * sam + k * sak], B(k, n) = B[k * sbk + n * sbn];
// epilogue: + bias[n], activation; fixed summation order (k ascending: the same bits whatever the tile size), one thread
// per (TM_ / 16) x (TN_ / 16) outputs.  64 x 64 tiles by default, 32 x 32 when those would leave most SMs without a CTA.
// The small tile takes 64-wide k slabs (a quarter of the barriers; the per-output k order, hence the bits, are unchanged).
// The next k slab is fetched into registers while the current one is multiplied (the batches here are a few hundred
// rows: one CTA per SM at best, nothing else hides the global-memory latency).  Split-K (gridDim.z > 1): CTA z takes the
// k range [z * k_per, (z + 1) * k_per) and writes its partial tile to C + z * split_stride without the epilogue;
// splitk_reduce_kernel adds the partials in z order.  The K = 2000 products of Conv_AE (N = 128 or 250: 40 - 150 CTAs with
// a 125-iteration k loop) and the weight-gradient products (k = batch rows) run that way.
template <int TM_, int TN_, int TK_>
__global__ void __launch_bounds__(GT)
gemm_strided_kernel(const float* __restrict__ A, const int64_t sam, const int64_t sak, const float* __restrict__ B,
                    const int64_t sbk, const int64_t sbn, float* __restrict__ C, const int64_t ldc, const int M, const int N,
                    const int K, const float* __restrict__ bias, const int act, const int k_per, const int64_t split_stride) {
  constexpr int RM = TM_ / 16, RN = TN_ / 16, EA = TK_ * TM_ / GT, EB = TK_ * TN_ / GT;
  __shared__ float As[TK_][TM_ + 1];
  __shared__ float Bs[TK_][TN_ + 1];
  const int m0 = blockIdx.y * TM_, n0 = blockIdx.x * TN_;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int k_begin = blockIdx.z * k_per, k_end = k_begin + k_per < K ? k_begin + k_per : K;
  float acc[RM][RN] = {};
  float ra[EA], rb[EB];
  auto fetch = [&](const int k0) {
#pragma unroll
    for (int i = 0; i < EA; ++i) {
      const int e = tid + i * GT, kk = e / TM_, mm = e - kk * TM_;
      const int m = m0 + mm, k = k0 + kk;
      ra[i] = (m < M && k < k_end) ? __ldg(A + (int64_t)m * sam + (int64_t)k * sak) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < EB; ++i) {
      const int e = tid + i * GT, kk = e / TN_, nn = e - kk * TN_;
      const int n = n0 + nn, k = k0 + kk;
      rb[i] = (n < N && k < k_end) ? __ldg(B + (int64_t)k * sbk + (int64_t)n * sbn) : 0.f;
    }
  };
  fetch(k_begin);
  for (int k0 = k_begin; k0 < k_end; k0 += TK_) {
#pragma unroll
    for (int i = 0; i < EA; ++i) {
      const int e = tid + i * GT, kk = e / TM_;
      As[kk][e - kk * TM_] = ra[i];
    }
#pragma unroll
    for (int i = 0; i < EB; ++i) {
      const int e = tid + i * GT, kk = e / TN_;
      Bs[kk][e - kk * TN_] = rb[i];
    }
    __syncthreads();
    if (k0 + TK_ < k_end) fetch(k0 + TK_);
#pragma unroll
    for (int kk = 0; kk < TK_; ++kk) {
      float a[RM], b[RN];
#pragma unroll
      for (int i = 0; i < RM; ++i) a[i] = As[kk][ty * RM + i];
#pragma unroll
      for (int j = 0; j < RN; ++j) b[j] = Bs[kk][tx * RN + j];
#pragma unroll
      for (int i = 0; i < RM; ++i)
#pragma unroll
        for (int j = 0; j < RN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  const bool split = gridDim.z > 1;
  float* Cz = C + (int64_t)blockIdx.z * split_stride;
#pragma unroll
  for (int i = 0; i < RM; ++i) {
    const int m = m0 + ty * RM + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < RN; ++j) {
      const int n = n0 + tx * RN + j;
      if (n < N) Cz[(int64_t)m * ldc + n] = split ? acc[i][j] : act_fwd(acc[i][j] + (bias ? __ldg(bias + n) : 0.f), act);
    }
  }
}

// C[m][n] = act(sum_z part[z][m][n] + bias[n]), z ascending (reproducible)
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ part, const int S, const int64_t split_stride,
                                                            float* __restrict__ C, const int64_t ldc, const int M, const int N,
                                                            const float* __restrict__ bias, const int act) {
  const int64_t total = (int64_t)M * N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int m = (int)(e / N), n = (int)(e - (int64_t)m * N);
    float v = 0.f;
    for (int z = 0; z < S; ++z) v += part[(int64_t)z * split_stride + (int64_t)m * ldc + n];
    C[(int64_t)m * ldc + n] = act_fwd(v + (bias ? __ldg(bias + n) : 0.f), act);
  }
}

// dA_L = 2 (recon - x) / C and the batch loss sum((recon - x)^2) / C (one partial per block, fixed order)
__global__ void __launch_bounds__(256) loss_seed_kernel(const float* __restrict__ recon, const float* __restrict__ x,
                                                        const int64_t n, const float inv_c, float* __restrict__ dA,
                                                        float* __restrict__ loss_part) {
  __shared__ float red[256];
  float s = 0.f;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const float d = recon[e] - x[e];
    s += d * d * inv_c;
    if (dA) dA[e] = 2.f * d * inv_c;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss_part[blockIdx.x] = red[0];
}

// dZ = dA * act'(A) in place (A is the post-activation value: its sign is the pre-activation's)
__global__ void __launch_bounds__(256) act_bwd_kernel(float* __restrict__ dA, const float* __restrict__ A_out, const int64_t n,
                                                      const int act) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    if (act == BB_ACT_LEAKY) dA[e] *= A_out[e] > 0.f ? 1.f : BB_LEAKY;
    else if (act == BB_ACT_RELU) dA[e] *= A_out[e] > 0.f ? 1.f : 0.f;
  }
}

// db[n] = sum_m dZ[m][n]: one block per 32 columns, 8 row groups that each add their rows in ascending order, combined
// in group order (reproducible)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ dZ, const int M, const int N, float* __restrict__ db) {
  __shared__ float red[8][33];
  const int c = threadIdx.x & 31, rg = threadIdx.x >> 5, n = blockIdx.x * 32 + c;
  float s = 0.f;
  if (n < N)
    for (int m = rg; m < M; m += 8) s += dZ[(int64_t)m * N + n];
  red[rg][c] = s;
  __syncthreads();
  if (rg == 0 && n < N) {
    float v = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) v += red[q][c];
    db[n] = v;
  }
}

__device__ __forceinline__ float block_sum_256(float v, float* red) {
  __syncthreads();
  red[threadIdx.x] = v;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  return red[0];
}

constexpr float LBN_EPS = 1e-5f, LBN_MOMENTUM = 0.1f;

// BatchNorm over channel c = blockIdx.x of Z[rows][N] (channel c = columns c*S .. c*S + S - 1), then the activation, in
// place.  training: batch statistics (saved for the backward pass in mean_rstd, running statistics updated);
// otherwise the running statistics.  xhat (nullable) receives the normalised values, pre (nullable) the input values.
// `updates`: running-statistics updates from this batch (2 for the encoder under loss_function_swae, which upstream
// encodes a second time with the same batch statistics).
__global__ void __launch_bounds__(256) bn_fwd_kernel(float* __restrict__ Z, float* __restrict__ xhat, const int rows, const int N,
                                                     const int S, const int C, const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, float* __restrict__ running,
                                                     float* __restrict__ mean_rstd, const int training, const int act,
                                                     float* __restrict__ pre, const int updates) {
  __shared__ float red[256];
  const int c = blockIdx.x, M = rows * S;
  float mean, rstd;
  if (training) {
    float s = 0.f;
    for (int e = threadIdx.x; e < M; e += 256) s += Z[(int64_t)(e / S) * N + c * S + e % S];
    mean = block_sum_256(s, red) / M;
    s = 0.f;
    for (int e = threadIdx.x; e < M; e += 256) {
      const float d = Z[(int64_t)(e / S) * N + c * S + e % S] - mean;
      s += d * d;
    }
    const float var = block_sum_256(s, red) / M;
    rstd = 1.f / sqrtf(var + LBN_EPS);
    if (threadIdx.x == 0) {
      for (int u = 0; u < updates; ++u) {
        running[c] = (1.f - LBN_MOMENTUM) * running[c] + LBN_MOMENTUM * mean;
        running[C + c] = (1.f - LBN_MOMENTUM) * running[C + c] + LBN_MOMENTUM * (M > 1 ? var * M / (M - 1) : var);
      }
      mean_rstd[c] = mean;
      mean_rstd[C + c] = rstd;
    }
  } else {
    mean = running[c];
    rstd = 1.f / sqrtf(running[C + c] + LBN_EPS);
  }
  const float g = gamma[c], b = beta[c];
  for (int e = threadIdx.x; e < M; e += 256) {
    const int64_t i = (int64_t)(e / S) * N + c * S + e % S;
    const float z = Z[i], xh = (z - mean) * rstd;
    if (pre) pre[i] = z;
    if (xhat) xhat[i] = xh;
    Z[i] = act_fwd(g * xh + b, act);
  }
}

// dY (already multiplied by act') -> dZ in place; dgamma, dbeta of channel c
__global__ void __launch_bounds__(256) bn_bwd_kernel(float* __restrict__ dY, const float* __restrict__ xhat, const int rows,
                                                     const int N, const int S, const int C, const float* __restrict__ gamma,
                                                     const float* __restrict__ mean_rstd, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta) {
  __shared__ float red[256];
  const int c = blockIdx.x, M = rows * S;
  float s1 = 0.f, s2 = 0.f;
  for (int e = threadIdx.x; e < M; e += 256) {
    const int64_t i = (int64_t)(e / S) * N + c * S + e % S;
    s1 += dY[i];
    s2 += dY[i] * xhat[i];
  }
  s1 = block_sum_256(s1, red);
  s2 = block_sum_256(s2, red);
  if (threadIdx.x == 0) { dgamma[c] = s2; dbeta[c] = s1; }
  const float k = gamma[c] * mean_rstd[C + c], m1 = s1 / M, m2 = s2 / M;
  for (int e = threadIdx.x; e < M; e += 256) {
    const int64_t i = (int64_t)(e / S) * N + c * S + e % S;
    dY[i] = k * (dY[i] - m1 - xhat[i] * m2);
  }
}

// AE_Dropout_BN encoder: Z[rows][N] = act(keep ? Z * scale : 0) in place (dropout before the activation, models.py:263-275)
__device__ __forceinline__ bool ldrop_keep(const unsigned char* mask, const unsigned long long seed, const unsigned long long step,
                                           const int l, const int r, const int j, const int N) {
  return mask ? mask[(int64_t)r * N + j] != 0 : bb_philox_keep(seed, step, l, r, j);
}

__global__ void __launch_bounds__(256) dropout_fwd_kernel(float* __restrict__ Z, const int rows, const int N, const int l,
                                                          const unsigned long long seed, const unsigned long long step,
                                                          const unsigned char* __restrict__ mask, const float scale, const int act) {
  const int64_t total = (int64_t)rows * N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / N), j = (int)(e - (int64_t)r * N);
    Z[e] = act_fwd(ldrop_keep(mask, seed, step, l, r, j, N) ? Z[e] * scale : 0.f, act);
  }
}

// its backward in place: dA (w.r.t. the layer output A) -> dZ = keep ? dA * act'(A) * scale : 0
__global__ void __launch_bounds__(256) dropout_bwd_kernel(float* __restrict__ dA, const float* __restrict__ A_out, const int rows,
                                                          const int N, const int l, const unsigned long long seed,
                                                          const unsigned long long step, const unsigned char* __restrict__ mask,
                                                          const float scale, const int act) {
  const int64_t total = (int64_t)rows * N;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / N), j = (int)(e - (int64_t)r * N);
    float g = dA[e];
    if (act == BB_ACT_LEAKY) g *= A_out[e] > 0.f ? 1.f : BB_LEAKY;
    else if (act == BB_ACT_RELU) g *= A_out[e] > 0.f ? 1.f : 0.f;
    dA[e] = ldrop_keep(mask, seed, step, l, r, j, N) ? g * scale : 0.f;
  }
}

// activation extraction: out[i][j] = mean over `rows` rows of column j of src[i] ([rows][n[i]]), NaN for j >= n[i]; a block
// takes 32 columns of one matrix, 8 row groups add their rows in ascending order in double, combined in group order
struct ColMeanSrc {
  const float* a[6];
  int n[6];
};

__global__ void __launch_bounds__(256) col_means_kernel(const __grid_constant__ ColMeanSrc src, const int rows, const int width,
                                                        double* __restrict__ out) {
  __shared__ double red[8][33];
  const int i = blockIdx.y, c = threadIdx.x & 31, rg = threadIdx.x >> 5, j = blockIdx.x * 32 + c, n = src.n[i];
  double s = 0.0;
  if (j < n)
    for (int r = rg; r < rows; r += 8) s += (double)src.a[i][(int64_t)r * n + j];
  red[rg][c] = s;
  __syncthreads();
  if (rg == 0 && j < width) {
    double v = 0.0;
#pragma unroll
    for (int q = 0; q < 8; ++q) v += red[q][c];
    out[i * width + j] = j < n && rows > 0 ? v / rows : (double)NAN;
  }
}

// dense matrix / bias of a weight-sharing layer from its trainable kernel and per-channel bias
__global__ void __launch_bounds__(256) tied_expand_kernel(const int32_t* __restrict__ map, const float* __restrict__ w,
                                                          float* __restrict__ Wd, const int n_dense, const float* __restrict__ b,
                                                          float* __restrict__ bd, const int N, const int S) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_dense) Wd[i] = map[i] >= 0 ? w[map[i]] : 0.f;
  if (i < N) bd[i] = b[i / S];
}

// gradient of the shared weights: sum of the dense gradient over the entries that use weight j (ascending entry order)
__global__ void __launch_bounds__(256) tied_reduce_kernel(const int32_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                                                          const float* __restrict__ gWd, float* __restrict__ gw, const int n_w,
                                                          const float* __restrict__ gbd, float* __restrict__ gb, const int n_b,
                                                          const int S) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n_w) {
    float s = 0.f;
    for (int e = ptr[j]; e < ptr[j + 1]; ++e) s += gWd[idx[e]];
    gw[j] = s;
  }
  if (j < n_b) {
    float s = 0.f;
    for (int q = 0; q < S; ++q) s += gbd[j * S + q];
    gb[j] = s;
  }
}

// ---- sliced-Wasserstein term of utils.loss_function_swae (utils.py:27-76), one block per projection s:
//   w_i = sort(lat[:, s])_i - sort(pri[:, s])_i;  part[s] = sum_i w_i^2;  d lat[perm_i, s] = 2 w_i * coef
// lat / pri are [rows][S] (projections of the latent batch and of the prior draws); lat is overwritten by its gradient.
constexpr int SWD_MAX_ROWS = 2048;

__device__ void bitonic_sort_smem(float* key, int* idx, const int n) {
  for (int k = 2; k <= n; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int p = i ^ j;
        if (p > i) {
          const bool up = (i & k) == 0;
          const float a = key[i], b = key[p];
          if ((a > b) == up) {
            key[i] = b; key[p] = a;
            if (idx) { const int t = idx[i]; idx[i] = idx[p]; idx[p] = t; }
          }
        }
      }
      __syncthreads();
    }
}

__global__ void __launch_bounds__(256) swd_sort_kernel(float* __restrict__ lat, const float* __restrict__ pri, const int rows,
                                                       const int S, const int n_pow2, const float coef,
                                                       float* __restrict__ part) {
  extern __shared__ float sw[];
  float* lk = sw;                       // n_pow2 latent projections
  float* pk = lk + n_pow2;              // n_pow2 prior projections
  int* li = (int*)(pk + n_pow2);        // row of every latent projection
  __shared__ float red[256];
  const int s = blockIdx.x;
  for (int i = threadIdx.x; i < n_pow2; i += 256) {
    lk[i] = i < rows ? lat[(int64_t)i * S + s] : INFINITY;
    pk[i] = i < rows ? pri[(int64_t)i * S + s] : INFINITY;
    li[i] = i;
  }
  __syncthreads();
  bitonic_sort_smem(lk, li, n_pow2);
  bitonic_sort_smem(pk, nullptr, n_pow2);
  float acc = 0.f;
  for (int i = threadIdx.x; i < rows; i += 256) {
    const float w = lk[i] - pk[i];
    acc += w * w;
    lat[(int64_t)li[i] * S + s] = 2.f * w * coef;
  }
  acc = block_sum_256(acc, red);
  if (threadIdx.x == 0) part[s] = acc;
}

// Batches above SWD_MAX_ROWS: the projections are kept transposed (latT / priT [S][rows], one contiguous segment per
// projection) and one block sorts each segment in global memory with a stable LSD radix sort: SWR_PASSES passes of
// SWR_BITS bits over order-preserving keys, -0 folded onto +0, so that equal values are ties kept in row order as
// np.argsort(kind="stable") keeps them.  Each pass scatters the segment in chunks of 256 keys, in order: a key's slot is
// its digit's running offset + the count of that digit in the chunk's earlier warps + its rank among its warp's equal
// digits.  The loss partial and the scatter of the gradient are those of swd_sort_kernel.
constexpr int SWR_BITS = 8, SWR_BINS = 1 << SWR_BITS, SWR_PASSES = 32 / SWR_BITS, SWR_WARPS = 256 / 32;
static_assert(SWR_BINS == 256, "one digit per thread");

__device__ __forceinline__ uint32_t swr_key(float f) {
  uint32_t b = __float_as_uint(f);
  if ((b << 1) == 0u) b = 0u;  // -0 -> +0
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ float swr_value(const uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct SwrShared {
  int hist[SWR_PASSES][SWR_BINS];
  int wc[2][SWR_WARPS][SWR_BINS];  // per-warp digit counts, then their slots; two chunks in flight
};

// the digit histograms of all passes, from the float segment src[n]
__device__ void swr_histogram(SwrShared& sh, const float* src, const int n) {
  for (int i = threadIdx.x; i < SWR_PASSES * SWR_BINS; i += 256) (&sh.hist[0][0])[i] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += 256) {
    const uint32_t k = swr_key(src[i]);
#pragma unroll
    for (int p = 0; p < SWR_PASSES; ++p) atomicAdd(&sh.hist[p][(k >> (p * SWR_BITS)) & (SWR_BINS - 1)], 1);
  }
  __syncthreads();
}

// one stable pass: keys of src (pass 0: the float segment fsrc, row i's index i) -> kdst / idst (idst nullable)
__device__ void swr_pass(SwrShared& sh, const float* fsrc, const uint32_t* ksrc, const int* isrc, uint32_t* kdst, int* idst,
                         const int n, const int pass) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, shift = pass * SWR_BITS;
  int next = 0;  // thread t: first free slot of digit t
  for (int d = 0; d < tid; ++d) next += sh.hist[pass][d];
  for (int c0 = 0, buf = 0; c0 < n; c0 += 256, buf ^= 1) {
    const int i = c0 + tid;
    uint32_t k = 0;
    int ix = i, d = -1 - lane;  // lanes past the end: a digit of their own
    if (i < n) {
      k = fsrc ? swr_key(fsrc[i]) : ksrc[i];
      if (isrc) ix = isrc[i];
      d = (int)((k >> shift) & (SWR_BINS - 1));
    }
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & ((1u << lane) - 1u));
    if (d >= 0 && rank == 0) sh.wc[buf][warp][d] = __popc(peers);
    __syncthreads();
    int run = next;
#pragma unroll
    for (int w = 0; w < SWR_WARPS; ++w) {
      const int cnt = sh.wc[buf][w][tid];
      sh.wc[buf][w][tid] = run;
      sh.wc[buf ^ 1][w][tid] = 0;  // the other buffer's last readers finished before the barrier above
      run += cnt;
    }
    next = run;
    __syncthreads();
    if (d >= 0) {
      const int pos = sh.wc[buf][warp][d] + rank;
      kdst[pos] = k;
      if (idst) idst[pos] = ix;
    }
  }
  __syncthreads();  // the pass's writes are visible to the next pass's readers of the block ...
#pragma unroll
  for (int w = 0; w < SWR_WARPS; ++w) sh.wc[0][w][tid] = sh.wc[1][w][tid] = 0;  // ... which start from zero counts
  __syncthreads();
}

// block s: sorts priT's segment (its keys end in priT) and latT's with its row indices (ending in kb / ib), then
// part[s] and the gradient d latT[s][perm_i] = 2 w_i coef, written over latT
__global__ void __launch_bounds__(256) swd_radix_kernel(float* __restrict__ latT, float* __restrict__ priT, const int rows,
                                                        uint32_t* __restrict__ ka, uint32_t* __restrict__ kb,
                                                        int* __restrict__ ia, int* __restrict__ ib, const float coef,
                                                        float* __restrict__ part) {
  static_assert(SWR_PASSES == 4, "the ping-pong below ends in kb / ib and priT");
  __shared__ SwrShared sh;
  __shared__ float red[256];
  const size_t off = (size_t)blockIdx.x * rows;
  float *lat = latT + off, *pri = priT + off;
  uint32_t *a = ka + off, *b = kb + off, *pk = reinterpret_cast<uint32_t*>(pri);
  int *xa = ia + off, *xb = ib + off;
  for (int i = threadIdx.x; i < 2 * SWR_WARPS * SWR_BINS; i += 256) (&sh.wc[0][0][0])[i] = 0;  // (every pass leaves it so)
  swr_histogram(sh, pri, rows);
  swr_pass(sh, pri, nullptr, nullptr, a, nullptr, rows, 0);
  swr_pass(sh, nullptr, a, nullptr, b, nullptr, rows, 1);
  swr_pass(sh, nullptr, b, nullptr, a, nullptr, rows, 2);
  swr_pass(sh, nullptr, a, nullptr, pk, nullptr, rows, 3);
  swr_histogram(sh, lat, rows);
  swr_pass(sh, lat, nullptr, nullptr, a, xa, rows, 0);
  swr_pass(sh, nullptr, a, xa, b, xb, rows, 1);
  swr_pass(sh, nullptr, b, xb, a, xa, rows, 2);
  swr_pass(sh, nullptr, a, xa, b, xb, rows, 3);
  float acc = 0.f;
  for (int i = threadIdx.x; i < rows; i += 256) {
    const float w = swr_value(b[i]) - swr_value(pk[i]);
    acc += w * w;
    lat[xb[i]] = 2.f * w * coef;
  }
  acc = block_sum_256(acc, red);
  if (threadIdx.x == 0) part[blockIdx.x] = acc;
}

// loss_part[0] += coef * sum_s part[s] (fixed order);  dst[e] += src[e]
__global__ void __launch_bounds__(256) swd_fold_kernel(const float* __restrict__ part, const int S, const float coef,
                                                       float* __restrict__ loss_part) {
  __shared__ float red[256];
  float acc = 0.f;
  for (int i = threadIdx.x; i < S; i += 256) acc += part[i];
  acc = block_sum_256(acc, red);
  if (threadIdx.x == 0) loss_part[0] += coef * acc;
}

__global__ void __launch_bounds__(256) add_inplace_kernel(float* __restrict__ dst, const float* __restrict__ src, const int64_t n) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) dst[e] += src[e];
}

// mode 0: Adam update + fold the loss partials into grads[n_params] and *loss_accum; 1: only the loss fold (phase 1 of a
// data-parallel step / validation); 2: Adam update with the (all-reduced) grads, loss from grads[n_params]
__global__ void __launch_bounds__(256) ladam_kernel(const int n_params, const int mode, float* __restrict__ grads,
                                                    float* __restrict__ params, float* __restrict__ m, float* __restrict__ v,
                                                    const float lr_bc1, const float inv_sqrt_bc2, const float beta1,
                                                    const float beta2, const float eps, const float* __restrict__ loss_part,
                                                    const int n_loss_parts, double* __restrict__ loss_accum) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n_params && mode != 1) {
    const float g = grads[p];
    const float mn = m[p] + (g - m[p]) * (1.f - beta1);           // exp_avg.lerp_(g, 1 - beta1)
    const float vn = v[p] * beta2 + (1.f - beta2) * g * g;        // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)
    m[p] = mn; v[p] = vn;
    params[p] -= lr_bc1 * mn / (sqrtf(vn) * inv_sqrt_bc2 + eps);  // p.addcdiv_(m, sqrt(v) / sqrt(bc2) + eps, -lr / bc1)
  }
  if (p == 0) {
    float loss;
    if (mode == 2) loss = grads[n_params];
    else {
      loss = 0.f;
      for (int i = 0; i < n_loss_parts; ++i) loss += loss_part[i];
      grads[n_params] = loss;
    }
    if (mode != 1 && loss_accum) *loss_accum += (double)loss;
  }
}

constexpr int LOSS_BLOCKS = 64;

}  // namespace

constexpr int LT_MAX_LAYERS = 16;

struct LLayer {
  int K = 0, N = 0, act = 0;
  int n_w = 0, n_b = 0, bn_c = 0;            // trainable weights / biases, BatchNorm channels (0: none)
  int w_off = 0, b_off = 0, g_off = 0;       // offsets into the trainable vectors (weights, biases, gamma then beta)
  bool tied = false;                         // weight sharing: dense matrix / bias kept apart from the trainable vector
  float *Wd = nullptr, *bd = nullptr, *gWd = nullptr, *gbd = nullptr;  // what the GEMMs read / write (alias when !tied)
  float* dense = nullptr;                    // owns Wd | bd | gWd | gbd when tied
  int32_t *map = nullptr, *csr_ptr = nullptr, *csr_idx = nullptr;
  float *xhat = nullptr, *mean_rstd = nullptr, *running = nullptr;  // BatchNorm: saved xhat, batch (mean, rstd), running (mean | var)
  long long nbt = 0;                         // BatchNorm: num_batches_tracked (training forward passes)
  bool bn_post = false;                      // BatchNorm after the activation (AE_Dropout_BN decoder layers 0-2) ...
  float* pre = nullptr;                      // ... and the activation it normalised, kept for act' in the backward pass
  int drop = -1;                             // dropout before the activation: Philox layer / mask slot (-1: none)
  float drop_scale = 1.f;                    // fp32(1 / (1 - p))
};

struct bb_ltrainer {
  bb_ctx* ctx = nullptr;
  int n_layers = 0, max_batch = 0, n_params = 0, max_dim = 0, loss_columns = 0, n_running = 0;
  LLayer lay[LT_MAX_LAYERS];
  size_t a_off[LT_MAX_LAYERS + 1] = {0};  // float offsets of A_0 .. A_L in `act` (max_batch rows each)
  float *params = nullptr, *grads = nullptr, *m = nullptr, *v = nullptr, *act = nullptr, *dz[2] = {nullptr, nullptr};
  float* running_all = nullptr;           // running statistics of all BatchNorm layers, layer after layer
  // loss_function_swae: projections of the latent batch / of the prior draws [max_batch][S], latent gradient, partials
  float *sw_lat = nullptr, *sw_pri = nullptr, *sw_dz = nullptr, *sw_part = nullptr;
  int sw_S = 0;
  // batches above SWD_MAX_ROWS (max_batch > SWD_MAX_ROWS only): ping-pong keys and row indices of swd_radix_kernel
  uint32_t* sw_key[2] = {nullptr, nullptr};
  int* sw_idx[2] = {nullptr, nullptr};
  float* loss_part = nullptr;
  double* loss_accum = nullptr;
  long long step = 0;
  float* splitk = nullptr;                // split-K partials: SPLIT_MAX x the largest GEMM output
  size_t splitk_floats = 0;
  int last_rows = 0;                      // rows of the most recent forward pass (activation extraction)
  // AE_Dropout_BN (bb_ltrainer_create_dbn): dropout from Philox (seed, step = Adam updates before this one) or injected masks
  bool dbn = false;
  unsigned long long seed = 0;
  const unsigned char* mask_dev[4] = {nullptr, nullptr, nullptr, nullptr};
  HostWindow* win = nullptr;              // device window of bb_ltrainer_epoch_host / _validate_host (kept between calls)
};

namespace {

constexpr int SMALL_TILE_BELOW = 148;  // 64 x 64 grids with fewer CTAs than one per SM use 32 x 32 tiles

constexpr int SPLIT_MAX = 8, SPLIT_MIN_K = 128;  // split-K: at most 8 ways, slices of at least 128

void lgemm(bb_ltrainer* t, cudaStream_t s, const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbk, int64_t sbn, float* C,
           int64_t ldc, int M, int N, int K, const float* bias, int act) {
  dim3 grid((N + TN - 1) / TN, (M + TM - 1) / TM);
  const bool small = (int)(grid.x * grid.y) < SMALL_TILE_BELOW;
  if (small) grid = dim3((N + 31) / 32, (M + 31) / 32);
  // split the contraction when the tiles alone leave SMs idle and the k loop is long
  int S = 1;
  const int ctas = (int)(grid.x * grid.y), target = 2 * t->ctx->sm_count;
  // Only the backward products (TN: weight gradients, NN: input gradients) are split.  The forward products keep the
  // single ascending k order: their results decide ReLU / LeakyReLU signs, and a pre-activation that is zero to fp32
  // rounding may land on either side under a different summation order - measured on the reference's Conv_AE step: one of
  // 38,400 outputs of the 2000 -> 128 Linear flips and moves that layer's bias gradient by 6e-4 (both are valid fp32
  // results; the parity fixtures hold the reference's float64 side of the edge, which the ascending order reproduces).
  static const int split_mask = getenv("BALER_B200_SPLIT_MASK") ? atoi(getenv("BALER_B200_SPLIT_MASK")) : 6;  // (diagnostics)
  const int kind_bit = sam == 1 ? 2 : (sbn == 1 ? 4 : 1);  // TN / NN / NT
  if ((split_mask & kind_bit) && ctas < target && K >= 2 * SPLIT_MIN_K) {
    S = (target + ctas - 1) / ctas;
    if (S > SPLIT_MAX) S = SPLIT_MAX;
    if (S > K / SPLIT_MIN_K) S = K / SPLIT_MIN_K;
    if ((size_t)S * M * ldc > t->splitk_floats) S = 1;
  }
  int k_per = K;
  if (S > 1) {
    k_per = ((K + S - 1) / S + 63) / 64 * 64;  // whole k slabs of either tile shape
    S = (K + k_per - 1) / k_per;
  }
  float* out = S > 1 ? t->splitk : C;
  const int64_t stride = (int64_t)M * ldc;
  grid.z = S;
  if (!small) gemm_strided_kernel<TM, TN, TK><<<grid, GT, 0, s>>>(A, sam, sak, B, sbk, sbn, out, ldc, M, N, K, bias, act, k_per, stride);
  else gemm_strided_kernel<32, 32, 64><<<grid, GT, 0, s>>>(A, sam, sak, B, sbk, sbn, out, ldc, M, N, K, bias, act, k_per, stride);
  if (S > 1) {
    const int64_t total = (int64_t)M * N;
    const int blocks = (int)((total + 255) / 256 < 4 * t->ctx->sm_count ? (total + 255) / 256 : 4 * t->ctx->sm_count);
    splitk_reduce_kernel<<<blocks, 256, 0, s>>>(t->splitk, S, stride, C, ldc, M, N, bias, act);
  }
}

void expand_tied(bb_ltrainer* t, cudaStream_t s) {
  for (int l = 0; l < t->n_layers; ++l) {
    const LLayer& y = t->lay[l];
    if (!y.tied) continue;
    const int n = y.N * y.K;
    tied_expand_kernel<<<(n + 255) / 256, 256, 0, s>>>(y.map, t->params + y.w_off, y.Wd, n, t->params + y.b_off, y.bd, y.N, y.N / y.n_b);
  }
}

// forward (+ loss, + backward into grads when `backward`); BatchNorm layers use batch statistics iff `backward`
struct SwaeArgs {
  const float *prior, *proj;   // [rows][D] prior draws, [S][D] unit projection directions (device)
  int S, latent_layer;         // the latent is the output of layer `latent_layer`
  float reg_weight;
};

int lforward_backward(bb_ltrainer* t, const float* x, int rows, bool backward, cudaStream_t s, const SwaeArgs* sw = nullptr) {
  const int L = t->n_layers;
  const int ew_blocks = t->ctx->sm_count * 2;  // elementwise kernels
  t->last_rows = rows;
  BB_CUDA(cudaMemcpyAsync(t->act + t->a_off[0], x, sizeof(float) * (size_t)rows * t->lay[0].K, cudaMemcpyDeviceToDevice, s));
  for (int l = 0; l < L; ++l) {
    LLayer& y = t->lay[l];
    const bool drop = backward && y.drop >= 0;  // eval mode: dropout is the identity
    float* A = t->act + t->a_off[l + 1];
    // A_{l+1}[rows x N] = act(A_l[rows x K] . W_l[N x K]^T + b_l)
    lgemm(t, s, t->act + t->a_off[l], y.K, 1, y.Wd, 1, y.K, A, y.N, rows, y.N, y.K, y.bd,
          (y.bn_c && !y.bn_post) || drop ? BB_ACT_NONE : y.act);
    if (drop)
      dropout_fwd_kernel<<<ew_blocks, 256, 0, s>>>(A, rows, y.N, y.drop, t->seed, (unsigned long long)t->step, t->mask_dev[y.drop],
                                                   y.drop_scale, y.act);
    if (y.bn_c) {
      // loss_function_swae: upstream's second model.encode(inputs) sees the same batch and weights, so the encoder's
      // BatchNorm layers compute the same statistics again and update their running statistics a second time
      const int updates = sw && l <= sw->latent_layer ? 2 : 1;
      bn_fwd_kernel<<<y.bn_c, 256, 0, s>>>(A, backward ? y.xhat : nullptr, rows, y.N, y.N / y.bn_c, y.bn_c, t->params + y.g_off,
                                           t->params + y.g_off + y.bn_c, y.running, y.mean_rstd, backward ? 1 : 0,
                                           y.bn_post ? BB_ACT_NONE : y.act, backward && y.bn_post ? y.pre : nullptr, updates);
      if (backward) y.nbt += updates;
    }
  }
  const int C = t->lay[L - 1].N;
  float* dA = t->dz[0];
  loss_seed_kernel<<<LOSS_BLOCKS, 256, 0, s>>>(t->act + t->a_off[L], x, (int64_t)rows * C, 1.f / t->loss_columns,
                                                backward ? dA : nullptr, t->loss_part);
  if (sw) {
    // utils.compute_swd (utils.py:56-76): reg_weight / (B (B - 1)) * mean_{s, i} (sort(z P)_{s,i} - sort(prior P)_{s,i})^2
    const int D = t->lay[sw->latent_layer].N, S = sw->S;
    const float* Z = t->act + t->a_off[sw->latent_layer + 1];
    if (rows <= SWD_MAX_ROWS) {
      lgemm(t, s, Z, D, 1, sw->proj, 1, D, t->sw_lat, S, rows, S, D, nullptr, BB_ACT_NONE);
      lgemm(t, s, sw->prior, D, 1, sw->proj, 1, D, t->sw_pri, S, rows, S, D, nullptr, BB_ACT_NONE);
      int n_pow2 = 1;
      while (n_pow2 < rows) n_pow2 <<= 1;
      const float coef = sw->reg_weight / ((float)rows * (float)(rows - 1)) / ((float)S * (float)rows);
      swd_sort_kernel<<<S, 256, sizeof(float) * 3 * n_pow2, s>>>(t->sw_lat, t->sw_pri, rows, S, n_pow2, coef, t->sw_part);
      swd_fold_kernel<<<1, 256, 0, s>>>(t->sw_part, S, coef, t->loss_part);
      // d latent = d(z P) . P^T... as [rows][S] . [S][D]
      if (backward) lgemm(t, s, t->sw_lat, S, 1, sw->proj, D, 1, t->sw_dz, D, rows, D, S, nullptr, BB_ACT_NONE);
    } else {
      // transposed projections [S][rows] (the same products, k ascending), sorted segment by segment in global memory;
      // the weight in float64, rounded once: B (B - 1) is not exact in float32 above 4096 rows
      lgemm(t, s, sw->proj, D, 1, Z, 1, D, t->sw_lat, rows, S, rows, D, nullptr, BB_ACT_NONE);
      lgemm(t, s, sw->proj, D, 1, sw->prior, 1, D, t->sw_pri, rows, S, rows, D, nullptr, BB_ACT_NONE);
      const float coef = (float)((double)sw->reg_weight / ((double)rows * (double)(rows - 1)) / ((double)S * (double)rows));
      swd_radix_kernel<<<S, 256, 0, s>>>(t->sw_lat, t->sw_pri, rows, t->sw_key[0], t->sw_key[1], t->sw_idx[0], t->sw_idx[1], coef,
                                         t->sw_part);
      swd_fold_kernel<<<1, 256, 0, s>>>(t->sw_part, S, coef, t->loss_part);
      // d latent [rows][D] = (d latT)^T . P
      if (backward) lgemm(t, s, t->sw_lat, 1, rows, sw->proj, D, 1, t->sw_dz, D, rows, D, S, nullptr, BB_ACT_NONE);
    }
  }
  if (!backward) return (int)cudaGetLastError();
  int cur = 0;
  for (int l = L - 1; l >= 0; --l) {
    const LLayer& y = t->lay[l];
    const int K = y.K, N = y.N;
    float* dZ = t->dz[cur];
    if (sw && l == sw->latent_layer)  // the encoder sees the decoder's gradient plus the sliced-Wasserstein one
      add_inplace_kernel<<<t->ctx->sm_count, 256, 0, s>>>(dZ, t->sw_dz, (int64_t)rows * N);
    if (y.drop >= 0) {
      dropout_bwd_kernel<<<ew_blocks, 256, 0, s>>>(dZ, t->act + t->a_off[l + 1], rows, N, y.drop, t->seed, (unsigned long long)t->step,
                                                   t->mask_dev[y.drop], y.drop_scale, y.act);
    } else if (y.bn_post) {  // Linear -> act -> BatchNorm: through the BatchNorm first, then act' of its input
      bn_bwd_kernel<<<y.bn_c, 256, 0, s>>>(dZ, y.xhat, rows, N, 1, y.bn_c, t->params + y.g_off, y.mean_rstd, t->grads + y.g_off,
                                           t->grads + y.g_off + y.bn_c);
      act_bwd_kernel<<<ew_blocks, 256, 0, s>>>(dZ, y.pre, (int64_t)rows * N, y.act);
    } else {
      act_bwd_kernel<<<ew_blocks, 256, 0, s>>>(dZ, t->act + t->a_off[l + 1], (int64_t)rows * N, y.act);
      if (y.bn_c)
        bn_bwd_kernel<<<y.bn_c, 256, 0, s>>>(dZ, y.xhat, rows, N, N / y.bn_c, y.bn_c, t->params + y.g_off, y.mean_rstd,
                                             t->grads + y.g_off, t->grads + y.g_off + y.bn_c);
    }
    // dW_l[N x K] = dZ^T[N x rows] . A_l[rows x K]
    lgemm(t, s, dZ, 1, N, t->act + t->a_off[l], K, 1, y.gWd, K, N, K, rows, nullptr, BB_ACT_NONE);
    colsum_kernel<<<(N + 31) / 32, 256, 0, s>>>(dZ, rows, N, y.gbd);
    if (y.tied) {
      const int n = y.n_w > y.n_b ? y.n_w : y.n_b;
      tied_reduce_kernel<<<(n + 255) / 256, 256, 0, s>>>(y.csr_ptr, y.csr_idx, y.gWd, t->grads + y.w_off, y.n_w, y.gbd,
                                                         t->grads + y.b_off, y.n_b, N / y.n_b);
    }
    if (l > 0)  // dA_l[rows x K] = dZ[rows x N] . W_l[N x K]
      lgemm(t, s, dZ, N, 1, y.Wd, K, 1, t->dz[cur ^ 1], K, rows, K, N, nullptr, BB_ACT_NONE);
    cur ^= 1;
  }
  return (int)cudaGetLastError();
}

template <typename T>
int dev_upload(T** dst, const std::vector<T>& src) {
  int rc = (int)cudaMalloc(dst, sizeof(T) * (src.empty() ? 1 : src.size()));
  if (rc == BB_OK && !src.empty()) rc = (int)cudaMemcpy(*dst, src.data(), sizeof(T) * src.size(), cudaMemcpyHostToDevice);
  return rc;
}

}  // namespace

extern "C" {

int bb_ltrainer_create_ex(bb_ctx* ctx, int n_layers, const int* dims, const int* acts, const int* n_shared_w,
                          const int32_t* const* w_maps, const int* n_bias, const int* bn_channels,
                          const double* const* weights_host, const double* const* biases_host, const double* const* bn_host,
                          int loss_columns, int max_batch, bb_ltrainer** out) {
  if (!ctx || !dims || !acts || !weights_host || !biases_host || !out || n_layers < 1 || n_layers > LT_MAX_LAYERS || max_batch < 1)
    return BB_ERR_INVALID;
  if (dims[0] != dims[n_layers]) return BB_ERR_INVALID;  // an autoencoder: the loss compares the output with the input
  BB_CUDA(cudaSetDevice(ctx->device));
  bb_ltrainer* t = new (std::nothrow) bb_ltrainer();
  if (!t) return BB_ERR_NOMEM;
  t->ctx = ctx; t->n_layers = n_layers; t->max_batch = max_batch;
  t->loss_columns = loss_columns > 0 ? loss_columns : dims[n_layers];
  int p = 0;
  size_t a = 0;
  for (int l = 0; l <= n_layers; ++l) {
    if (dims[l] < 1) { delete t; return BB_ERR_INVALID; }
    t->max_dim = dims[l] > t->max_dim ? dims[l] : t->max_dim;
    t->a_off[l] = a;
    a += (size_t)max_batch * dims[l];
  }
  for (int l = 0; l < n_layers; ++l) {
    LLayer& y = t->lay[l];
    y.K = dims[l]; y.N = dims[l + 1]; y.act = acts[l];
    y.tied = n_shared_w && n_shared_w[l] > 0;
    y.n_w = y.tied ? n_shared_w[l] : y.K * y.N;
    y.n_b = y.tied && n_bias && n_bias[l] > 0 ? n_bias[l] : y.N;
    y.bn_c = bn_channels ? bn_channels[l] : 0;
    const bool bad = (y.tied && (!w_maps || !w_maps[l])) || y.N % y.n_b != 0 || (!y.tied && y.n_b != y.N) || y.bn_c < 0 ||
                     (y.bn_c && (y.N % y.bn_c != 0 || !bn_host || !bn_host[l]));
    if (bad) { delete t; return BB_ERR_INVALID; }
    y.w_off = p; p += y.n_w;
    y.b_off = p; p += y.n_b;
    y.g_off = p; p += 2 * y.bn_c;
    t->n_running += 2 * y.bn_c;
  }
  t->n_params = p;
  std::vector<float> hp(p), hrun(t->n_running);
  int roff = 0;
  for (int l = 0; l < n_layers; ++l) {
    const LLayer& y = t->lay[l];
    for (int i = 0; i < y.n_w; ++i) hp[y.w_off + i] = (float)weights_host[l][i];
    for (int n = 0; n < y.n_b; ++n) hp[y.b_off + n] = (float)biases_host[l][n];
    for (int c = 0; c < 2 * y.bn_c; ++c) hp[y.g_off + c] = (float)bn_host[l][c];                     // gamma | beta
    for (int c = 0; c < 2 * y.bn_c; ++c) hrun[roff + c] = (float)bn_host[l][2 * y.bn_c + c];         // running mean | var
    roff += 2 * y.bn_c;
  }
  int rc = (int)cudaMalloc(&t->params, sizeof(float) * p);
  if (rc == BB_OK) rc = (int)cudaMalloc(&t->grads, sizeof(float) * (p + 1));
  if (rc == BB_OK) rc = (int)cudaMalloc(&t->m, sizeof(float) * p);
  if (rc == BB_OK) rc = (int)cudaMalloc(&t->v, sizeof(float) * p);
  if (rc == BB_OK) rc = (int)cudaMalloc(&t->act, sizeof(float) * a);
  for (int i = 0; i < 2 && rc == BB_OK; ++i) rc = (int)cudaMalloc(&t->dz[i], sizeof(float) * (size_t)max_batch * t->max_dim);
  if (rc == BB_OK) rc = (int)cudaMalloc(&t->loss_part, sizeof(float) * LOSS_BLOCKS);
  if (rc == BB_OK) rc = (int)cudaMalloc(&t->loss_accum, sizeof(double));
  {
    size_t big = (size_t)max_batch * (t->max_dim > 2048 ? t->max_dim : 2048);  // (2048: the projections of loss_function_swae)
    for (int l = 0; l < n_layers; ++l)
      if ((size_t)dims[l] * dims[l + 1] > big) big = (size_t)dims[l] * dims[l + 1];
    t->splitk_floats = (size_t)SPLIT_MAX * big;
    if (rc == BB_OK) rc = (int)cudaMalloc(&t->splitk, sizeof(float) * t->splitk_floats);
  }
  if (rc == BB_OK) rc = dev_upload(&t->running_all, hrun);
  if (rc == BB_OK) rc = (int)cudaMemcpy(t->params, hp.data(), sizeof(float) * p, cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemset(t->m, 0, sizeof(float) * p);
  if (rc == BB_OK) rc = (int)cudaMemset(t->v, 0, sizeof(float) * p);
  if (rc == BB_OK) rc = (int)cudaMemset(t->grads, 0, sizeof(float) * (p + 1));
  if (rc == BB_OK) rc = (int)cudaMemset(t->loss_accum, 0, sizeof(double));
  roff = 0;
  for (int l = 0; l < n_layers && rc == BB_OK; ++l) {
    LLayer& y = t->lay[l];
    if (y.bn_c) {
      y.running = t->running_all + roff;
      roff += 2 * y.bn_c;
      rc = (int)cudaMalloc(&y.xhat, sizeof(float) * (size_t)max_batch * y.N);
      if (rc == BB_OK) rc = (int)cudaMalloc(&y.mean_rstd, sizeof(float) * 2 * y.bn_c);
      if (rc != BB_OK) break;
    }
    if (!y.tied) {
      y.Wd = t->params + y.w_off; y.bd = t->params + y.b_off;
      y.gWd = t->grads + y.w_off; y.gbd = t->grads + y.b_off;
      continue;
    }
    const int n = y.N * y.K;
    std::vector<int32_t> map(w_maps[l], w_maps[l] + n), ptr(y.n_w + 1, 0), idx;
    for (int i = 0; i < n; ++i) {
      if (map[i] >= y.n_w) { rc = BB_ERR_INVALID; break; }
      if (map[i] >= 0) ptr[map[i] + 1] += 1;
    }
    if (rc != BB_OK) break;
    for (int j = 0; j < y.n_w; ++j) ptr[j + 1] += ptr[j];
    idx.resize(ptr[y.n_w]);
    std::vector<int32_t> fill(ptr.begin(), ptr.end() - 1);
    for (int i = 0; i < n; ++i)
      if (map[i] >= 0) idx[fill[map[i]]++] = i;
    rc = dev_upload(&y.map, map);
    if (rc == BB_OK) rc = dev_upload(&y.csr_ptr, ptr);
    if (rc == BB_OK) rc = dev_upload(&y.csr_idx, idx);
    if (rc == BB_OK) rc = (int)cudaMalloc(&y.dense, sizeof(float) * 2 * (size_t)(n + y.N));
    if (rc == BB_OK) { y.Wd = y.dense; y.bd = y.Wd + n; y.gWd = y.bd + y.N; y.gbd = y.gWd + n; }
  }
  if (rc == BB_OK) {
    expand_tied(t, nullptr);
    rc = (int)cudaDeviceSynchronize();
  }
  if (rc != BB_OK) { bb_ltrainer_destroy(t); return rc; }
  *out = t;
  return BB_OK;
}

int bb_ltrainer_create(bb_ctx* ctx, int n_layers, const int* dims, const int* acts, const double* const* weights_host,
                       const double* const* biases_host, int max_batch, bb_ltrainer** out) {
  return bb_ltrainer_create_ex(ctx, n_layers, dims, acts, nullptr, nullptr, nullptr, nullptr, weights_host, biases_host, nullptr, 0,
                               max_batch, out);
}

int bb_ltrainer_create_dbn(bb_ctx* ctx, int n_features, int z_dim, const double* const* weights_host,
                           const double* const* biases_host, const double* const* bn_weight_host,
                           const double* const* bn_bias_host, const double* const* bn_mean_host,
                           const double* const* bn_var_host, const long long* bn_batches_tracked, int max_batch,
                           bb_ltrainer** out) {
  if (!bn_weight_host || !bn_bias_host || !bn_mean_host || !bn_var_host || n_features < 1 || z_dim < 1) return BB_ERR_INVALID;
  // models.py:256-313: encoder 4 x (Linear -> Dropout -> LeakyReLU), decoder 3 x (Linear -> LeakyReLU -> BatchNorm1d),
  // then Linear -> BatchNorm1d -> ReLU
  const int dims[9] = {n_features, 200, 100, 50, z_dim, 50, 100, 200, n_features};
  const int acts[8] = {BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_RELU};
  const float drop_scale[4] = {1.f / 0.5f, 1.f / 0.6f, 1.f / 0.7f, 1.f / 0.8f};  // the fused dbn steps' keep_scale
  int bn_c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  std::vector<double> bn[4];
  const double* bn_ptr[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  for (int i = 0; i < 4; ++i) {
    const int n = dims[5 + i];
    if (!bn_weight_host[i] || !bn_bias_host[i] || !bn_mean_host[i] || !bn_var_host[i]) return BB_ERR_INVALID;
    bn[i].resize(4 * (size_t)n);
    for (int j = 0; j < n; ++j) {
      bn[i][j] = bn_weight_host[i][j];
      bn[i][n + j] = bn_bias_host[i][j];
      bn[i][2 * n + j] = bn_mean_host[i][j];
      bn[i][3 * n + j] = bn_var_host[i][j];
    }
    bn_c[4 + i] = n;
    bn_ptr[4 + i] = bn[i].data();
  }
  bb_ltrainer* t = nullptr;
  int rc = bb_ltrainer_create_ex(ctx, 8, dims, acts, nullptr, nullptr, nullptr, bn_c, weights_host, biases_host, bn_ptr, 0,
                                 max_batch, &t);
  if (rc != BB_OK) return rc;
  t->dbn = true;
  for (int l = 0; l < 4; ++l) {
    t->lay[l].drop = l;
    t->lay[l].drop_scale = drop_scale[l];
  }
  for (int i = 0; i < 4 && rc == BB_OK; ++i) {
    LLayer& y = t->lay[4 + i];
    y.nbt = bn_batches_tracked ? bn_batches_tracked[i] : 0;
    y.bn_post = i < 3;
    if (y.bn_post) rc = (int)cudaMalloc(&y.pre, sizeof(float) * (size_t)max_batch * y.N);
  }
  if (rc != BB_OK) { bb_ltrainer_destroy(t); return rc; }
  *out = t;
  return BB_OK;
}

int bb_ltrainer_set_dropout(bb_ltrainer* t, unsigned long long seed, const unsigned char* const* masks_dev) {
  if (!t || !t->dbn) return BB_ERR_INVALID;
  t->seed = seed;
  for (int i = 0; i < 4; ++i) t->mask_dev[i] = masks_dev ? masks_dev[i] : nullptr;
  return BB_OK;
}

int bb_ltrainer_bn_batches_tracked(bb_ltrainer* t, long long* out) {
  if (!t || !out) return BB_ERR_INVALID;
  for (int l = 0; l < t->n_layers; ++l) out[l] = t->lay[l].bn_c ? t->lay[l].nbt : 0;
  return BB_OK;
}

int bb_ltrainer_activation_means(bb_ltrainer* t, double* out_host_6x200) {
  if (!t || !out_host_6x200) return BB_ERR_INVALID;
  // the 8-Linear autoencoders (AE family): A_l = output of layer l - 1 for l = 1, 2, 3, 5, 6, 7, as bb_trainer_activation_means
  const int layers[6] = {1, 2, 3, 5, 6, 7}, width = 200;
  if (t->n_layers != 8) return BB_ERR_UNSUPPORTED;
  ColMeanSrc src;
  for (int i = 0; i < 6; ++i) {
    src.a[i] = t->act + t->a_off[layers[i]];
    src.n[i] = t->lay[layers[i] - 1].N;
    if (src.n[i] > width) return BB_ERR_UNSUPPORTED;
  }
  BB_CUDA(cudaSetDevice(t->ctx->device));
  double* dev = nullptr;
  BB_CUDA(cudaDeviceSynchronize());  // the last forward pass ran on the caller's stream
  BB_CUDA(cudaMalloc(&dev, sizeof(double) * 6 * width));
  col_means_kernel<<<dim3(width / 32 + 1, 6), 256>>>(src, t->last_rows, width, dev);
  int rc = (int)cudaGetLastError();
  if (rc == BB_OK) rc = (int)cudaMemcpy(out_host_6x200, dev, sizeof(double) * 6 * width, cudaMemcpyDeviceToHost);
  cudaFree(dev);
  return rc;
}

int bb_ltrainer_destroy(bb_ltrainer* t) {
  if (!t) return BB_OK;
  void* ptrs[] = {t->params, t->grads, t->m, t->v, t->act, t->dz[0], t->dz[1], t->loss_part, t->loss_accum, t->running_all,
                  t->sw_lat, t->sw_pri, t->sw_dz, t->sw_part, t->sw_key[0], t->sw_key[1], t->sw_idx[0], t->sw_idx[1], t->splitk};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  for (int l = 0; l < t->n_layers; ++l) {
    LLayer& y = t->lay[l];
    void* lp[] = {y.dense, y.map, y.csr_ptr, y.csr_idx, y.xhat, y.mean_rstd, y.pre};
    for (void* p : lp)
      if (p) cudaFree(p);
  }
  bb_host_window_free(t->win);
  delete t;
  return BB_OK;
}

int bb_ltrainer_param_count(const bb_ltrainer* t) { return t ? t->n_params : 0; }
float* bb_ltrainer_params_dev(bb_ltrainer* t) { return t ? t->params : nullptr; }
float* bb_ltrainer_grads_dev(bb_ltrainer* t) { return t ? t->grads : nullptr; }
float* bb_ltrainer_bn_running_dev(bb_ltrainer* t, int* n_floats) {
  if (n_floats) *n_floats = t ? t->n_running : 0;
  return t ? t->running_all : nullptr;
}

int bb_ltrainer_get_params(bb_ltrainer* t, double* const* weights_host, double* const* biases_host) {
  if (!t || !weights_host || !biases_host) return BB_ERR_INVALID;
  std::vector<float> hp(t->n_params);
  BB_CUDA(cudaMemcpy(hp.data(), t->params, sizeof(float) * hp.size(), cudaMemcpyDeviceToHost));
  for (int l = 0; l < t->n_layers; ++l) {
    const LLayer& y = t->lay[l];
    for (int i = 0; i < y.n_w; ++i) weights_host[l][i] = (double)hp[y.w_off + i];
    for (int n = 0; n < y.n_b; ++n) biases_host[l][n] = (double)hp[y.b_off + n];
  }
  return BB_OK;
}

int bb_ltrainer_get_bn(bb_ltrainer* t, double* const* bn_host) {
  if (!t || !bn_host) return BB_ERR_INVALID;
  std::vector<float> hp(t->n_params), hr(t->n_running);
  BB_CUDA(cudaMemcpy(hp.data(), t->params, sizeof(float) * hp.size(), cudaMemcpyDeviceToHost));
  if (t->n_running) BB_CUDA(cudaMemcpy(hr.data(), t->running_all, sizeof(float) * hr.size(), cudaMemcpyDeviceToHost));
  int roff = 0;
  for (int l = 0; l < t->n_layers; ++l) {
    const LLayer& y = t->lay[l];
    if (!y.bn_c) continue;
    if (!bn_host[l]) return BB_ERR_INVALID;
    for (int c = 0; c < 2 * y.bn_c; ++c) bn_host[l][c] = (double)hp[y.g_off + c];
    for (int c = 0; c < 2 * y.bn_c; ++c) bn_host[l][2 * y.bn_c + c] = (double)hr[roff + c];
    roff += 2 * y.bn_c;
  }
  return BB_OK;
}

static int lstep(bb_ltrainer* t, const float* x_dev, int batch_rows, const bb_train_hyper* h, int phase, double* loss_accum_dev,
                 bb_stream_t stream, const SwaeArgs* sw) {
  if (!t || !h || !x_dev || batch_rows < 1 || batch_rows > t->max_batch || phase < 0 || phase > 2) return BB_ERR_INVALID;
  if (h->l1) return BB_ERR_UNSUPPORTED;  // the reference never trains the L1 term (training.py:83-89); fused kernels have the opt-in
  cudaStream_t s = (cudaStream_t)stream;
  if (phase != 2) {
    const int rc = lforward_backward(t, x_dev, batch_rows, true, s, sw);
    if (rc != BB_OK) return rc;
  }
  float lr_bc1 = 0.f, inv_sqrt_bc2 = 0.f;
  if (phase != 1) {
    t->step += 1;
    lr_bc1 = (float)(h->lr / (1.0 - std::pow(h->beta1, (double)t->step)));
    inv_sqrt_bc2 = (float)(1.0 / std::sqrt(1.0 - std::pow(h->beta2, (double)t->step)));
  }
  ladam_kernel<<<(t->n_params + 255) / 256, 256, 0, s>>>(t->n_params, phase, t->grads, t->params, t->m, t->v, lr_bc1, inv_sqrt_bc2,
                                                        (float)h->beta1, (float)h->beta2, (float)h->eps, t->loss_part, LOSS_BLOCKS,
                                                        loss_accum_dev);
  if (phase != 1) expand_tied(t, s);
  return (int)cudaGetLastError();
}

int bb_ltrainer_step(bb_ltrainer* t, const float* x_dev, int batch_rows, const bb_train_hyper* h, int phase,
                     double* loss_accum_dev, bb_stream_t stream) {
  return lstep(t, x_dev, batch_rows, h, phase, loss_accum_dev, stream, nullptr);
}

int bb_ltrainer_step_swae(bb_ltrainer* t, const float* x_dev, int batch_rows, const bb_train_hyper* h, int phase,
                          const float* prior_dev, const float* proj_dev, int n_projections, int latent_layer, float reg_weight,
                          double* loss_accum_dev, bb_stream_t stream) {
  if (!t || !prior_dev || !proj_dev || n_projections < 1 || latent_layer < 0 || latent_layer >= t->n_layers - 1)
    return BB_ERR_INVALID;
  if (batch_rows < 2) return BB_ERR_UNSUPPORTED;  // B (B - 1) in the weight
  for (int l = 0; l < t->n_layers; ++l)
    if (t->lay[l].drop >= 0) return BB_ERR_UNSUPPORTED;  // upstream's second encode would draw other dropout masks
  if (t->sw_S != n_projections) {
    BB_CUDA(cudaSetDevice(t->ctx->device));
    BB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    void* old[] = {t->sw_lat, t->sw_pri, t->sw_dz, t->sw_part, t->sw_key[0], t->sw_key[1], t->sw_idx[0], t->sw_idx[1]};
    for (void* p : old)
      if (p) cudaFree(p);
    t->sw_lat = t->sw_pri = t->sw_dz = t->sw_part = nullptr;
    t->sw_key[0] = t->sw_key[1] = nullptr;
    t->sw_idx[0] = t->sw_idx[1] = nullptr;
    t->sw_S = 0;
    const size_t n = (size_t)t->max_batch * n_projections;
    BB_CUDA(cudaMalloc(&t->sw_lat, sizeof(float) * n));
    BB_CUDA(cudaMalloc(&t->sw_pri, sizeof(float) * n));
    BB_CUDA(cudaMalloc(&t->sw_dz, sizeof(float) * (size_t)t->max_batch * t->max_dim));
    BB_CUDA(cudaMalloc(&t->sw_part, sizeof(float) * n_projections));
    for (int i = 0; i < 2 && t->max_batch > SWD_MAX_ROWS; ++i) {
      BB_CUDA(cudaMalloc(&t->sw_key[i], sizeof(uint32_t) * n));
      BB_CUDA(cudaMalloc(&t->sw_idx[i], sizeof(int) * n));
    }
    t->sw_S = n_projections;
  }
  SwaeArgs sw{prior_dev, proj_dev, n_projections, latent_layer, reg_weight};
  return lstep(t, x_dev, batch_rows, h, phase, loss_accum_dev, stream, &sw);
}

}  // extern "C"

namespace {
// the training steps of the batches of rows [0, n_rows) of x in order, their losses added to t->loss_accum: the body of an
// epoch over a device table and of every window of a streamed host table (windows hold whole batches)
int ltrain_rows(bb_ltrainer* t, const float* x, int64_t n_rows, int batch, const bb_train_hyper* h, cudaStream_t s) {
  for (int64_t r0 = 0; r0 < n_rows; r0 += batch) {
    const int rows = (int)(n_rows - r0 < batch ? n_rows - r0 : batch);
    const int rc = bb_ltrainer_step(t, x + (size_t)r0 * t->lay[0].K, rows, h, 0, t->loss_accum, s);
    if (rc != BB_OK) return rc;
  }
  return BB_OK;
}

// the eval-mode forward passes of the same batches, their losses added to t->loss_accum
int leval_rows(bb_ltrainer* t, const float* x, int64_t n_rows, int batch, cudaStream_t s) {
  for (int64_t r0 = 0; r0 < n_rows; r0 += batch) {
    const int rows = (int)(n_rows - r0 < batch ? n_rows - r0 : batch);
    int rc = lforward_backward(t, x + (size_t)r0 * t->lay[0].K, rows, false, s);
    if (rc != BB_OK) return rc;
    // mode 1 folds the loss partials into grads[n_params]; mode 2 with zero parameters adds that slot to the accumulator
    ladam_kernel<<<1, 256, 0, s>>>(t->n_params, 1, t->grads, nullptr, nullptr, nullptr, 0.f, 0.f, 0.f, 0.f, 0.f, t->loss_part,
                                   LOSS_BLOCKS, nullptr);
    ladam_kernel<<<1, 256, 0, s>>>(0, 2, t->grads + t->n_params, nullptr, nullptr, nullptr, 0.f, 0.f, 0.f, 0.f, 0.f, nullptr, 0,
                                   t->loss_accum);
    BB_CUDA(cudaGetLastError());
  }
  return BB_OK;
}

// epoch loss = the summed batch losses over the number of batches (training.py:99); synchronises s
int lfinish(bb_ltrainer* t, int64_t n_rows, int batch, double* epoch_loss_host, cudaStream_t s) {
  double total = 0.0;
  BB_CUDA(cudaMemcpyAsync(&total, t->loss_accum, sizeof(double), cudaMemcpyDeviceToHost, s));
  BB_CUDA(cudaStreamSynchronize(s));
  *epoch_loss_host = total / (double)((n_rows + batch - 1) / batch);
  return BB_OK;
}

// a host table this trainer streams: float32 rows, a window of whole batches
bool lhost_ok(bb_ltrainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch, int64_t window_rows,
              const double* epoch_loss_host) {
  return t && x_host && x_dtype == BB_F32 && n_rows >= 1 && batch >= 1 && batch <= t->max_batch && window_rows >= batch &&
         window_rows % batch == 0 && epoch_loss_host;
}
}  // namespace

extern "C" {

int bb_ltrainer_epoch(bb_ltrainer* t, const float* x_dev, int64_t n_rows, int batch, const bb_train_hyper* h,
                      double* epoch_loss_host, bb_stream_t stream) {
  if (!t || !h || !x_dev || n_rows < 1 || batch < 1 || batch > t->max_batch || !epoch_loss_host) return BB_ERR_INVALID;
  if (h->world_size > 1) return BB_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  const int rc = ltrain_rows(t, x_dev, n_rows, batch, h, s);
  return rc != BB_OK ? rc : lfinish(t, n_rows, batch, epoch_loss_host, s);
}

int bb_ltrainer_validate(bb_ltrainer* t, const float* x_dev, int64_t n_rows, int batch, double* epoch_loss_host,
                         bb_stream_t stream) {
  if (!t || !x_dev || n_rows < 1 || batch < 1 || batch > t->max_batch || !epoch_loss_host) return BB_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  const int rc = leval_rows(t, x_dev, n_rows, batch, s);
  return rc != BB_OK ? rc : lfinish(t, n_rows, batch, epoch_loss_host, s);
}

int bb_ltrainer_epoch_host(bb_ltrainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch,
                           const bb_train_hyper* h, int64_t window_rows, double* epoch_loss_host, bb_stream_t stream) {
  if (!h || !lhost_ok(t, x_host, x_dtype, n_rows, batch, window_rows, epoch_loss_host)) return BB_ERR_INVALID;
  if (h->world_size > 1) return BB_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  BB_CUDA(cudaSetDevice(t->ctx->device));
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  const size_t row_bytes = (size_t)t->lay[0].K * sizeof(float);
  const int rc = bb_host_window_run(&t->win, x_host, row_bytes, n_rows, window_rows, s, [&](const void* x, int64_t rows) {
    return ltrain_rows(t, (const float*)x, rows, batch, h, s);
  });
  return rc != BB_OK ? rc : lfinish(t, n_rows, batch, epoch_loss_host, s);
}

int bb_ltrainer_validate_host(bb_ltrainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch,
                              int64_t window_rows, double* epoch_loss_host, bb_stream_t stream) {
  if (!lhost_ok(t, x_host, x_dtype, n_rows, batch, window_rows, epoch_loss_host)) return BB_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  BB_CUDA(cudaSetDevice(t->ctx->device));
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  const size_t row_bytes = (size_t)t->lay[0].K * sizeof(float);
  const int rc = bb_host_window_run(&t->win, x_host, row_bytes, n_rows, window_rows, s, [&](const void* x, int64_t rows) {
    return leval_rows(t, (const float*)x, rows, batch, s);
  });
  return rc != BB_OK ? rc : lfinish(t, n_rows, batch, epoch_loss_host, s);
}

}  // extern "C"
