// Layer-by-layer dense chain for shapes whose weights do not fit the fused kernels' shared memory
// (Conv_AE as its dense-equivalent chain with the 128 -> 2000 -> z Linears, models.py:316-407; CFD_dense_AE on
// 2500-feature snapshots, models.py:186-226).  Each layer is one fp32 GEMM launch
//     Y[n x N] = act(X[n x K] . W[N x K]^T + b)        (W row-major (out, in), exactly as nn.Linear stores it)
// with activations ping-ponging through global scratch in row chunks.  Both operands are K-major, tiles of
// 128 x 64 x 16 are staged through shared memory (transposed on the way in so the inner product loop reads
// 128-bit vectors), 8 x 4 outputs per thread, register prefetch of the next K slab.  All leading dimensions are
// padded to multiples of 4 floats (zero weights / zero bias in the padding) so every global access is a 16-byte
// vector.  Normalisation, dtype conversion and un-normalisation run as thin elementwise kernels around the GEMMs.
//
// BB_PREC_SPLIT16 (the default when the shape is not served by the fused kernels): the same GEMM on the tensor cores,
// dense_layer_tc_kernel - warp-level MMA (mma.sync m16n8k16, SASS HMMA) with the fp16 hi / lo 3-product split of the
// fused kernels (x = hi + lo / 2048; hi*hi + (hi*lo + lo*hi) / 2048, fp32 accumulate).  96 % of Conv_AE's FLOPs are its
// 128 -> 2000 -> z Linears (models.py:320-321,343).  Why mma.sync and not tcgen05 here: the weight images (6 MB for
// Conv_AE) stream through shared memory tile by tile like in any GEMM, the activations arrive as fp32 from the previous
// layer and are split on the way into shared memory; this is the layer-at-a-time fallback path, one kernel serves every
// layer shape, inference and (bb_train_layered.cu) training alike.
#include <cstdlib>

#include "bb_common.cuh"

namespace {

constexpr int BM = 128, BN = 64, BK = 16, LT = 256;

__device__ __forceinline__ float act_l(float v, int act) {
  if (act == BB_ACT_LEAKY) return v > 0.f ? v : BB_LEAKY * v;
  if (act == BB_ACT_RELU) return fmaxf(v, 0.f);
  return v;
}

__global__ void __launch_bounds__(LT)
dense_layer_kernel(const float* __restrict__ X, const int ldx, const float* __restrict__ W, const int ldw,
                   const float* __restrict__ bias, float* __restrict__ Y, const int ldy, const int n, const int K,
                   const int Np, const int act) {
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Bs[2][BK][BN + 4];
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  // loader mapping: one float4 (4 consecutive k) per thread and slab; A needs two rows per thread
  const int lr = tid >> 2, lk = (tid & 3) << 2;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  auto load = [&](int k0, float4& a0, float4& a1, float4& b0) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    const bool kv = k0 + lk < K;  // K is padded to a multiple of 4, so a float4 is all-in or all-out
    a0 = (kv && m0 + lr < n) ? __ldg(reinterpret_cast<const float4*>(X + (size_t)(m0 + lr) * ldx + k0 + lk)) : z;
    a1 = (kv && m0 + lr + 64 < n) ? __ldg(reinterpret_cast<const float4*>(X + (size_t)(m0 + lr + 64) * ldx + k0 + lk)) : z;
    b0 = (kv && n0 + lr < Np) ? __ldg(reinterpret_cast<const float4*>(W + (size_t)(n0 + lr) * ldw + k0 + lk)) : z;
  };
  auto stash = [&](int buf, const float4& a0, const float4& a1, const float4& b0) {
    As[buf][lk + 0][lr] = a0.x; As[buf][lk + 1][lr] = a0.y; As[buf][lk + 2][lr] = a0.z; As[buf][lk + 3][lr] = a0.w;
    As[buf][lk + 0][lr + 64] = a1.x; As[buf][lk + 1][lr + 64] = a1.y; As[buf][lk + 2][lr + 64] = a1.z; As[buf][lk + 3][lr + 64] = a1.w;
    Bs[buf][lk + 0][lr] = b0.x; Bs[buf][lk + 1][lr] = b0.y; Bs[buf][lk + 2][lr] = b0.z; Bs[buf][lk + 3][lr] = b0.w;
  };
  float4 a0, a1, b0;
  load(0, a0, a1, b0);
  stash(0, a0, a1, b0);
  __syncthreads();
  int buf = 0;
  for (int k0 = 0; k0 < K; k0 += BK) {
    const bool more = k0 + BK < K;
    if (more) load(k0 + BK, a0, a1, b0);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 x0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8]);
      const float4 x1 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8 + 4]);
      const float4 w0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
      const float wv[4] = {w0.x, w0.y, w0.z, w0.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xv[i], wv[j], acc[i][j]);
    }
    if (more) {
      stash(buf ^ 1, a0, a1, b0);
      __syncthreads();
      buf ^= 1;
    }
  }
  const int c = n0 + tx * 4;
  if (c < Np) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(bias + c));
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = m0 + ty * 8 + i;
      if (r < n) {
        float4 o;
        o.x = act_l(acc[i][0] + b.x, act); o.y = act_l(acc[i][1] + b.y, act);
        o.z = act_l(acc[i][2] + b.z, act); o.w = act_l(acc[i][3] + b.w, act);
        *reinterpret_cast<float4*>(Y + (size_t)r * ldy + c) = o;
      }
    }
  }
}


// ------------------------------------------------------------------------------------------------ tensor-core GEMM
constexpr int TBM = 128, TBN = 64, TBK = 32, TLD = 40, TNT = 256;  // TLD: row stride in halves (80 B: ldmatrix rows hit distinct banks)
constexpr float T_LO = 2048.f, T_LO_INV = 1.f / 2048.f;
constexpr int T_SMEM = 2 * 2 * (TBM + TBN) * TLD * 2;  // [2 stages][hi | lo][A 128 rows + B 64 rows][40 halves]

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], const uint32_t a) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a) : "memory");
}
__device__ __forceinline__ void hmma(float (&d)[4], const uint32_t (&a)[4], const uint32_t b0, const uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(const uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
// 4 floats -> packed fp16 hi (2 words) and packed scaled lo (2 words)
__device__ __forceinline__ void split4(const float4 v, uint2& hi, uint2& lo) {
  const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
  const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
  const __half2 l0 = __floats2half2_rn((v.x - f0.x) * T_LO, (v.y - f0.y) * T_LO);
  const __half2 l1 = __floats2half2_rn((v.z - f1.x) * T_LO, (v.w - f1.y) * T_LO);
  hi = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
  lo = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
}

// Y[n x Np4] = act(X[n x K] . W[N x K]^T + b).  X fp32 rows of pitch ldx (valid and zero padded up to kx columns), W as
// two fp16 images [rows padded to 64][Kp] (hi, and lo scaled by 2048; zero padding), 128 x 64 tiles, 8 warps of 32 x 32.
__global__ void __launch_bounds__(TNT, 2)
dense_layer_tc_kernel(const float* __restrict__ X, const int ldx, const int kx, const __half* __restrict__ Whi,
                      const __half* __restrict__ Wlo, const int Kp, const float* __restrict__ bias, float* __restrict__ Y,
                      const int ldy, const int n, const int Np4, const int act, int* __restrict__ flag) {
  extern __shared__ __align__(16) unsigned char tsm[];
  // stage s: [A hi | A lo | B hi | B lo]
  constexpr int A_B = TBM * TLD * 2, B_B = TBN * TLD * 2, STAGE = 2 * A_B + 2 * B_B;
  const uint32_t sb = smem_addr(tsm);
  const int m0 = blockIdx.y * TBM, n0 = blockIdx.x * TBN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = (warp & 3) * 32, wn = (warp >> 2) * 32;
  // loaders: A 4 x float4 per thread (rows lr + 32 i, 4 consecutive k), B one 16-byte chunk per image
  const int lr = tid >> 3, lc = (tid & 7) * 4;
  const int br = tid >> 2, bc = (tid & 3) * 8;
  float hh[2][4][4], cr[2][4][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) hh[i][j][q] = cr[i][j][q] = 0.f;
  float4 av[4];
  auto load_a = [&](const int k0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = m0 + lr + 32 * i;
      av[i] = (r < n && k0 + lc < kx) ? __ldg(reinterpret_cast<const float4*>(X + (size_t)r * ldx + k0 + lc))
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stash_a = [&](const int st) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint2 hi, lo;
      split4(av[i], hi, lo);
      const uint32_t off = (uint32_t)(st * STAGE + ((lr + 32 * i) * TLD + lc) * 2);
      asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(sb + off), "r"(hi.x), "r"(hi.y) : "memory");
      asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(sb + off + A_B), "r"(lo.x), "r"(lo.y) : "memory");
    }
  };
  auto load_b = [&](const int st, const int k0) {
    const size_t src = (size_t)(n0 + br) * Kp + k0 + bc;
    const uint32_t dst = sb + st * STAGE + 2 * A_B + (br * TLD + bc) * 2;
    cp_async16(dst, Whi + src);
    cp_async16(dst + B_B, Wlo + src);
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  load_a(0);
  load_b(0, 0);
  stash_a(0);
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  // ldmatrix lane addresses inside a stage
  const uint32_t a_lane = (uint32_t)(((wm + (lane & 7) + ((lane >> 3) & 1) * 8) * TLD + (lane >> 4) * 8) * 2);
  const uint32_t b_lane = (uint32_t)(2 * A_B + ((wn + (lane & 7) + ((lane >> 4) & 1) * 8) * TLD + ((lane >> 3) & 1) * 8) * 2);
  int st = 0;
  for (int k0 = 0; k0 < Kp; k0 += TBK) {
    const bool more = k0 + TBK < Kp;
    if (more) {
      load_a(k0 + TBK);
      load_b(st ^ 1, k0 + TBK);
    }
    const uint32_t base = sb + st * STAGE;
#pragma unroll
    for (int ks = 0; ks < TBK / 16; ++ks) {
      uint32_t ah[2][4], al[2][4], bh[2][4], bl[2][4];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        ldsm4(ah[i], base + a_lane + (i * 16 * TLD + ks * 16) * 2);
        ldsm4(al[i], base + a_lane + A_B + (i * 16 * TLD + ks * 16) * 2);
      }
#pragma unroll
      for (int p = 0; p < 2; ++p) {
        ldsm4(bh[p], base + b_lane + (p * 16 * TLD + ks * 16) * 2);
        ldsm4(bl[p], base + b_lane + B_B + (p * 16 * TLD + ks * 16) * 2);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) hmma(hh[i][j], ah[i], bh[j >> 1][(j & 1) * 2], bh[j >> 1][(j & 1) * 2 + 1]);
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) hmma(cr[i][j], ah[i], bl[j >> 1][(j & 1) * 2], bl[j >> 1][(j & 1) * 2 + 1]);
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) hmma(cr[i][j], al[i], bh[j >> 1][(j & 1) * 2], bh[j >> 1][(j & 1) * 2 + 1]);
    }
    if (more) {
      stash_a(st ^ 1);
      asm volatile("cp.async.wait_all;" ::: "memory");
      __syncthreads();
      st ^= 1;
    }
  }
  const int g = lane >> 2, t = lane & 3;
  bool bad = false;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = n0 + wn + j * 8 + 2 * t;
    if (c < Np4) {
      const float2 b = __ldg(reinterpret_cast<const float2*>(bias + c));
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int r = m0 + wm + i * 16 + g + 8 * h;
          if (r < n) {
            float2 o;
            o.x = act_l(fmaf(cr[i][j][2 * h], T_LO_INV, hh[i][j][2 * h]) + b.x, act);
            o.y = act_l(fmaf(cr[i][j][2 * h + 1], T_LO_INV, hh[i][j][2 * h + 1]) + b.y, act);
            bad = bad || !(fabsf(o.x) <= 3.0e38f) || !(fabsf(o.y) <= 3.0e38f);
            *reinterpret_cast<float2*>(Y + (size_t)r * ldy + c) = o;
          }
        }
    }
  }
  if (bad && flag != nullptr) *flag = 1;  // a value left the fp16 range on the way (inf / NaN): BB_PREC_AUTO callers re-run in fp32
}

// in (f32 | f16, compact rows of `dim`) -> scratch rows of pitch `ld` (zero padded), optionally (x - min) / range
__global__ void __launch_bounds__(256) stage_in_kernel(const void* __restrict__ in, const int in_dtype, const int64_t n,
                                                       const int dim, const int ld, const float* __restrict__ mn,
                                                       const float* __restrict__ rg, float* __restrict__ out) {
  const uint32_t total = (uint32_t)(n * ld), G = gridDim.x * blockDim.x;  // (< 2^31 per chunk, as in stage_out_kernel)
  for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += G) {
    const int64_t r = e / (uint32_t)ld;
    const int c = (int)(e - (uint32_t)r * (uint32_t)ld);
    float v = 0.f;
    if (c < dim) {
      v = in_dtype == BB_F16 ? __half2float(reinterpret_cast<const __half*>(in)[r * dim + c]) : reinterpret_cast<const float*>(in)[r * dim + c];
      if (mn != nullptr) v = __fdiv_rn(__fsub_rn(v, __ldg(mn + c)), __ldg(rg + c));
    }
    out[e] = v;
  }
}

// scratch rows of pitch `ld` -> compact rows of `dim` (f32 | f16), optionally y * range + min
__global__ void __launch_bounds__(256) stage_out_kernel(const float* __restrict__ in, const int64_t n, const int dim,
                                                        const int ld, const float* __restrict__ mn,
                                                        const float* __restrict__ rg, void* __restrict__ out,
                                                        const int out_dtype) {
  // (chunks hold < 2^31 values - checked by the launcher: 32-bit index arithmetic, a 64-bit division per element costs
  // more than the copy)
  const uint32_t total = (uint32_t)(n * dim), G = gridDim.x * blockDim.x;
  // four independent elements per trip: the loads are all issued before the first store
  for (uint32_t e0 = blockIdx.x * blockDim.x + threadIdx.x; e0 < total; e0 += 4 * G) {
    float v[4];
    int c[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t e = e0 + u * G;
      const uint32_t r = e / (uint32_t)dim;
      c[u] = (int)(e - r * (uint32_t)dim);
      v[u] = e < total ? in[(size_t)r * ld + c[u]] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t e = e0 + u * G;
      if (e >= total) break;
      float y = v[u];
      if (mn != nullptr) y = fmaf(y, __ldg(rg + c[u]), __ldg(mn + c[u]));
      if (out_dtype == BB_F16) reinterpret_cast<__half*>(out)[e] = __float2half_rn(y);
      else reinterpret_cast<float*>(out)[e] = y;
    }
  }
}

inline int pad4(int x) { return (x + 3) & ~3; }
constexpr int64_t CHUNK_ROWS = 1 << 15;

}  // namespace

// uploads W (pitch padded to 4, extra zero rows up to a multiple of 4) and bias per layer
int bb_chain_layered_prepare(bb_ctx*, Chain* c) {
  const ChainDesc& d = c->desc;
  size_t total = 0;
  int max_ld = pad4(d.in_dim);
  for (int l = 0; l < d.n_layers; ++l) {
    total += (size_t)pad4(d.layer[l].N) * pad4(d.layer[l].K) + pad4(d.layer[l].N);
    max_ld = pad4(d.layer[l].N) > max_ld ? pad4(d.layer[l].N) : max_ld;
  }
  std::vector<float> blob(total, 0.f);
  size_t off = 0;
  for (int l = 0; l < d.n_layers; ++l) {
    const int K = d.layer[l].K, N = d.layer[l].N, Kp = pad4(K), Np = pad4(N);
    c->lay_w_off[l] = off;
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < K; ++k) blob[off + (size_t)n * Kp + k] = (float)c->w_host[l][(size_t)n * K + k];
    off += (size_t)Np * Kp;
    c->lay_b_off[l] = off;
    for (int n = 0; n < N; ++n) blob[off + n] = (float)c->b_host[l][n];
    off += Np;
  }
  if (c->lay_blob_dev) cudaFree(c->lay_blob_dev);
  BB_CUDA(cudaMalloc(&c->lay_blob_dev, blob.size() * sizeof(float)));
  BB_CUDA(cudaMemcpy(c->lay_blob_dev, blob.data(), blob.size() * sizeof(float), cudaMemcpyHostToDevice));
  c->lay_max_ld = max_ld;
  c->lay_ok = true;
  // tensor-core images: per layer W as fp16 hi and lo * 2048, rows padded to the 64-column tile, K to the 32-wide slab
  size_t halves = 0;
  for (int l = 0; l < d.n_layers; ++l) {
    c->lay_tc_off[l] = halves;
    halves += 2 * (size_t)((d.layer[l].N + TBN - 1) / TBN * TBN) * ((d.layer[l].K + TBK - 1) / TBK * TBK);
  }
  std::vector<__half> img(halves, __float2half(0.f));
  for (int l = 0; l < d.n_layers; ++l) {
    const int K = d.layer[l].K, N = d.layer[l].N, Kp = (K + TBK - 1) / TBK * TBK, Nr = (N + TBN - 1) / TBN * TBN;
    __half* hi = img.data() + c->lay_tc_off[l];
    __half* lo = hi + (size_t)Nr * Kp;
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < K; ++k) {
        const double w = c->w_host[l][(size_t)n * K + k];
        const __half h = __float2half_rn((float)w);
        hi[(size_t)n * Kp + k] = h;
        lo[(size_t)n * Kp + k] = __float2half_rn((float)((w - (double)__half2float(h)) * (double)T_LO));
      }
  }
  if (c->lay_tc_blob_dev) cudaFree(c->lay_tc_blob_dev);
  c->lay_tc_blob_dev = nullptr;
  BB_CUDA(cudaMalloc(&c->lay_tc_blob_dev, img.size() * sizeof(__half)));
  BB_CUDA(cudaMemcpy(c->lay_tc_blob_dev, img.data(), img.size() * sizeof(__half), cudaMemcpyHostToDevice));
  BB_CUDA(cudaFuncSetAttribute(dense_layer_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T_SMEM));
  c->lay_tc_ok = true;
  // the tcgen05 form of the same GEMMs (optional per shape)
  const int g5 = bb_gemm_tc5_prepare(nullptr, c);
  if (g5 != BB_OK && g5 != BB_ERR_UNSUPPORTED) return g5;
  return BB_OK;
}

int bb_chain_layered_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows,
                            const float* pre_min, const float* pre_range, const float* post_min,
                            const float* post_range, void* out, int out_dtype, int tensor_cores, int* flag_dev,
                            cudaStream_t stream) {
  if (!c->lay_ok || (tensor_cores && !c->lay_tc_ok)) return BB_ERR_UNSUPPORTED;
  if (n_rows == 0) return BB_OK;
  const ChainDesc& d = c->desc;
  // tensor cores: the tcgen05 GEMM (bb_gemm_tc5.cu) when the shape has it, else the mma.sync one below
  const bool tc5 = tensor_cores && c->g5_ok && !getenv("BALER_B200_LAYERED_MMA");
  // (tcgen05: persistent CTAs walk 128-row tiles; a whole number of tiles per SM leaves no partial wave on the
  // one-column-tile layers, and 8 per SM amortise the fill / drain of the ~7 launches per chunk: Conv_AE encode / decode
  // 148 / 153 M blocks/s with 2 tiles per SM, 157 / 165 with 4, 163 / 172 with 8 - 2 x 1.24 GB of scratch for 2000-wide layers)
  int64_t chunk_rows = CHUNK_ROWS;
  if (tc5) {
    int tiles = 8;  // ... halved while one ping-pong buffer would pass 2 GiB (wider models)
    while (tiles > 1 && bb_gemm_tc5_buf_bytes(c, (int64_t)tiles * ctx->sm_count * 128) > ((size_t)2 << 30)) tiles /= 2;
    chunk_rows = (int64_t)tiles * ctx->sm_count * 128;
  }
  if (const char* e = getenv("BALER_B200_LAYER_CHUNK")) chunk_rows = atoll(e) > 0 ? atoll(e) : chunk_rows;  // (tuning)
  const int64_t chunk = n_rows < chunk_rows ? n_rows : chunk_rows;
  if (chunk * (int64_t)(c->lay_max_ld > d.out_dim ? c->lay_max_ld : d.out_dim) >= (1ll << 31)) return BB_ERR_INVALID;  // staging: 32-bit indices
  const size_t buf_bytes = tc5 ? bb_gemm_tc5_buf_bytes(c, chunk) : (size_t)chunk * c->lay_max_ld * sizeof(float);
  const size_t need = 2 * buf_bytes;
  if (c->lay_scratch_bytes < need) {
    // grown only (never shrunk); stream-ordered work that still uses the old buffer has been enqueued before the free
    if (c->lay_scratch) BB_CUDA(cudaFree(c->lay_scratch));
    c->lay_scratch = nullptr;
    BB_CUDA(cudaMalloc(&c->lay_scratch, need));
    c->lay_scratch_bytes = need;
  }
  c->last_route = tc5 ? BB_ROUTE_LAYERED_TC5 : tensor_cores ? BB_ROUTE_LAYERED_MMA : BB_ROUTE_LAYERED_F32;
  c->last_tile_rows = (int)chunk;
  if (tc5) {
    const size_t in_esz5 = in_dtype == BB_F16 ? 2 : 4, out_esz5 = out_dtype == BB_F16 ? 2 : 4;
    char* b0 = reinterpret_cast<char*>(c->lay_scratch);
    for (int64_t r0 = 0; r0 < n_rows; r0 += chunk) {
      const int64_t rows = n_rows - r0 < chunk ? n_rows - r0 : chunk;
      int ob = 0, ldo = 0;
      const int rc = bb_gemm_tc5_chunk(ctx, c, (const char*)in + (size_t)r0 * d.in_dim * in_esz5, in_dtype, rows, pre_min, pre_range, b0,
                                       b0 + buf_bytes, flag_dev, &ob, &ldo, stream);
      if (rc != BB_OK) return rc;
      stage_out_kernel<<<ctx->sm_count * 8, 256, 0, stream>>>(reinterpret_cast<const float*>(b0 + (size_t)ob * buf_bytes), rows, d.out_dim, ldo,
                                                             post_min, post_range, (char*)out + (size_t)r0 * d.out_dim * out_esz5, out_dtype);
    }
    return (int)cudaGetLastError();
  }
  float* buf[2] = {c->lay_scratch, c->lay_scratch + (size_t)chunk * c->lay_max_ld};
  const size_t in_esz = in_dtype == BB_F16 ? 2 : 4, out_esz = out_dtype == BB_F16 ? 2 : 4;
  const int ew_grid = ctx->sm_count * 8;
  for (int64_t r0 = 0; r0 < n_rows; r0 += chunk) {
    const int64_t rows = n_rows - r0 < chunk ? n_rows - r0 : chunk;
    int ld = pad4(d.in_dim);
    stage_in_kernel<<<ew_grid, 256, 0, stream>>>((const char*)in + (size_t)r0 * d.in_dim * in_esz, in_dtype, rows, d.in_dim, ld,
                                                 pre_min, pre_range, buf[0]);
    int cur = 0;
    for (int l = 0; l < d.n_layers; ++l) {
      const int K = d.layer[l].K, N = d.layer[l].N, Kp = pad4(K), Np = pad4(N);
      if (tensor_cores) {
        const int Kt = (K + TBK - 1) / TBK * TBK, Nr = (N + TBN - 1) / TBN * TBN;
        const __half* whi = reinterpret_cast<const __half*>(c->lay_tc_blob_dev) + c->lay_tc_off[l];
        const dim3 grid((Np + TBN - 1) / TBN, (unsigned)((rows + TBM - 1) / TBM));
        dense_layer_tc_kernel<<<grid, TNT, T_SMEM, stream>>>(buf[cur], ld, ld, whi, whi + (size_t)Nr * Kt, Kt,
                                                            c->lay_blob_dev + c->lay_b_off[l], buf[cur ^ 1], Np, (int)rows, Np,
                                                            d.layer[l].act, flag_dev);
      } else {
        const dim3 grid((Np + BN - 1) / BN, (unsigned)((rows + BM - 1) / BM));
        dense_layer_kernel<<<grid, LT, 0, stream>>>(buf[cur], ld, c->lay_blob_dev + c->lay_w_off[l], Kp,
                                                   c->lay_blob_dev + c->lay_b_off[l], buf[cur ^ 1], Np, (int)rows, Kp, Np,
                                                   d.layer[l].act);
      }
      cur ^= 1;
      ld = Np;
    }
    stage_out_kernel<<<ew_grid, 256, 0, stream>>>(buf[cur], rows, d.out_dim, ld, post_min, post_range,
                                                  (char*)out + (size_t)r0 * d.out_dim * out_esz, out_dtype);
  }
  return (int)cudaGetLastError();
}
