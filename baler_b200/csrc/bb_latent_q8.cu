// 8-bit latent (latent_dtype "q8"): uint8 codes with a float32 affine pair (lo, step) per latent column and 128-row block.
//
// Format (baler_b200/latent_q8.py is the one definition; tests/latent_q8_ref.py its numpy mirror):
//   lo[b, j], hi[b, j]  min / max over the finite values of block b, column j (0 when there is none)
//   step[b, j]          float32((float64(hi) - float64(lo)) / 254)
//   code                255 for a non-finite value (decodes to NaN); 0 when step == 0;
//                       else clamp(rint((float64(v) - lo) * (1.0 / float64(step))), 0, 254)
//   value               float32(float64(lo) + float64(code) * float64(step))
// Every float64 operation is one IEEE operation in round-to-nearest (the __d*_rn intrinsics are never contracted into an
// FMA), so the codes are bit-equal to numpy's.  min / max compare order-preserving integer keys (-0 < +0, as
// colminmax_kernel), which fixes lo's sign bit whatever order the values are seen in.
#include <algorithm>
#include <climits>

#include "bb_common.cuh"

namespace {

constexpr int Q8_ROWS = 128;          // rows per block (BB_Q8_BLOCK_ROWS)
constexpr int Q8_THREADS = 256;       // 8 warps: warp w takes rows w, w + 8, ..., lane l column c0 + l of a 32-column tile
constexpr int Q8_WARPS = Q8_THREADS / 32;
constexpr int Q8_ROWS_PER_WARP = Q8_ROWS / Q8_WARPS;

__device__ __forceinline__ int32_t q8_key(uint32_t u) { return (int32_t)(u ^ ((uint32_t)((int32_t)u >> 31) & 0x7fffffffu)); }
__device__ __forceinline__ float q8_unkey(int32_t k) {
  return __uint_as_float(k >= 0 ? (uint32_t)k : ((uint32_t)k ^ 0x7fffffffu));
}
__device__ __forceinline__ bool q8_finite(uint32_t u) { return (u & 0x7fffffffu) < 0x7f800000u; }

// One CTA per group of blocks (grid-stride over the 128-row blocks).  Per 32-column tile: each warp folds the keys of its
// 16 rows per column, the 8 partials meet in shared memory and warp 0 folds them in warp order; the values stay in registers
// for the quantisation pass.  No atomics: the result does not depend on scheduling.
__global__ void __launch_bounds__(Q8_THREADS, 4) latent_q8_quantize_kernel(const float* __restrict__ z, int64_t n_rows, int Z,
                                                                        uint8_t* __restrict__ codes, float* __restrict__ lo_out,
                                                                        float* __restrict__ step_out) {
  __shared__ int32_t s_mn[Q8_WARPS][32], s_mx[Q8_WARPS][32];
  __shared__ double s_lo[32], s_inv[32];
  __shared__ float s_step[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n_blocks = (n_rows + Q8_ROWS - 1) / Q8_ROWS;
  for (int64_t b = blockIdx.x; b < n_blocks; b += gridDim.x) {
    const int64_t r0 = b * Q8_ROWS;
    const int rows = (int)min(n_rows - r0, (int64_t)Q8_ROWS);
    for (int c0 = 0; c0 < Z; c0 += 32) {
      const int j = c0 + lane;
      const bool col = j < Z;
      uint32_t u[Q8_ROWS_PER_WARP];
      int32_t mn = INT_MAX, mx = INT_MIN;
#pragma unroll
      for (int i = 0; i < Q8_ROWS_PER_WARP; ++i) {
        const int r = warp + Q8_WARPS * i;
        u[i] = 0x7fc00000u;  // rows past the end behave as NaN: they never reach the min / max
        if (col && r < rows) u[i] = __float_as_uint(__ldg(z + (r0 + r) * Z + j));
        if (q8_finite(u[i])) {
          const int32_t k = q8_key(u[i]);
          mn = min(mn, k);
          mx = max(mx, k);
        }
      }
      s_mn[warp][lane] = mn;
      s_mx[warp][lane] = mx;
      __syncthreads();
      if (warp == 0) {
        for (int w = 1; w < Q8_WARPS; ++w) {
          mn = min(mn, s_mn[w][lane]);
          mx = max(mx, s_mx[w][lane]);
        }
        const bool any = mn <= mx;
        const float lo = any ? q8_unkey(mn) : 0.0f, hi = any ? q8_unkey(mx) : 0.0f;
        const float step = __double2float_rn(__ddiv_rn(__dsub_rn((double)hi, (double)lo), 254.0));
        if (col) {
          lo_out[b * Z + j] = lo;
          step_out[b * Z + j] = step;
        }
        s_lo[lane] = (double)lo;
        s_step[lane] = step;
        s_inv[lane] = step != 0.0f ? __ddiv_rn(1.0, (double)step) : 0.0;
      }
      __syncthreads();
      const double lo = s_lo[lane], inv = s_inv[lane];
      const bool flat = s_step[lane] == 0.0f;
#pragma unroll
      for (int i = 0; i < Q8_ROWS_PER_WARP; ++i) {
        const int r = warp + Q8_WARPS * i;
        if (!col || r >= rows) continue;
        uint32_t q = 255u;
        if (q8_finite(u[i])) {
          q = 0u;
          if (!flat) {
            const double t = rint(__dmul_rn(__dsub_rn((double)__uint_as_float(u[i]), lo), inv));
            q = (uint32_t)fmin(fmax(t, 0.0), 254.0);
          }
        }
        codes[(r0 + r) * Z + j] = (uint8_t)q;
      }
      __syncthreads();  // shared memory of this tile is read before the next tile writes it
    }
  }
}

// codes + (lo, step) -> float32 latent, one element per thread and step; index arithmetic inside a block is 32-bit
__global__ void __launch_bounds__(Q8_THREADS) latent_q8_dequantize_kernel(const uint8_t* __restrict__ codes,
                                                                          const float* __restrict__ lo,
                                                                          const float* __restrict__ step, int64_t n_rows,
                                                                          int Z, float* __restrict__ z) {
  const int64_t n_blocks = (n_rows + Q8_ROWS - 1) / Q8_ROWS;
  for (int64_t b = blockIdx.x; b < n_blocks; b += gridDim.x) {
    const int64_t e0 = b * Q8_ROWS * Z;
    const unsigned n = (unsigned)(min(n_rows - b * Q8_ROWS, (int64_t)Q8_ROWS) * Z);
    const float* blo = lo + b * Z;
    const float* bst = step + b * Z;
    for (unsigned e = threadIdx.x; e < n; e += Q8_THREADS) {
      const unsigned j = e % (unsigned)Z;
      const uint32_t c = codes[e0 + e];
      z[e0 + e] = c == 255u ? __uint_as_float(0x7fc00000u)
                            : __double2float_rn(__dadd_rn((double)__ldg(blo + j), __dmul_rn((double)c, (double)__ldg(bst + j))));
    }
  }
}

int q8_grid(const bb_ctx* ctx, int64_t n_rows) {
  const int64_t n_blocks = (n_rows + Q8_ROWS - 1) / Q8_ROWS;
  return (int)std::min<int64_t>(n_blocks, (int64_t)ctx->sm_count * (2048 / Q8_THREADS));
}

}  // namespace

int bb_latent_q8_quantize_launch(bb_ctx* ctx, const float* z, int64_t n_rows, int Z, uint8_t* codes, float* lo, float* step,
                                 cudaStream_t stream) {
  if (n_rows == 0) return BB_OK;
  latent_q8_quantize_kernel<<<q8_grid(ctx, n_rows), Q8_THREADS, 0, stream>>>(z, n_rows, Z, codes, lo, step);
  return (int)cudaGetLastError();
}

int bb_latent_q8_dequantize_launch(bb_ctx* ctx, const uint8_t* codes, const float* lo, const float* step, int64_t n_rows,
                                   int Z, float* z, cudaStream_t stream) {
  if (n_rows == 0) return BB_OK;
  latent_q8_dequantize_kernel<<<q8_grid(ctx, n_rows), Q8_THREADS, 0, stream>>>(codes, lo, step, n_rows, Z, z);
  return (int)cudaGetLastError();
}

extern "C" {

int bb_latent_quantize_q8(bb_ctx* ctx, const float* z_dev, int64_t n_rows, int z_dim, uint8_t* codes_dev, float* lo_dev,
                          float* step_dev, bb_stream_t stream) {
  if (!ctx || n_rows < 0 || z_dim < 1 || (n_rows && (!z_dev || !codes_dev || !lo_dev || !step_dev))) return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(ctx->device));
  return bb_latent_q8_quantize_launch(ctx, z_dev, n_rows, z_dim, codes_dev, lo_dev, step_dev, (cudaStream_t)stream);
}

int bb_latent_dequantize_q8(bb_ctx* ctx, const uint8_t* codes_dev, const float* lo_dev, const float* step_dev,
                            int64_t n_rows, int z_dim, float* z_dev, bb_stream_t stream) {
  if (!ctx || n_rows < 0 || z_dim < 1 || (n_rows && (!z_dev || !codes_dev || !lo_dev || !step_dev))) return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(ctx->device));
  return bb_latent_q8_dequantize_launch(ctx, codes_dev, lo_dev, step_dev, n_rows, z_dim, z_dev, (cudaStream_t)stream);
}

}  // extern "C"
