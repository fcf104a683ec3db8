// Quantised latent (latent_dtype "q2" ... "q8"): b-bit codes, packed row by row, with a float32 affine pair (lo, step) per
// latent column and 128-row block.
//
// Format (baler_b200/latent_q8.py is the one definition; tests/latent_packed_ref.py its numpy mirror), L = 2^b - 2:
//   lo[k, j], hi[k, j]  min / max over the finite values of block k, column j (0 when there is none)
//   step[k, j]          float32((float64(hi) - float64(lo)) / L)
//   code                2^b - 1 for a non-finite value (decodes to NaN); 0 when step == 0;
//                       else clamp(rint((float64(v) - lo) * (1.0 / float64(step))), 0, L)
//   value               float32(float64(lo) + float64(code) * float64(step))
//   packing             row r is row_bytes = ceil(z * b / 8) bytes; column j's code is bits [j b, j b + b) of the row, bit
//                       k being bit k % 8 of byte k / 8; unused high bits of the last byte are 0.  b = 8: one byte per code
// Every float64 operation is one IEEE operation in round-to-nearest (the __d*_rn intrinsics are never contracted into an
// FMA), so the codes are bit-equal to numpy's.  min / max compare order-preserving integer keys (-0 < +0, as
// colminmax_kernel), which fixes lo's sign bit whatever order the values are seen in.
#include <algorithm>
#include <climits>

#include "bb_common.cuh"

namespace {

constexpr int Q_ROWS = 128;          // rows per block (BB_Q8_BLOCK_ROWS)
constexpr int Q_THREADS = 256;       // 8 warps: warp w takes rows w, w + 8, ..., lane l column c0 + l of a 32-column tile
constexpr int Q_WARPS = Q_THREADS / 32;
constexpr int Q_ROWS_PER_WARP = Q_ROWS / Q_WARPS;

__device__ __forceinline__ int32_t q_key(uint32_t u) { return (int32_t)(u ^ ((uint32_t)((int32_t)u >> 31) & 0x7fffffffu)); }
__device__ __forceinline__ float q_unkey(int32_t k) {
  return __uint_as_float(k >= 0 ? (uint32_t)k : ((uint32_t)k ^ 0x7fffffffu));
}
__device__ __forceinline__ bool q_finite(uint32_t u) { return (u & 0x7fffffffu) < 0x7f800000u; }

int row_bytes_of(int Z, int bits) { return (Z * bits + 7) / 8; }

// Dynamic shared memory of the quantise kernel: the block's packed rows (128 * row_bytes bytes, a multiple of 16) and, for
// b < 8, its unpacked codes behind them (128 * Z bytes).  For b = 8 the two are the same bytes.
size_t quantize_smem(int Z, int bits) {
  return (size_t)Q_ROWS * row_bytes_of(Z, bits) + (bits < 8 ? (size_t)Q_ROWS * Z : 0);
}

// One CTA per group of blocks (grid-stride over the 128-row blocks).  Per 32-column tile: each warp folds the keys of its
// 16 rows per column, the 8 partials meet in shared memory and warp 0 folds them in warp order; the values stay in registers
// for the quantisation pass, whose codes go to shared memory.  No atomics: the result does not depend on scheduling.  Then
// each row's codes are packed (b < 8) and the block's rows leave as one contiguous segment, 16 bytes per store.
template <int BITS>
__global__ void __launch_bounds__(Q_THREADS, 4) latent_quantize_kernel(const float* __restrict__ z, int64_t n_rows, int Z,
                                                                     uint8_t* __restrict__ codes, float* __restrict__ lo_out,
                                                                     float* __restrict__ step_out) {
  constexpr uint32_t NAN_CODE = (1u << BITS) - 1u;
  constexpr double LEVELS = (double)((1 << BITS) - 2);
  extern __shared__ __align__(16) uint8_t s_dyn[];
  __shared__ int32_t s_mn[Q_WARPS][32], s_mx[Q_WARPS][32];
  __shared__ double s_lo[32], s_inv[32];
  __shared__ float s_step[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // s_dyn: the packed rows [128][row_bytes], then (b < 8) the codes [128][Z].  Offsets are computed where they are used:
  // kept live across the tile loop they cost the registers the 16 staged values need (the b = 8 kernel then spills)
  const int64_t n_blocks = (n_rows + Q_ROWS - 1) / Q_ROWS;
  for (int64_t b = blockIdx.x; b < n_blocks; b += gridDim.x) {
    const int64_t r0 = b * Q_ROWS;
    const int rows = (int)min(n_rows - r0, (int64_t)Q_ROWS);
    for (int c0 = 0; c0 < Z; c0 += 32) {
      const int j = c0 + lane;
      const bool col = j < Z;
      uint32_t u[Q_ROWS_PER_WARP];
      int32_t mn = INT_MAX, mx = INT_MIN;
#pragma unroll
      for (int i = 0; i < Q_ROWS_PER_WARP; ++i) {
        const int r = warp + Q_WARPS * i;
        u[i] = 0x7fc00000u;  // rows past the end behave as NaN: they never reach the min / max
        if (col && r < rows) u[i] = __float_as_uint(__ldg(z + (r0 + r) * Z + j));
        if (q_finite(u[i])) {
          const int32_t k = q_key(u[i]);
          mn = min(mn, k);
          mx = max(mx, k);
        }
      }
      s_mn[warp][lane] = mn;
      s_mx[warp][lane] = mx;
      __syncthreads();
      if (warp == 0) {
        for (int w = 1; w < Q_WARPS; ++w) {
          mn = min(mn, s_mn[w][lane]);
          mx = max(mx, s_mx[w][lane]);
        }
        const bool any = mn <= mx;
        const float lo = any ? q_unkey(mn) : 0.0f, hi = any ? q_unkey(mx) : 0.0f;
        const float step = __double2float_rn(__ddiv_rn(__dsub_rn((double)hi, (double)lo), LEVELS));
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
      for (int i = 0; i < Q_ROWS_PER_WARP; ++i) {
        const int r = warp + Q_WARPS * i;
        if (!col || r >= rows) continue;
        const int sidx = r * Z + j;
        uint32_t q = NAN_CODE;
        if (q_finite(u[i])) {
          q = 0u;
          if (!flat) {
            const double t = rint(__dmul_rn(__dsub_rn((double)__uint_as_float(u[i]), lo), inv));
            q = (uint32_t)fmin(fmax(t, 0.0), LEVELS);
          }
        }
        s_dyn[BITS == 8 ? sidx : Q_ROWS * ((Z * BITS + 7) / 8) + sidx] = (uint8_t)q;
      }
      __syncthreads();  // shared memory of this tile is read before the next tile writes it
    }
    const int row_bytes = (Z * BITS + 7) / 8;
    const uint8_t* s_pack = s_dyn;
    if (BITS < 8) {  // pack: one thread per row, low bits first
      uint8_t* s_codes = s_dyn + Q_ROWS * row_bytes;
      for (int r = threadIdx.x; r < rows; r += Q_THREADS) {
        const uint8_t* src = s_codes + r * Z;
        uint8_t* dst = s_dyn + r * row_bytes;
        uint32_t acc = 0;
        int have = 0;
        for (int c = 0; c < Z; ++c) {
          acc |= (uint32_t)src[c] << have;
          have += BITS;
          if (have >= 8) {
            *dst++ = (uint8_t)acc;
            acc >>= 8;
            have -= 8;
          }
        }
        if (have > 0) *dst = (uint8_t)acc;
      }
      __syncthreads();
    }
    // the block's rows are bytes [r0 * row_bytes, (r0 + rows) * row_bytes) of `codes`; a whole block is a multiple of 16
    const int bytes = rows * row_bytes;
    uint8_t* out = codes + r0 * row_bytes;
    const int n16 = ((uintptr_t)out & 15u) == 0 ? bytes / 16 : 0;
    for (int i = threadIdx.x; i < n16; i += Q_THREADS)
      reinterpret_cast<uint4*>(out)[i] = reinterpret_cast<const uint4*>(s_pack)[i];
    for (int i = n16 * 16 + threadIdx.x; i < bytes; i += Q_THREADS) out[i] = s_pack[i];
    __syncthreads();  // the staged rows are stored before the next block overwrites them
  }
}

// codes + (lo, step) -> float32 latent, one element per thread and step; index arithmetic inside a block is 32-bit
template <int BITS>
__global__ void __launch_bounds__(Q_THREADS) latent_dequantize_kernel(const uint8_t* __restrict__ codes,
                                                                      const float* __restrict__ lo,
                                                                      const float* __restrict__ step, int64_t n_rows,
                                                                      int Z, float* __restrict__ z) {
  constexpr uint32_t NAN_CODE = (1u << BITS) - 1u;
  const unsigned row_bytes = (unsigned)(Z * BITS + 7) / 8;
  const int64_t n_blocks = (n_rows + Q_ROWS - 1) / Q_ROWS;
  for (int64_t b = blockIdx.x; b < n_blocks; b += gridDim.x) {
    const int64_t e0 = b * Q_ROWS * Z;
    const unsigned n = (unsigned)(min(n_rows - b * Q_ROWS, (int64_t)Q_ROWS) * Z);
    const uint8_t* bc = codes + b * Q_ROWS * row_bytes;
    const float* blo = lo + b * Z;
    const float* bst = step + b * Z;
    for (unsigned e = threadIdx.x; e < n; e += Q_THREADS) {
      const unsigned j = e % (unsigned)Z;
      uint32_t c;
      if (BITS == 8) {
        c = bc[e];
      } else {  // a code spans at most two bytes, both inside its row
        const unsigned pos = j * BITS;
        const uint8_t* p = bc + (e / (unsigned)Z) * row_bytes + (pos >> 3);
        uint32_t v = __ldg(p);
        if ((pos & 7u) + BITS > 8u) v |= (uint32_t)__ldg(p + 1) << 8;
        c = (v >> (pos & 7u)) & NAN_CODE;
      }
      z[e0 + e] = c == NAN_CODE ? __uint_as_float(0x7fc00000u)
                                : __double2float_rn(__dadd_rn((double)__ldg(blo + j), __dmul_rn((double)c, (double)__ldg(bst + j))));
    }
  }
}

int q_grid(const bb_ctx* ctx, int64_t n_rows) {
  const int64_t n_blocks = (n_rows + Q_ROWS - 1) / Q_ROWS;
  return (int)std::min<int64_t>(n_blocks, (int64_t)ctx->sm_count * (2048 / Q_THREADS));
}

template <int BITS>
int quantize_launch(bb_ctx* ctx, const float* z, int64_t n_rows, int Z, uint8_t* codes, float* lo, float* step,
                    cudaStream_t stream) {
  const size_t smem = quantize_smem(Z, BITS);
  if (smem > 40 * 1024) {  // (with the static shared memory, beyond the 48 KB a launch gets without opting in)
    cudaFuncAttributes fa{};
    BB_CUDA(cudaFuncGetAttributes(&fa, latent_quantize_kernel<BITS>));
    if (smem + fa.sharedSizeBytes > ctx->smem_optin) return BB_ERR_UNSUPPORTED;
    BB_CUDA(cudaFuncSetAttribute(latent_quantize_kernel<BITS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  latent_quantize_kernel<BITS><<<q_grid(ctx, n_rows), Q_THREADS, smem, stream>>>(z, n_rows, Z, codes, lo, step);
  return (int)cudaGetLastError();
}

template <int BITS>
int dequantize_launch(bb_ctx* ctx, const uint8_t* codes, const float* lo, const float* step, int64_t n_rows, int Z, float* z,
                      cudaStream_t stream) {
  latent_dequantize_kernel<BITS><<<q_grid(ctx, n_rows), Q_THREADS, 0, stream>>>(codes, lo, step, n_rows, Z, z);
  return (int)cudaGetLastError();
}

}  // namespace

int bb_latent_quantize_launch(bb_ctx* ctx, const float* z, int64_t n_rows, int Z, int bits, uint8_t* codes, float* lo,
                              float* step, cudaStream_t stream) {
  if (n_rows == 0) return BB_OK;
  switch (bits) {
    case 2: return quantize_launch<2>(ctx, z, n_rows, Z, codes, lo, step, stream);
    case 3: return quantize_launch<3>(ctx, z, n_rows, Z, codes, lo, step, stream);
    case 4: return quantize_launch<4>(ctx, z, n_rows, Z, codes, lo, step, stream);
    case 5: return quantize_launch<5>(ctx, z, n_rows, Z, codes, lo, step, stream);
    case 6: return quantize_launch<6>(ctx, z, n_rows, Z, codes, lo, step, stream);
    case 7: return quantize_launch<7>(ctx, z, n_rows, Z, codes, lo, step, stream);
    case 8: return quantize_launch<8>(ctx, z, n_rows, Z, codes, lo, step, stream);
    default: return BB_ERR_INVALID;
  }
}

int bb_latent_dequantize_launch(bb_ctx* ctx, int bits, const uint8_t* codes, const float* lo, const float* step,
                                int64_t n_rows, int Z, float* z, cudaStream_t stream) {
  if (n_rows == 0) return BB_OK;
  switch (bits) {
    case 2: return dequantize_launch<2>(ctx, codes, lo, step, n_rows, Z, z, stream);
    case 3: return dequantize_launch<3>(ctx, codes, lo, step, n_rows, Z, z, stream);
    case 4: return dequantize_launch<4>(ctx, codes, lo, step, n_rows, Z, z, stream);
    case 5: return dequantize_launch<5>(ctx, codes, lo, step, n_rows, Z, z, stream);
    case 6: return dequantize_launch<6>(ctx, codes, lo, step, n_rows, Z, z, stream);
    case 7: return dequantize_launch<7>(ctx, codes, lo, step, n_rows, Z, z, stream);
    case 8: return dequantize_launch<8>(ctx, codes, lo, step, n_rows, Z, z, stream);
    default: return BB_ERR_INVALID;
  }
}

extern "C" {

int bb_latent_quantize_packed(bb_ctx* ctx, const float* z_dev, int64_t n_rows, int z_dim, int bits, uint8_t* codes_dev,
                              float* lo_dev, float* step_dev, bb_stream_t stream) {
  if (!ctx || n_rows < 0 || z_dim < 1 || bits < BB_LATENT_MIN_BITS || bits > BB_LATENT_MAX_BITS ||
      (n_rows && (!z_dev || !codes_dev || !lo_dev || !step_dev)))
    return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(ctx->device));
  return bb_latent_quantize_launch(ctx, z_dev, n_rows, z_dim, bits, codes_dev, lo_dev, step_dev, (cudaStream_t)stream);
}

int bb_latent_dequantize_packed(bb_ctx* ctx, int bits, const uint8_t* codes_dev, const float* lo_dev, const float* step_dev,
                                int64_t n_rows, int z_dim, float* z_dev, bb_stream_t stream) {
  if (!ctx || n_rows < 0 || z_dim < 1 || bits < BB_LATENT_MIN_BITS || bits > BB_LATENT_MAX_BITS ||
      (n_rows && (!z_dev || !codes_dev || !lo_dev || !step_dev)))
    return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(ctx->device));
  return bb_latent_dequantize_launch(ctx, bits, codes_dev, lo_dev, step_dev, n_rows, z_dim, z_dev, (cudaStream_t)stream);
}

int bb_latent_quantize_q8(bb_ctx* ctx, const float* z_dev, int64_t n_rows, int z_dim, uint8_t* codes_dev, float* lo_dev,
                          float* step_dev, bb_stream_t stream) {
  return bb_latent_quantize_packed(ctx, z_dev, n_rows, z_dim, 8, codes_dev, lo_dev, step_dev, stream);
}

int bb_latent_dequantize_q8(bb_ctx* ctx, const uint8_t* codes_dev, const float* lo_dev, const float* step_dev,
                            int64_t n_rows, int z_dim, float* z_dev, bb_stream_t stream) {
  return bb_latent_dequantize_packed(ctx, 8, codes_dev, lo_dev, step_dev, n_rows, z_dim, z_dev, stream);
}

}  // extern "C"
