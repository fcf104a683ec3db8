// Fused 4-layer dense chain on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// Same contract as bb_chain_f32.cu ([normalise ->] 4 dense layers [-> un-normalise], one HBM read and one
// HBM write per row) but the matrix products run as tcgen05.mma kind::f16 with fp32 accumulation in TMEM.
//
// Precision.  The reference computes in float64 and the parity bar is 1e-5 (max-norm and l2, per tensor).
// A single fp16 product misses that by ~30x, so every operand is split x = hi + lo with hi = fp16(x) and
// lo = fp16(x - hi) (22 significant bits) and each product is three MMAs accumulated into the same
// TMEM accumulator: hi*hi + hi*lo + lo*hi (lo*lo ~ 2^-22 is dropped).  Weights are split on the host
// from the float64 state dict after a per-layer power-of-two scaling that keeps their lo parts out of the
// fp16 subnormal range (undone exactly in the epilogue); activations are split in the epilogue.
// BB_PREC_FAST16 issues only the hi*hi product (opt-in, outside the tolerance).
//
// Data flow per 128-row tile (rows are the MMA M dimension, one row per TMEM lane / per thread):
//   global -> smem stage (cp.async, prefetched one tile ahead) -> registers (normalise, split)
//   -> tcgen05.st A1 (fp16 hi|lo packed two per column) -> MMA -> D1 (fp32, TMEM) -> tcgen05.ld
//   -> scale, activation, split -> tcgen05.st A2 IN PLACE over D1 -> MMA -> ... -> D4 -> registers
//   -> smem stage -> coalesced global store.
// The A operand of every MMA is read from TMEM (the ".ts" form), the B operand (weights, hi and lo
// images of all four layers, 149 KiB) stays resident in shared memory for the whole kernel in the
// canonical no-swizzle K-major core-matrix layout (8 rows x 16 bytes per core matrix), loaded once per
// CTA with cp.async.bulk.  Biases ride along as one extra K column: every padded A operand has a spare
// K slot that holds 1.0 (produced by an extra weight row of the previous layer), and the matching weight
// column holds the bias, so the epilogue has no bias add.
//
// TMEM budget.  fp32 accumulator columns and packed hi|lo A columns have the same footprint, so the
// conversion is in place.  The 200-wide layer is processed in two N halves (112 + 96) that reuse one
// region, which keeps a tile pipeline at 256 columns (X 112 | Y 112 | Z 32): two independent pipelines
// (tiles interleaved) share the SM.
//
// Warp roles (576 threads): per pipeline 8 epilogue warps (two per TMEM lane quarter, splitting the 32-column
// chunks of an accumulator region) and one MMA-issuer warp.  Synchronisation is mbarrier-only on the hot
// path: the issuer commits a step's MMAs to `full_d`; epilogue warps drain chunk by chunk and arrive on
// `chunk_ready[c]` as soon as chunk c has been rewritten as the next A operand, so the issuer starts the next
// layer's k-steps on chunk c while later chunks are still being converted (the MMA latency hides behind the
// epilogue instead of adding to it).
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "bb_common.cuh"

namespace {

constexpr int TILE = 128;      // rows per tile = MMA M
constexpr int GROUP_T = 256;   // epilogue threads per pipeline: 2 warps per TMEM lane quarter, splitting the columns
constexpr int MAX_KITER = 40;  // k-steps of all MMAs of one program (28 for the CMS AE)
constexpr int MAX_STEPS = 6;
constexpr int REG_X = 0, REG_Y = 112, REG_Z = 224, PIPE_COLS = 256;

struct TcMma {
  int a_col, a_w;          // A operand region (TMEM columns == K elements: hi|lo packed per 32/16-column chunk)
  int ks0, ks_n;           // B k-step offset, number of k-steps (K = 16 per step)
  uint32_t b_hi, b_lo;     // smem byte offsets of the hi / lo weight images (already offset for N splits)
  uint32_t lbo;            // byte distance between the two 8-element K chunks of one k-step = Npad * 16
  int n, d_col, acc;       // MMA N, accumulator region, accumulate onto existing D
  int dep;                 // A operand is produced chunk by chunk by the previous step's epilogue
};
struct TcEpi {
  int col, w;              // accumulator region to drain
  float scale;             // 2^-sw: undoes the weight scaling
  int act, final;
};
struct TcStep { int n_mma; TcMma mma[2]; TcEpi epi; };
struct TcProgram {
  int n_steps, in_dim, out_dim;
  int a1_col, a1_w;        // where the loader puts the first A operand (a1_w = padded K of layer 0)
  int a1_after_step;       // that region is free for the NEXT tile once full_d of this step has been observed
  int out_stride;          // floats per row in the output stage (odd -> conflict-free)
  uint32_t w_bytes;        // size of the resident weight image
  TcStep step[MAX_STEPS];
};

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  // try_wait with a suspend-time hint parks the warp in hardware until the phase completes (or ~20 us pass), so
  // waiting warps do not burn issue slots the other pipeline's epilogue needs.  A protocol bug must not hang
  // the GPU: give up (trap -> launch error) after ~2 s.
  for (uint32_t spins = 0;; ++spins) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
    if (done) return;
    if (spins > 100000u) __trap();
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void group_bar(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(GROUP_T) : "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
#define TC_REGS16(v, o) "=r"(v[o+0]), "=r"(v[o+1]), "=r"(v[o+2]), "=r"(v[o+3]), "=r"(v[o+4]), "=r"(v[o+5]), "=r"(v[o+6]), "=r"(v[o+7]), \
                        "=r"(v[o+8]), "=r"(v[o+9]), "=r"(v[o+10]), "=r"(v[o+11]), "=r"(v[o+12]), "=r"(v[o+13]), "=r"(v[o+14]), "=r"(v[o+15])
#define TC_IN8(v, o) "r"(v[o+0]), "r"(v[o+1]), "r"(v[o+2]), "r"(v[o+3]), "r"(v[o+4]), "r"(v[o+5]), "r"(v[o+6]), "r"(v[o+7])

// each thread receives 32 / 16 consecutive fp32 columns of its own lane (row)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : TC_REGS16(v, 0), TC_REGS16(v, 16) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : TC_REGS16(v, 0) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[32], const int o) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
               TC_IN8(v, o), TC_IN8(v, o + 8) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[32], const int o) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), TC_IN8(v, o) : "memory");
}

// smem matrix descriptor: no swizzle, K-major; core matrix = 8 rows x 16 B, rows 16 B apart;
// SBO = 128 B between 8-row groups, LBO = distance between the two K chunks of a k-step
__device__ __forceinline__ uint32_t make_idesc(int n) {
  // c_format F32 (1) @4, a/b format F16 (0) @7/@10, a/b K-major, N>>3 @17, M>>4 @24
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);
}

// split two fp32 values into packed fp16 hi and lo words: hi = top 11 significant bits (truncated, so
// that x - hi is exact in fp32), lo = fp16_rn(x - hi)
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const float ah = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u);
  const float bh = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
  const __half2 h = __floats2half2_rn(ah, bh);
  const __half2 l = __floats2half2_rn(a - ah, b - bh);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ float act_apply(float s, int act) {
  if (act == BB_ACT_LEAKY) return fmaxf(s, BB_LEAKY * s);
  if (act == BB_ACT_RELU) return fmaxf(s, 0.f);
  return s;
}

// TMEM column of the hi part of k-step s of an A region (width w columns, chunked 32 | 16); lo = hi + half chunk
__device__ __forceinline__ void a_cols(int col, int w, int s, uint32_t& hi, uint32_t& lo) {
  const int base = col + ((s >> 1) << 5);
  const bool full = ((s >> 1) << 5) + 32 <= w;
  hi = base + (full ? ((s & 1) << 3) : 0);
  lo = hi + (full ? 16 : 8);
}

// ------------------------------------------------------------------------------------------------ kernel
// One k-step of the issue table: TMEM columns (relative to the pipeline) and the low descriptor words.
struct __align__(16) KIter { uint32_t a_hi, a_lo, b_hi, b_lo, d_acc, idesc, wait, pad; };
constexpr uint32_t B_DESC_HI = (128u >> 4) | (1u << 14);  // SBO = 128 B, descriptor version 1 (bit 46)
constexpr int MAX_CHUNKS = 4;                             // 32-column chunks of the widest accumulator region (112)

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// packed fp32x2 arithmetic (FFMA2 / FMUL2 on sm_100): two elements per instruction
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  return (uint64_t)__float_as_uint(lo) | ((uint64_t)__float_as_uint(hi) << 32);
}
__device__ __forceinline__ float lo32(uint64_t v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float hi32(uint64_t v) { return __uint_as_float((uint32_t)(v >> 32)); }
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// drain CW accumulator columns: scale, activation, split into fp16 hi|lo, write back in place
template <int CW, int ACT>
__device__ __forceinline__ void epi_chunk_inplace(const uint32_t taddr, const float scale) {
  uint32_t v[32], pk[32];
  if constexpr (CW == 32) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
  tc_wait_ld();
  const uint64_t c1 = pack2(scale, scale), c2 = pack2(scale * BB_LEAKY, scale * BB_LEAKY);
#pragma unroll
  for (int j = 0; j < CW / 2; ++j) {
    const uint64_t vv = pack2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
    const uint64_t sv = mul2(vv, c1);
    float a = lo32(sv), b = hi32(sv);
    if constexpr (ACT == BB_ACT_LEAKY) {
      const uint64_t lv = mul2(vv, c2);
      a = fmaxf(a, lo32(lv)); b = fmaxf(b, hi32(lv));
    } else if constexpr (ACT == BB_ACT_RELU) {
      a = fmaxf(a, 0.f); b = fmaxf(b, 0.f);
    }
    // hi = top 11 significant bits (truncated so that x - hi is exact in fp32), lo = fp16_rn(x - hi)
    const float ah = __uint_as_float(__float_as_uint(a) & 0xFFFFE000u);
    const float bh = __uint_as_float(__float_as_uint(b) & 0xFFFFE000u);
    const uint64_t dl = sub2(pack2(a, b), pack2(ah, bh));
    const __half2 h = __floats2half2_rn(ah, bh);
    const __half2 l = __floats2half2_rn(lo32(dl), hi32(dl));
    pk[j] = *reinterpret_cast<const uint32_t*>(&h);
    pk[CW / 2 + j] = *reinterpret_cast<const uint32_t*>(&l);
  }
  if constexpr (CW == 32) { tmem_st16(taddr, pk, 0); tmem_st16(taddr + 16, pk, 16); }
  else { tmem_st8(taddr, pk, 0); tmem_st8(taddr + 8, pk, 8); }
}

template <int CW>
__device__ __forceinline__ void epi_chunk_dispatch(const uint32_t taddr, const float scale, const int act) {
  if (act == BB_ACT_LEAKY) epi_chunk_inplace<CW, BB_ACT_LEAKY>(taddr, scale);
  else if (act == BB_ACT_RELU) epi_chunk_inplace<CW, BB_ACT_RELU>(taddr, scale);
  else epi_chunk_inplace<CW, BB_ACT_NONE>(taddr, scale);
}

template <int NGROUPS>
__global__ void __launch_bounds__(NGROUPS * (GROUP_T + 32), 1)
chain_tc_kernel(const __grid_constant__ TcProgram prog, const uint8_t* __restrict__ wimg, const void* __restrict__ in,
                const int in_dtype, const int in_aligned, const int64_t n_rows, const float* __restrict__ pre_min,
                const float* __restrict__ pre_range, const float* __restrict__ post_min,
                const float* __restrict__ post_range, void* __restrict__ out, const int out_dtype, const int fast,
                int* __restrict__ flag, const int dbg_step, float* __restrict__ dbg_out) {
  extern __shared__ __align__(128) uint8_t smem[];
  // per pipeline: [0,1] full_d of even / odd tiles (MMA -> epilogue; two so that the issuer may run one tile
  // ahead without phase aliasing), [2] a1_ready (loader -> MMA), [3..6] chunk_ready (epilogue -> MMA)
  __shared__ __align__(8) uint64_t bars[1 + NGROUPS * (3 + MAX_CHUNKS)];
  __shared__ uint32_t tmem_base_s;
  __shared__ KIter kit[MAX_KITER + 1];  // + one spare slot: the issuer prefetches entry e + 1
  __shared__ int kit_begin[MAX_STEPS + 1];
  __shared__ float norm_s[4][32];  // pre_min, pre_range, post_min, post_range (first 32 features)

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const bool is_mma = warp >= NGROUPS * (GROUP_T / 32);
  const int g = is_mma ? warp - NGROUPS * (GROUP_T / 32) : warp / (GROUP_T / 32);  // pipeline index
  const int tg = tid - g * GROUP_T;       // epilogue thread within the pipeline
  const int row = tg & (TILE - 1);        // tile row == TMEM lane
  const int half = (tg >> 7) & 1;         // which half of the column chunks this warp drains
  const int in_dim = prog.in_dim, out_dim = prog.out_dim;
  const int in_esz = in_dtype == BB_F16 ? 2 : 4;
  const uint32_t in_stage_bytes = (uint32_t)((TILE * in_dim * in_esz + 127) & ~127);
  const uint32_t out_stage_bytes = (uint32_t)((TILE * prog.out_stride * 4 + 127) & ~127);
  uint8_t* w_s = smem;
  uint8_t* in_s0 = smem + prog.w_bytes + g * (2 * in_stage_bytes + out_stage_bytes);  // two input stages
  float* out_s = reinterpret_cast<float*>(in_s0 + 2 * in_stage_bytes);
  const uint32_t bar_w = smem_u32(&bars[0]);
  const uint32_t bar_full = smem_u32(&bars[1 + g * (3 + MAX_CHUNKS)]);  // + 8 * (tile parity)
  const uint32_t bar_a1 = bar_full + 16;
  const uint32_t bar_chunk0 = bar_full + 24;

  if (tid == 0) {
    mbar_init(bar_w, 1);
    for (int i = 0; i < NGROUPS; ++i) {
      const uint32_t b0 = smem_u32(&bars[1 + i * (3 + MAX_CHUNKS)]);
      mbar_init(b0, 1);                      // full_d (even tiles): one tcgen05.commit
      mbar_init(b0 + 8, 1);                  // full_d (odd tiles)
      mbar_init(b0 + 16, GROUP_T / 32);      // a1_ready: every epilogue warp
      for (int c = 0; c < MAX_CHUNKS; ++c) mbar_init(b0 + 24 + 8 * c, 4);  // chunk_ready: the 4 warps of one half
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // issue table: every k-step of every MMA of the program, in issue order
    int n = 0;
    for (int s = 0; s < prog.n_steps; ++s) {
      kit_begin[s] = n;
      for (int m = 0; m < prog.step[s].n_mma; ++m) {
        const TcMma& mm = prog.step[s].mma[m];
        for (int k = 0; k < mm.ks_n; ++k, ++n) {
          KIter e;
          a_cols(mm.a_col, mm.a_w, k, e.a_hi, e.a_lo);
          const uint32_t koff = (uint32_t)(mm.ks0 + k) * 2u * mm.lbo;  // two 8-wide K chunks per k-step
          const uint32_t lbo_f = ((mm.lbo >> 4) & 0x3FFF) << 16;
          e.b_hi = (((smem_u32(w_s) + mm.b_hi + koff) >> 4) & 0x3FFF) | lbo_f;
          e.b_lo = (((smem_u32(w_s) + mm.b_lo + koff) >> 4) & 0x3FFF) | lbo_f;
          e.d_acc = (uint32_t)mm.d_col | ((k > 0 || mm.acc) ? 0x80000000u : 0u);
          e.idesc = make_idesc(mm.n);
          e.wait = (mm.dep && (k & 1) == 0) ? (uint32_t)(k >> 1) + 1u : 0u;  // first k-step of a 32-column chunk
          e.pad = 0;
          kit[n] = e;
        }
      }
    }
    kit_begin[prog.n_steps] = n;
  }
  if (tid < 128) {  // column (de)normalisation vectors, read by every thread for every row
    const int which = tid >> 5, k = tid & 31;
    const float* src = which == 0 ? pre_min : which == 1 ? pre_range : which == 2 ? post_min : post_range;
    const int dim = which < 2 ? in_dim : out_dim;
    float v = (src != nullptr && k < dim) ? src[k] : (which & 1 ? 1.f : 0.f);
    if (which == 1) v = __frcp_rn(v);  // the loader multiplies by 1 / range
    norm_s[which][k] = v;
  }
  if (tid < 32) {  // warp 0 owns the TMEM allocation
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  if (tid == 0) {  // resident weight image: global -> smem through the async proxy (what the MMA reads through)
    mbar_expect_tx(bar_w, prog.w_bytes);
    for (uint32_t off = 0; off < prog.w_bytes; off += 32768) {
      const uint32_t n = prog.w_bytes - off < 32768 ? prog.w_bytes - off : 32768;
      bulk_g2s(smem_u32(w_s + off), wimg + off, n, bar_w);
    }
  }

  const int64_t n_tiles = (n_rows + TILE - 1) / TILE;
  const int64_t tile_stride = (int64_t)gridDim.x * NGROUPS;
  const int64_t tile0 = (int64_t)blockIdx.x * NGROUPS + g;
  const uint32_t tcol0 = tmem_base + g * PIPE_COLS;
  // test hook, dbg_step == -2: SM-clock timestamps of the pipeline events of CTA 0 / pipeline 0, 64 slots per
  // tile (0..31 epilogue warp 0, 32..63 MMA issuer), first 16 tiles
  const bool tracing = dbg_out != nullptr && dbg_step == -2 && blockIdx.x == 0 && g == 0;
  auto trace = [&](int64_t local_tile, int slot) {
    if (tracing && local_tile < 16) reinterpret_cast<uint32_t*>(dbg_out)[local_tile * 64 + slot] = (uint32_t)clock64();
  };

  if (is_mma) {
    // ================================================================== MMA issuer (one lane per pipeline)
    // The whole warp runs this loop converged (all values are warp-uniform); only the tcgen05 instructions are
    // predicated on one elected lane.  A lane-0-only loop makes the compiler wrap every UTCHMMA in an
    // ELECT / R2UR / BRA.U.ANY serialisation sequence (~130 cycles per MMA).
    {
      mbar_wait(bar_w, 0);  // weights resident
      uint32_t par_a1 = 0, par_chunk = 0;
      int64_t lt = 0;
      const bool lane0 = (tid & 31) == 0;
      // Everything the tcgen05 instructions consume is warp-uniform and is derived here from kernel parameters
      // (constant bank) and two shuffled values, so the compiler keeps descriptors and TMEM addresses in uniform
      // registers: a k-step costs a handful of uniform adds, not a shared-memory table read plus a dozen R2UR.
      const uint32_t tcol_u = __shfl_sync(0xffffffffu, tcol0, 0);
      const uint32_t w_addr = __shfl_sync(0xffffffffu, smem_u32(w_s), 0);
      const uint32_t bar_full_u = __shfl_sync(0xffffffffu, bar_full, 0);
      const uint32_t bar_chunk_u = bar_full_u + 24u, bar_a1_u = bar_full_u + 16u;
      for (int64_t tile = tile0; tile < n_tiles; tile += tile_stride, ++lt) {
        if (lane0) trace(lt, 32);
        mbar_wait(bar_a1_u, par_a1);
        par_a1 ^= 1u;
        tc_fence_after();
        if (lane0) trace(lt, 33);
#pragma unroll
        for (int s = 0; s < MAX_STEPS; ++s) {
          if (s < prog.n_steps) {
#pragma unroll
            for (int m = 0; m < 2; ++m) {
              if (m < prog.step[s].n_mma) {
                const TcMma& mm = prog.step[s].mma[m];
                const uint32_t idesc = make_idesc(mm.n);
                const uint32_t lbo_f = ((mm.lbo >> 4) & 0x3FFFu) << 16;
                const uint32_t k_off = (uint32_t)mm.ks0 * 2u * mm.lbo;
                uint32_t bh = (((w_addr + mm.b_hi + k_off) >> 4) & 0x3FFFu) | lbo_f;
                uint32_t bl = (((w_addr + mm.b_lo + k_off) >> 4) & 0x3FFFu) | lbo_f;
                const uint32_t b_step = (2u * mm.lbo) >> 4;  // two 8-wide K chunks per k-step
                const uint32_t d_addr = tcol_u + (uint32_t)mm.d_col;
                const int ks_n = mm.ks_n, a_w = mm.a_w, dep = mm.dep;
                const uint32_t a_base = tcol_u + (uint32_t)mm.a_col;
                for (int k = 0; k < ks_n; ++k) {
                  if (dep && (k & 1) == 0) {  // this k-step opens a chunk the previous step's epilogue is still producing
                    const uint32_t c = (uint32_t)k >> 1;
                    mbar_wait(bar_chunk_u + 8u * c, (par_chunk >> c) & 1u);
                    par_chunk ^= 1u << c;
                    tc_fence_after();
                    if (lane0) trace(lt, 34 + 5 * s + (int)c);
                  }
                  // A columns of k-step k: 32-column chunks hold hi k-steps at +0 / +8 and lo at +16 / +24; a trailing
                  // 16-column chunk holds hi at +0 and lo at +8
                  const uint32_t cb = ((uint32_t)k >> 1) << 5;
                  const bool full = (int)cb + 32 <= a_w;
                  const uint32_t a_hi = a_base + cb + (full ? ((uint32_t)k & 1u) << 3 : 0u);
                  const uint32_t a_lo = a_hi + (full ? 16u : 8u);
                  const uint32_t acc = (k > 0 || mm.acc) ? 1u : 0u;
                  // hi*hi (accumulate flag), then hi*lo and lo*hi (always accumulate)
                  if (!fast) {
                    asm volatile(
                        "{\n\t.reg .pred e, p, t;\n\t.reg .b64 bh, bl;\n\t"
                        "elect.sync _|e, 0xffffffff;\n\t"
                        "setp.ne.b32 p, %6, 0;\n\t"
                        "setp.eq.b32 t, %6, %6;\n\t"
                        "mov.b64 bh, {%2, %7};\n\t"
                        "mov.b64 bl, {%3, %7};\n\t"
                        "@e tcgen05.mma.cta_group::1.kind::f16 [%4], [%0], bh, %5, p;\n\t"
                        "@e tcgen05.mma.cta_group::1.kind::f16 [%4], [%0], bl, %5, t;\n\t"
                        "@e tcgen05.mma.cta_group::1.kind::f16 [%4], [%1], bh, %5, t;\n\t}"
                        ::"r"(a_hi), "r"(a_lo), "r"(bh), "r"(bl), "r"(d_addr), "r"(idesc), "r"(acc), "r"(B_DESC_HI) : "memory");
                  } else {
                    asm volatile(
                        "{\n\t.reg .pred e, p;\n\t.reg .b64 bh;\n\t"
                        "elect.sync _|e, 0xffffffff;\n\t"
                        "setp.ne.b32 p, %4, 0;\n\t"
                        "mov.b64 bh, {%1, %5};\n\t"
                        "@e tcgen05.mma.cta_group::1.kind::f16 [%2], [%0], bh, %3, p;\n\t}"
                        ::"r"(a_hi), "r"(bh), "r"(d_addr), "r"(idesc), "r"(acc), "r"(B_DESC_HI) : "memory");
                  }
                  bh += b_step; bl += b_step;
                }
              }
            }
            asm volatile(
                "{\n\t.reg .pred e;\n\t"
                "elect.sync _|e, 0xffffffff;\n\t"
                "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar_full_u + 8u * (uint32_t)(lt & 1)) : "memory");
            if (lane0) trace(lt, 34 + 5 * s + 4);
          }
        }
      }
    }
    __syncwarp();
  } else {
    // ================================================================== loader + epilogue warps
    const uint32_t lane_addr = (uint32_t)((row & ~31) << 16);  // TMEM lane base of this warp (32 lanes per warp)
    const bool has_pre = pre_min != nullptr, has_post = post_min != nullptr;
    const int bar_id = 1 + g;

    // cooperative copy of one input tile into a stage (16-byte cp.async when aligned and full)
    auto fetch = [&](int64_t tile, uint8_t* dst) {
      const int rows = (int)min((int64_t)TILE, n_rows - tile * TILE);
      const size_t base = (size_t)tile * TILE * in_dim * in_esz;
      const int bytes = rows * in_dim * in_esz;
      const uint8_t* src = reinterpret_cast<const uint8_t*>(in) + base;
      if (in_aligned && rows == TILE) {
        for (int c = tg * 16; c < bytes; c += GROUP_T * 16) cp_async16(smem_u32(dst + c), src + c);
      } else if (in_esz == 4) {
        for (int e = tg; e < bytes / 4; e += GROUP_T) reinterpret_cast<float*>(dst)[e] = reinterpret_cast<const float*>(src)[e];
      } else {
        for (int e = tg; e < bytes / 2; e += GROUP_T) reinterpret_cast<__half*>(dst)[e] = reinterpret_cast<const __half*>(src)[e];
      }
    };

    // first A operand of a tile: this thread's row, k-step `half` (16 features) -> normalise -> 1.0 in the bias
    // slot -> split -> TMEM, then tell the issuer.
    auto convert_a1 = [&](int64_t tile, const uint8_t* in_s) {
      const int rows = (int)min((int64_t)TILE, n_rows - tile * TILE);
      if (half * 16 < prog.a1_w) {
        uint32_t pk[32];
        float xv[16];
        const int k0 = half * 16;
        if (in_esz == 4 && (in_dim & 3) == 0) {  // 128-bit loads of this row's 16 features
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k0 + 4 * q < in_dim && row < rows) t = reinterpret_cast<const float4*>(in_s)[(row * in_dim + k0) / 4 + q];
            xv[4 * q] = t.x; xv[4 * q + 1] = t.y; xv[4 * q + 2] = t.z; xv[4 * q + 3] = t.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int k = k0 + j;
            float x = 0.f;
            if (k < in_dim && row < rows)
              x = in_esz == 4 ? reinterpret_cast<const float*>(in_s)[row * in_dim + k]
                              : __half2float(reinterpret_cast<const __half*>(in_s)[row * in_dim + k]);
            xv[j] = x;
          }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int k = k0 + j;
          // numpy float32 (x - min) / range (data_processing.py:151); here the quotient is x * rcp_rn(range):
          // within 1 ulp of the IEEE quotient, far inside the 1e-5 budget of the latent
          if (k < in_dim) { if (has_pre && row < rows) xv[j] = __fsub_rn(xv[j], norm_s[0][k]) * norm_s[1][k]; }
          else xv[j] = k == in_dim ? 1.f : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) split2(xv[2 * j], xv[2 * j + 1], pk[j], pk[8 + j]);
        // k-step s of a 32-wide chunk: hi words at +8s, lo words at +16+8s; a 16-wide chunk: hi +0, lo +8
        const uint32_t taddr = tcol0 + lane_addr + prog.a1_col + (prog.a1_w >= 32 ? half * 8 : 0);
        tmem_st8(taddr, pk, 0);
        tmem_st8(taddr + (prog.a1_w >= 32 ? 16 : 8), pk, 8);
        tc_wait_st();
      }
      tc_fence_before();
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(bar_a1);
    };

    if (tile0 < n_tiles) fetch(tile0, in_s0);
    cp_async_commit();
    uint32_t parity2 = 0;  // bit p: phase parity of full_d[p]
    int64_t lt = 0;
    const bool tr0 = tg == 0;
    // Variant tried and dropped: converting the NEXT tile's first operand mid-tile (as soon as its TMEM region is
    // free) so the issuer runs a tile ahead.  TMEM loads queue in order behind every MMA already issued on the SM,
    // so the run-ahead MMAs delayed the remaining epilogues by more than the loader latency they hid
    // (2.81 vs 3.15 G rows/s, profiles/r01_tc_trace.md).

    for (int64_t tile = tile0; tile < n_tiles; tile += tile_stride, ++lt) {
      const int rows = (int)min((int64_t)TILE, n_rows - tile * TILE);
      const uint32_t tp = (uint32_t)(lt & 1);
      if (tr0) trace(lt, 0);
      {  // prefetch this pipeline's next tile into the other stage, then wait for the current one
        const int64_t nxt = tile + tile_stride;
        if (nxt < n_tiles) fetch(nxt, in_s0 + (uint32_t)((lt + 1) & 1) * in_stage_bytes);
        cp_async_commit();
        cp_async_wait_1();
      }
      group_bar(bar_id);
      if (tr0) trace(lt, 1);
      convert_a1(tile, in_s0 + (uint32_t)(lt & 1) * in_stage_bytes);
      if (tr0) trace(lt, 2);

      for (int s = 0; s < prog.n_steps; ++s) {
        mbar_wait(bar_full + 8u * tp, (parity2 >> tp) & 1u);  // the accumulator of step s is complete
        parity2 ^= 1u << tp;
        tc_fence_after();
        if (tr0) trace(lt, 3 + 4 * s);
        const TcEpi& ep = prog.step[s].epi;
        const int ep_w = ep.w, ep_col = ep.col, ep_act = ep.act;
        const float ep_scale = ep.scale;
        if (dbg_out != nullptr) {  // test hook: dump the scaled accumulator before it is rewritten in place
          if (dbg_step == s && half == 0) {
            for (int c0 = 0; c0 < ep_w; c0 += 16) {
              uint32_t v[32];
              tmem_ld16(tcol0 + lane_addr + ep_col + c0, v);  // .sync.aligned: the whole warp, also rows past the tail
              tc_wait_ld();
              if (row < rows) {
#pragma unroll
                for (int j = 0; j < 16; ++j) dbg_out[((size_t)tile * TILE + row) * ep_w + c0 + j] = __uint_as_float(v[j]) * ep_scale;
              }
            }
          }
          group_bar(bar_id);
        }
        if (!ep.final) {
          for (int c0 = half * 32; c0 < ep_w; c0 += 64) {
            const uint32_t taddr = tcol0 + lane_addr + ep_col + c0;
            if (ep_w - c0 >= 32) epi_chunk_dispatch<32>(taddr, ep_scale, ep_act);
            else epi_chunk_dispatch<16>(taddr, ep_scale, ep_act);
            tc_wait_st();
            tc_fence_before();
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(bar_chunk0 + 8u * (uint32_t)(c0 >> 5));  // chunk c0/32 is a valid A operand now
            if (tr0) trace(lt, 4 + 4 * s + (c0 >> 6));
          }
        } else if (half == 0) {
          uint32_t v[32];
          const uint32_t taddr = tcol0 + lane_addr + ep_col;
          if (ep_w > 16) tmem_ld32(taddr, v); else tmem_ld16(taddr, v);
          tc_wait_ld();
          bool bad = false;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (j < out_dim && j < ep_w) {
              float y = act_apply(__uint_as_float(v[j]) * ep_scale, ep_act);
              bad |= !(fabsf(y) <= 3.0e38f);  // inf / NaN: an fp16 operand overflowed somewhere upstream
              if (has_post) y = fmaf(y, norm_s[3][j], norm_s[2][j]);  // y * range + min (data_processing.py:203)
              out_s[row * prog.out_stride + j] = y;
            }
          }
          if (bad && row < rows) atomicOr(flag, 1);
        }
      }
      if (tr0) trace(lt, 24);
      tc_fence_before();
      group_bar(bar_id);
      if (tr0) trace(lt, 25);
      // ---- coalesced store of the output tile (the stage is dense row-major, so this is a flat copy)
      {
        const size_t base = (size_t)tile * TILE * out_dim;
        const int n_el = rows * out_dim;
        if (out_dtype == BB_F32 && rows == TILE && (reinterpret_cast<uintptr_t>(out) & 15u) == 0) {
          float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + base);
          for (int e = tg; e < n_el / 4; e += GROUP_T) dst[e] = reinterpret_cast<const float4*>(out_s)[e];
        } else {
          for (int e = tg; e < n_el; e += GROUP_T) {
            const float y = out_s[e];
            if (out_dtype == BB_F16) reinterpret_cast<__half*>(out)[base + e] = __float2half_rn(y);
            else reinterpret_cast<float*>(out)[base + e] = y;
          }
        }
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (tid < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
}

// ------------------------------------------------------------------------------------------------ host side
struct TcHost {
  TcProgram prog;
  int n_groups;
  size_t smem_bytes;
};

inline int rup16(int x) { return (x + 15) & ~15; }

uint16_t f2h(float f) {  // float -> fp16 bits, round to nearest even (host)
  __half h = __float2half_rn(f);
  uint16_t u;
  memcpy(&u, &h, 2);
  return u;
}
float h2f(uint16_t u) {
  __half h;
  memcpy(&h, &u, 2);
  return __half2float(h);
}

}  // namespace

// Builds the weight image + step program for a 4-layer chain whose only wide layer is 113..208 padded
// columns (the hidden 200) and whose other padded widths fit 112; anything else stays on the fp32 kernel.
int bb_tc_prepare(bb_ctx* ctx, Chain* c) {
  c->tc_ok = false;
  const ChainDesc& d = c->desc;
  if (d.n_layers != 4) return BB_ERR_UNSUPPORTED;
  int K[4], N[4], Kp[4], Np[4];
  for (int l = 0; l < 4; ++l) { K[l] = d.layer[l].K; N[l] = d.layer[l].N; Kp[l] = rup16(K[l] + 1); }
  for (int l = 0; l < 4; ++l) Np[l] = l < 3 ? Kp[l + 1] : rup16(N[l]);
  // region plan (see header comment): exactly one wide layer, at position 0 (encoder) or 2 (decoder)
  int wide = -1;
  for (int l = 0; l < 4; ++l)
    if (Np[l] > 112) { if (wide >= 0 || Np[l] > 208) return BB_ERR_UNSUPPORTED; wide = l; }
  if (wide != 0 && wide != 2) return BB_ERR_UNSUPPORTED;
  if (Kp[0] > 32 || Np[3] > 32 || d.in_dim > 31 || d.out_dim > 32) return BB_ERR_UNSUPPORTED;  // first A operand / last accumulator live in Z (32 columns)
  if (wide == 0 && (Np[2] > 112 || Np[1] > 112)) return BB_ERR_UNSUPPORTED;
  if (wide == 2 && (Np[0] > 112 || Np[1] > 112)) return BB_ERR_UNSUPPORTED;

  TcHost* h = new TcHost();
  TcProgram& p = h->prog;
  memset(&p, 0, sizeof(p));
  p.in_dim = d.in_dim; p.out_dim = d.out_dim;
  p.out_stride = d.out_dim;  // dense rows: the tile leaves the stage as one flat copy
  // ---- weight image: per layer hi then lo, canonical K-major core matrices: ((k/8) * Np + n) * 16 B + (k%8) * 2 B
  uint32_t off = 0, b_hi[4], b_lo[4];
  float scale[4];
  std::vector<uint8_t> img;
  for (int l = 0; l < 4; ++l) {
    const size_t mat = (size_t)Np[l] * Kp[l] * 2;
    b_hi[l] = off; b_lo[l] = off + (uint32_t)mat; off += 2 * (uint32_t)mat;
    img.resize(off, 0);
    std::vector<double> w((size_t)Np[l] * Kp[l], 0.0);
    double mx = 1.0;
    for (int n = 0; n < N[l]; ++n) {
      for (int k = 0; k < K[l]; ++k) w[(size_t)n * Kp[l] + k] = c->w_host[l][(size_t)n * K[l] + k];
      w[(size_t)n * Kp[l] + K[l]] = c->b_host[l][n];   // bias rides on the constant-one K slot
    }
    if (l < 3) w[(size_t)N[l] * Kp[l] + K[l]] = 1.0;    // produces the constant one of the next layer's bias slot
    for (double v : w) mx = std::fabs(v) > mx ? std::fabs(v) : mx;
    const int sw = (int)std::floor(std::log2(2047.0 / mx));
    scale[l] = (float)std::ldexp(1.0, -sw);
    uint16_t* hi = reinterpret_cast<uint16_t*>(img.data() + b_hi[l]);
    uint16_t* lo = reinterpret_cast<uint16_t*>(img.data() + b_lo[l]);
    for (int n = 0; n < Np[l]; ++n)
      for (int k = 0; k < Kp[l]; ++k) {
        const double v = std::ldexp(w[(size_t)n * Kp[l] + k], sw);
        const uint16_t hb = f2h((float)v);
        const uint16_t lb = f2h((float)(v - (double)h2f(hb)));
        const size_t idx = ((size_t)(k / 8) * Np[l] + n) * 8 + (k % 8);
        hi[idx] = hb; lo[idx] = lb;
      }
  }
  p.w_bytes = off;
  // ---- step program
  auto mma = [&](int l, int a_col, int a_w, int ks0, int ks_n, int n0, int n, int d_col, int acc) {
    TcMma m;
    m.a_col = a_col; m.a_w = a_w; m.ks0 = ks0; m.ks_n = ks_n;
    m.b_hi = b_hi[l] + (uint32_t)n0 * 16; m.b_lo = b_lo[l] + (uint32_t)n0 * 16;
    m.lbo = (uint32_t)Np[l] * 16; m.n = n; m.d_col = d_col; m.acc = acc; m.dep = 0;
    return m;
  };
  auto epi = [&](int l, int col, int w, int fin) {
    TcEpi e;
    e.col = col; e.w = w; e.scale = scale[l]; e.act = d.layer[l].act; e.final = fin;
    return e;
  };
  // the first A operand lives where nothing else is live at the start of a tile AND becomes free early, so the next
  // tile's operand can be written while this tile is still running: encoder Z (read by steps 0 and 1), decoder Y
  // (A1 is read by step 0; Y then holds D2/A3 until step 3 has consumed it, and is idle during the last step)
  p.a1_col = wide == 0 ? REG_Z : REG_Y; p.a1_w = Kp[0];
  p.a1_after_step = wide == 0 ? 1 : 3;  // informational: first step after which the A1 region is idle
  int s = 0;
  if (wide == 0) {  // encoder: K0 -> 208 -> Np1 -> Np2 -> Np3
    const int na = 112, nb = Np[0] - 112;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(0, REG_Z, Kp[0], 0, Kp[0] / 16, 0, na, REG_X, 0); p.step[s].epi = epi(0, REG_X, na, 0); ++s;
    p.step[s].n_mma = 2; p.step[s].mma[0] = mma(1, REG_X, na, 0, na / 16, 0, Np[1], REG_Y, 0);
    p.step[s].mma[1] = mma(0, REG_Z, Kp[0], 0, Kp[0] / 16, na, nb, REG_X, 0); p.step[s].epi = epi(0, REG_X, nb, 0); ++s;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(1, REG_X, nb, na / 16, nb / 16, 0, Np[1], REG_Y, 1); p.step[s].epi = epi(1, REG_Y, Np[1], 0); ++s;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(2, REG_Y, Np[1], 0, Np[1] / 16, 0, Np[2], REG_X, 0); p.step[s].epi = epi(2, REG_X, Np[2], 0); ++s;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(3, REG_X, Np[2], 0, Np[2] / 16, 0, Np[3], REG_Y, 0); p.step[s].epi = epi(3, REG_Y, Np[3], 1); ++s;
  } else {          // decoder: K0 -> Np0 -> Np1 -> 208 -> Np3
    const int na = 112, nb = Np[2] - 112;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(0, REG_Y, Kp[0], 0, Kp[0] / 16, 0, Np[0], REG_X, 0); p.step[s].epi = epi(0, REG_X, Np[0], 0); ++s;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(1, REG_X, Np[0], 0, Np[0] / 16, 0, Np[1], REG_Y, 0); p.step[s].epi = epi(1, REG_Y, Np[1], 0); ++s;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(2, REG_Y, Np[1], 0, Np[1] / 16, 0, na, REG_X, 0); p.step[s].epi = epi(2, REG_X, na, 0); ++s;
    p.step[s].n_mma = 2; p.step[s].mma[0] = mma(3, REG_X, na, 0, na / 16, 0, Np[3], REG_Z, 0);
    p.step[s].mma[1] = mma(2, REG_Y, Np[1], 0, Np[1] / 16, na, nb, REG_X, 0); p.step[s].epi = epi(2, REG_X, nb, 0); ++s;
    p.step[s].n_mma = 1; p.step[s].mma[0] = mma(3, REG_X, nb, na / 16, nb / 16, 0, Np[3], REG_Z, 1); p.step[s].epi = epi(3, REG_Z, Np[3], 1); ++s;
  }
  p.n_steps = s;
  // an MMA whose A region is the accumulator the previous step's epilogue rewrites in place can start chunk by chunk
  for (int i = 1; i < s; ++i)
    for (int m = 0; m < p.step[i].n_mma; ++m)
      p.step[i].mma[m].dep = (!p.step[i - 1].epi.final && p.step[i].mma[m].a_col == p.step[i - 1].epi.col) ? 1 : 0;
  // ---- shared memory: weight image + per pipeline (input stage + output stage); prefer two pipelines
  auto smem_need = [&](int groups, int in_esz) {
    const size_t in_b = ((size_t)TILE * d.in_dim * in_esz + 127) & ~(size_t)127;
    const size_t out_b = ((size_t)TILE * p.out_stride * 4 + 127) & ~(size_t)127;
    return (size_t)p.w_bytes + groups * (2 * in_b + out_b);
  };
  h->n_groups = smem_need(2, 4) + 4096 <= ctx->smem_optin ? 2 : (smem_need(1, 4) + 4096 <= ctx->smem_optin ? 1 : 0);
  if (h->n_groups == 0 || (p.w_bytes & 15)) { delete h; return BB_ERR_UNSUPPORTED; }
  h->smem_bytes = smem_need(h->n_groups, 4);
  if (c->tc_blob_dev) cudaFree(c->tc_blob_dev);
  BB_CUDA(cudaMalloc(&c->tc_blob_dev, img.size()));
  BB_CUDA(cudaMemcpy(c->tc_blob_dev, img.data(), img.size(), cudaMemcpyHostToDevice));
  c->tc_blob_bytes = img.size();
  // the attribute belongs to the kernel, not to this chain (encoder and decoder share the kernels): always
  // allow the device maximum
  cudaFuncAttributes fa;
  BB_CUDA(cudaFuncGetAttributes(&fa, chain_tc_kernel<2>));
  BB_CUDA(cudaFuncSetAttribute(chain_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(ctx->smem_optin - fa.sharedSizeBytes)));
  BB_CUDA(cudaFuncGetAttributes(&fa, chain_tc_kernel<1>));
  BB_CUDA(cudaFuncSetAttribute(chain_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(ctx->smem_optin - fa.sharedSizeBytes)));
  delete reinterpret_cast<TcHost*>(c->tc_host);
  c->tc_host = h;
  c->tc_ok = true;
  // the reference AE family (hidden 200 / 100 / 50) also runs on the statically shaped kernel (bb_chain_tc4.cu),
  // which reads the same weight image
  Tc4Plan& t4 = c->tc4;
  t4 = Tc4Plan();
  const bool enc_family = wide == 0 && Np[0] == 208 && Np[1] == 112 && Np[2] == 64;
  const bool dec_family = wide == 2 && Np[0] == 64 && Np[1] == 112 && Np[2] == 208;
  if ((enc_family || dec_family) && getenv("BALER_B200_TC_V3") == nullptr) {
    t4.ok = true; t4.enc = enc_family ? 1 : 0; t4.ka = Kp[0]; t4.nl = Np[3];
    for (int l = 0; l < 4; ++l) {
      const int act = d.layer[l].act;
      // activation as y = c1 * v + c2 * |v| (see convert16 in bb_chain_tc4.cu)
      t4.c1[l] = act == BB_ACT_LEAKY ? scale[l] * (0.5f + 0.5f * BB_LEAKY) : act == BB_ACT_RELU ? scale[l] * 0.5f : scale[l];
      t4.c2[l] = act == BB_ACT_LEAKY ? scale[l] * (0.5f - 0.5f * BB_LEAKY) : act == BB_ACT_RELU ? scale[l] * 0.5f : 0.f;
    }
  }
  return BB_OK;
}

void bb_tc_release(Chain* c) {
  delete reinterpret_cast<TcHost*>(c->tc_host);
  c->tc_host = nullptr;
}

int bb_tc_launch_dbg(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows, const float* pre_min,
                     const float* pre_range, const float* post_min, const float* post_range, void* out, int out_dtype,
                     int fast, int* flag_dev, int dbg_step, float* dbg_out, int force_groups, cudaStream_t stream) {
  if (!c->tc_ok) return BB_ERR_UNSUPPORTED;
  if (n_rows == 0) return BB_OK;
  if (c->tc4.ok && force_groups == 0 && (dbg_step == -1 || dbg_step == -2)) {
    // the statically shaped kernel: exact and fast arithmetic, float32 or (on the latent side) float16 rows
    const int rc = bb_tc4_launch(ctx, c, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out, out_dtype, fast,
                                 flag_dev, dbg_step == -2 ? reinterpret_cast<uint32_t*>(dbg_out) : nullptr, stream);
    if (rc == BB_OK) {
      c->last_route = BB_ROUTE_TC4;
      c->last_tile_rows = 2 * TILE;  // two pipelines per CTA (NPIPE of bb_chain_tc4.cu)
    }
    if (rc != BB_ERR_UNSUPPORTED) return rc;
  }
  const TcHost* h = reinterpret_cast<const TcHost*>(c->tc_host);
  const int groups = force_groups > 0 && force_groups < h->n_groups ? force_groups : h->n_groups;
  const int64_t n_tiles = (n_rows + TILE - 1) / TILE;
  const int64_t want = (n_tiles + groups - 1) / groups;
  const int grid = (int)(want < ctx->sm_count ? want : ctx->sm_count);
  const int aligned = (reinterpret_cast<uintptr_t>(in) & 15u) == 0;
  c->last_route = BB_ROUTE_TC;
  c->last_tile_rows = groups * TILE;
  if (groups == 2)
    chain_tc_kernel<2><<<grid, 2 * (GROUP_T + 32), h->smem_bytes, stream>>>(h->prog, (const uint8_t*)c->tc_blob_dev, in, in_dtype, aligned,
                                                                     n_rows, pre_min, pre_range, post_min, post_range, out,
                                                                     out_dtype, fast, flag_dev, dbg_step, dbg_out);
  else
    chain_tc_kernel<1><<<grid, GROUP_T + 32, h->smem_bytes, stream>>>(h->prog, (const uint8_t*)c->tc_blob_dev, in, in_dtype, aligned,
                                                                 n_rows, pre_min, pre_range, post_min, post_range, out,
                                                                 out_dtype, fast, flag_dev, dbg_step, dbg_out);
  return (int)cudaGetLastError();
}

int bb_tc_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows, const float* pre_min,
                 const float* pre_range, const float* post_min, const float* post_range, void* out, int out_dtype,
                 int fast, int* flag_dev, cudaStream_t stream) {
  return bb_tc_launch_dbg(ctx, c, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out, out_dtype, fast,
                          flag_dev, -1, nullptr, 0, stream);
}
