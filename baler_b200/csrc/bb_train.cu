// Training step of the dense autoencoder: forward, sum-MSE (+ optional L1 chain) loss, backward, Adam.
//
// Replaces the body of the batch loop of training.fit (reference baler/modules/training.py:64-97):
//   optimizer.zero_grad(); recon = model(x); loss = mse_sum_loss_l1(...); loss.backward(); optimizer.step()
// with utils.mse_sum_loss_l1 (utils.py:176-211) and torch.optim.Adam defaults (training.py:266).
//
// A step is three launches on one stream, no host synchronisation:
//   1. train_fwd_bwd_kernel  one CTA (512 threads) per 4 rows of the batch.  The CTA walks the 8 layers forward and
//      the 8 layers backward with every activation of its rows in shared memory; the weight matrix of the next
//      pass (W^T [K][N] forward, W [N][K] backward) is staged L2 -> shared memory with cp.async while the current
//      pass computes.  Narrow layers split the reduction over threads (KP partial sums, combined in a fixed
//      order).  It leaves the layer inputs A_l and the pre-activation gradients dZ_l (row-major [B][dim]) in
//      global scratch and one loss partial per CTA.
//   2. train_dw_kernel       dW_l = dZ_l^T A_l as 64x64 output tiles x 64-row splits, 4x4 register tiles,
//      written as per-split partial sums (no atomics: the sum order is fixed, results are reproducible).
//   3. train_adam_kernel     sums the split partials into the flat gradient, applies Adam and refreshes the
//      transposed weight copy.  With data parallelism the gradient (+ the batch loss in its last slot)
//      is all-reduced (SUM, because the loss is a sum: utils.py:195) between 2 and 3 by the caller.
// Everything is fp32 FFMA; a 512-row step is ~0.2 GFLOP, so the step is latency- not throughput-bound.
#include <cmath>
#include <cstring>
#include <new>

#include <cooperative_groups.h>
#include <curand_philox4x32_x.h>

#include "bb_common.cuh"
#include "bb_train_f64.cuh"
#include "bb_train_tc.cuh"

namespace {
// Programmatic dependent launch: the three kernels of a training step are launched back to back with
// cudaLaunchAttributeProgrammaticStreamSerialization, every kernel lets its successor's CTAs be scheduled at once
// (launch_dependents) and waits for its predecessor's results (wait) before touching global memory, so launch latency
// and CTA scheduling of kernel n + 1 overlap the execution of kernel n.  Both are no-ops in an ordinary launch.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KArgs, typename... Args>
cudaError_t pdl_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
}  // namespace

namespace {

constexpr int NL = 8;       // dense layers F-200-100-50-z-50-100-200-F
constexpr int RT = 4;       // rows per CTA in the forward/backward kernel (128 CTAs for a 512-row batch)
constexpr int NT = 256;      // dW and Adam kernels
constexpr int NT_FB = 512;   // forward/backward kernel: more warps to hide shared-memory latency, wider reduction splits
constexpr int DW_T = 64;    // dW tile edge and rows per split
constexpr int DW_LD = DW_T + 4;

struct TrainDims {
  int dims[NL + 1];
  int act[NL];           // activation after layer l in the model chain
  int w_off[NL], b_off[NL], wt_off[NL];
  int a_off[NL + 1];     // float offset of act_l rows in the per-row activation scratch (stride a_stride)
  int a_stride;          // sum of dims[0..8]
  int z_stride;          // sum of dims[1..8]
  int z_off[NL];         // offset of dZ_l in the per-row dZ scratch
  int n_params;
  int max_dim;
  int max_mat;           // floats of one staged weight matrix buffer (largest layer + alignment slack)
  // AE_Dropout_BN only: BatchNorm affine parameters follow the 8 Linear layers in the flat parameter vector
  int n_linear;          // number of Linear parameters (= n_params for the plain AE)
  int bn_g_off[4], bn_b_off[4];  // gamma / beta of the 4 decoder BatchNorms
  int bn_f_off[4];       // offset of BN layer i in per-feature BN arrays (running stats, xhat cache)
  int bn_f_total;        // sum of the 4 decoder widths
};

struct DwTile { int l, n0, k0; };

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// Weight staging.  A chain is a fixed sequence of passes (8 forward layers on W^T, then 7 backward layers
// 7..1 on W); the matrix of pass p+1 is copied L2 -> shared memory with cp.async while pass p computes, so the
// per-thread weight reads of the inner loops are shared-memory loads instead of exposed L2 latency.
struct WStage {
  float* buf[2];
  int gp, total, per_chain;  // global pass counter, number of passes of this launch, passes per chain (15 or 8)
};

__device__ __forceinline__ void pass_src(const TrainDims& d, const float* params, const float* wt, const int p,
                                         const float*& src, int& n) {
  if (p < NL) { src = wt + d.wt_off[p]; n = d.dims[p] * d.dims[p + 1]; }
  else { const int l = 2 * NL - 1 - p; src = params + d.w_off[l]; n = d.dims[l] * d.dims[l + 1]; }
}

__device__ __forceinline__ void prefetch_pass(const TrainDims& d, const float* params, const float* wt, const int p, float* buf) {
  const float* src; int n;
  pass_src(d, params, wt, p, src, n);
  const float* a = reinterpret_cast<const float*>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)15);
  const int n_chunk = ((int)(src - a) + n + 3) >> 2;  // 16-byte chunks from the aligned address below the matrix
  // every CTA copies the same matrix at the same time: start each CTA at a different offset so the requests
  // spread over the L2 slices instead of all SMs hammering one line after the other in lock-step
  const int rot = (int)(((long long)blockIdx.x * n_chunk) / gridDim.x);
  for (int i = threadIdx.x; i < n_chunk; i += NT_FB) {
    int c = i + rot;
    c = (c >= n_chunk ? c - n_chunk : c) << 2;
    cp_async16(smem_u32(buf + c), a + c);
  }
}

// start the copy of the next pass, wait for the current one; returns the shared-memory address of its matrix
__device__ __forceinline__ const float* acquire_pass(const TrainDims& d, const float* params, const float* wt, WStage& ws) {
  const int cur = ws.gp;
  if (cur + 1 < ws.total) prefetch_pass(d, params, wt, (cur + 1) % ws.per_chain, ws.buf[(cur + 1) & 1]);
  cp_async_commit();
  cp_async_wait_1();
  __syncthreads();
  const float* src; int n;
  pass_src(d, params, wt, cur % ws.per_chain, src, n);
  ws.gp = cur + 1;
  return ws.buf[cur & 1] + ((reinterpret_cast<uintptr_t>(src) & 15) >> 2);
}

__device__ __forceinline__ float act_fwd(float v, int act) {
  if (act == BB_ACT_LEAKY) return v > 0.f ? v : BB_LEAKY * v;
  if (act == BB_ACT_RELU) return fmaxf(v, 0.f);
  return v;
}

__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds_v4(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
// o -> (o / n, o % n) without a division per element: q = mulhi(o, ceil(2^32 / n)), exact for o * n < 2^32
struct FastDiv {
  unsigned n, magic;
  __device__ explicit FastDiv(int n_) : n((unsigned)n_), magic(n_ > 1 ? 0xFFFFFFFFu / (unsigned)n_ + 1u : 0u) {}
  __device__ __forceinline__ void divmod(int o, int& q, int& r) const {
    q = n > 1 ? (int)__umulhi((unsigned)o, magic) : o;
    r = o - q * (int)n;
  }
};

// acc[r] = sum_{i in [i0, i1)} in_s[i][r] * Wm[i * Dout + j]   (RT rows r); both operands in shared memory, addressed
// with 32-bit shared-window addresses (generic pointers cost 64-bit address arithmetic on every load)
__device__ __forceinline__ void gemv8_slice(const float* __restrict__ in_s, const float* __restrict__ Wm, const int Dout,
                                            const int j, const int i0, const int i1, float (&acc)[RT]) {
#pragma unroll
  for (int r = 0; r < RT; ++r) acc[r] = 0.f;
  uint32_t w = smem_u32(Wm) + (uint32_t)(i0 * Dout + j) * 4u;
  uint32_t a = smem_u32(in_s) + (uint32_t)(i0 * RT) * 4u;
  const uint32_t wstep = (uint32_t)Dout * 4u;
#pragma unroll 4
  for (int i = i0; i < i1; ++i) {
    const float wv = lds_f32(w);
#pragma unroll
    for (int q = 0; q < RT / 4; ++q) {
      const float4 a4 = lds_v4(a + 16u * q);
      acc[4 * q + 0] = fmaf(a4.x, wv, acc[4 * q + 0]); acc[4 * q + 1] = fmaf(a4.y, wv, acc[4 * q + 1]);
      acc[4 * q + 2] = fmaf(a4.z, wv, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(a4.w, wv, acc[4 * q + 3]);
    }
    w += wstep;
    a += RT * 4u;
  }
}

// red_s[kp][r][j] = partial sums of out[r][j] = sum_i in_s[i][r] * Wm[i * Dout + j]; narrow outputs split the
// reduction over KP thread groups (combined later in fixed order by red_sum).  Ends with __syncthreads.
__device__ __forceinline__ int gemv8(const float* __restrict__ in_s, const float* __restrict__ Wm, const int Din,
                                     const int Dout, float* __restrict__ red_s) {
  int KP = NT_FB / Dout;
  KP = KP < 1 ? 1 : (KP > 16 ? 16 : KP);
  float acc[RT];
  if (KP == 1) {
    for (int j = threadIdx.x; j < Dout; j += NT_FB) {
      gemv8_slice(in_s, Wm, Dout, j, 0, Din, acc);
#pragma unroll
      for (int r = 0; r < RT; ++r) red_s[r * Dout + j] = acc[r];
    }
  } else if (threadIdx.x < KP * Dout) {
    const int per = (Din + KP - 1) / KP;
    int kp, j;
    FastDiv(Dout).divmod((int)threadIdx.x, kp, j);
    const int i0 = min(Din, kp * per), i1 = min(Din, i0 + per);
    gemv8_slice(in_s, Wm, Dout, j, i0, i1, acc);
#pragma unroll
    for (int r = 0; r < RT; ++r) red_s[(kp * RT + r) * Dout + j] = acc[r];
  }
  __syncthreads();
  return KP;
}

__device__ __forceinline__ float red_sum(const float* red_s, int KP, int Dout, int r, int j) {
  float s = red_s[r * Dout + j];
  for (int kp = 1; kp < KP; ++kp) s += red_s[(kp * RT + r) * Dout + j];
  return s;
}

// One chain (model chain: activations from d.act; L1 chain: ReLU everywhere) forward + backward for RT rows.
//   chain 0: loss term sum((recon - x)^2) / C, seed gradient 2 (recon - x) / C
//   chain 1: loss term reg * sum_l mean|v_l|,  gradient reg / (B * N_l) injected at every layer output
template <int CHAIN>
__device__ void run_chain(const TrainDims& d, const float* __restrict__ params, const float* __restrict__ wt,
                          float* __restrict__ act_g, float* __restrict__ dz_g, const int row0, const int rows,
                          const bool backward, const float reg, const float inv_rows, float* act_s, float* dz_s0,
                          float* dz_s1, float* red_s, float& loss_local, WStage& ws) {
  // ---- forward: act_s[a_off[l]*RT + j*RT + r]
  for (int l = 0; l < NL; ++l) {
    const int K = d.dims[l], N = d.dims[l + 1];
    const float* in_s = act_s + d.a_off[l] * RT;
    float* out_s = act_s + d.a_off[l + 1] * RT;
    const int KP = gemv8(in_s, acquire_pass(d, params, wt, ws), K, N, red_s);
    const float* bias = params + d.b_off[l];
    const int act = CHAIN == 0 ? d.act[l] : BB_ACT_RELU;
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      int r, j;
      FastDiv(N).divmod(o, r, j);
      const float v = act_fwd(red_sum(red_s, KP, N, r, j) + __ldg(bias + j), act);
      out_s[j * RT + r] = v;
      if (r < rows && l + 1 < NL) act_g[(size_t)(row0 + r) * d.a_stride + d.a_off[l + 1] + j] = v;
      if (CHAIN == 1 && r < rows) loss_local += reg * inv_rows / N * fabsf(v);
    }
    __syncthreads();
  }
  // ---- seed gradient at the output
  const int F = d.dims[NL];
  float* dz_cur = dz_s0;
  float* dz_nxt = dz_s1;
  {
    const float* out_s = act_s + d.a_off[NL] * RT;
    const float* x_s = act_s;  // a_off[0] == 0
    for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
      int r, j;
      FastDiv(F).divmod(o, r, j);
      float g = 0.f;
      if (r < rows) {
        if (CHAIN == 0) {
          const float diff = out_s[j * RT + r] - x_s[j * RT + r];
          loss_local += diff * diff / F;
          g = 2.f * diff / F;
        } else {
          g = out_s[j * RT + r] > 0.f ? reg * inv_rows / F : 0.f;
        }
        if (backward) dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[NL - 1] + j] = g;
      }
      dz_cur[j * RT + r] = g;
    }
    __syncthreads();
  }
  if (!backward) return;
  // ---- backward: dZ_{l-1} = (dZ_l W_l [+ l1 seed]) * act'(A_l)
  for (int l = NL - 1; l >= 1; --l) {
    const int K = d.dims[l], N = d.dims[l + 1];
    const int KP = gemv8(dz_cur, acquire_pass(d, params, wt, ws), N, K, red_s);
    const float* a_s = act_s + d.a_off[l] * RT;  // output of layer l-1 (post-activation)
    const int act = CHAIN == 0 ? d.act[l - 1] : BB_ACT_RELU;
    const float seed = CHAIN == 1 ? reg * inv_rows / K : 0.f;
    for (int o = threadIdx.x; o < RT * K; o += NT_FB) {
      int r, j;
      FastDiv(K).divmod(o, r, j);
      float g = red_sum(red_s, KP, K, r, j) + seed;
      const float a = a_s[j * RT + r];
      if (act == BB_ACT_LEAKY) g *= (a > 0.f ? 1.f : BB_LEAKY);
      else if (act == BB_ACT_RELU) g = a > 0.f ? g : 0.f;
      if (r >= rows) g = 0.f;
      dz_nxt[j * RT + r] = g;
      if (r < rows) dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[l - 1] + j] = g;
    }
    __syncthreads();
    float* t = dz_cur; dz_cur = dz_nxt; dz_nxt = t;
  }
}

// scratch layout per chain c: act_g + c * B_max * a_stride ; dz_g + c * B_max * z_stride
__global__ void __launch_bounds__(NT_FB)
train_fwd_bwd_kernel(const __grid_constant__ TrainDims d, const float* __restrict__ params,
                     const float* __restrict__ wt, const float* __restrict__ x, const int batch_rows,
                     float* __restrict__ act_g, float* __restrict__ dz_g, const size_t chain_act_stride,
                     const size_t chain_dz_stride, const int backward, const int l1, const float reg,
                     const float inv_global_rows, float* __restrict__ loss_part) {
  extern __shared__ __align__(16) float smem[];
  pdl_launch_dependents();
  pdl_wait();  // parameters come from the previous step's Adam kernel
  float* act_s = smem;                           // a_stride * RT
  float* dz_s0 = act_s + d.a_stride * RT;        // max_dim * RT
  float* dz_s1 = dz_s0 + d.max_dim * RT;
  float* red_s = dz_s1 + d.max_dim * RT;         // max(max_dim, NT_FB) * RT
  __shared__ float warp_loss[NT_FB / 32];
  WStage ws;
  ws.buf[0] = red_s + (d.max_dim > NT_FB ? d.max_dim : NT_FB) * RT;
  ws.buf[1] = ws.buf[0] + d.max_mat;
  ws.per_chain = backward ? 2 * NL - 1 : NL;
  ws.total = ws.per_chain * (l1 ? 2 : 1);
  ws.gp = 0;
  prefetch_pass(d, params, wt, 0, ws.buf[0]);
  cp_async_commit();

  const int row0 = blockIdx.x * RT;
  const int rows = min(RT, batch_rows - row0);
  const int F = d.dims[0];
  for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
    int r, j;
    FastDiv(F).divmod(o, r, j);
    const float v = r < rows ? __ldg(x + (size_t)(row0 + r) * F + j) : 0.f;
    act_s[j * RT + r] = v;
    if (r < rows) act_g[(size_t)(row0 + r) * d.a_stride + j] = v;  // A_0 copy keeps the dW kernel uniform
  }
  __syncthreads();
  float loss_local = 0.f;
  run_chain<0>(d, params, wt, act_g, dz_g, row0, rows, backward != 0, 0.f, 0.f, act_s, dz_s0, dz_s1, red_s, loss_local, ws);
  if (l1) {
    __syncthreads();
    for (int o = threadIdx.x; o < RT * F; o += NT_FB) {  // A_0 of the second chain is x as well
      const int r = o / F, j = o - r * F;
      if (r < rows) act_g[chain_act_stride + (size_t)(row0 + r) * d.a_stride + j] = act_s[j * RT + r];
    }
    run_chain<1>(d, params, wt, act_g + chain_act_stride, dz_g + chain_dz_stride, row0, rows, backward != 0, reg,
                 inv_global_rows, act_s, dz_s0, dz_s1, red_s, loss_local, ws);
  }
  // block-reduce the loss partial in a fixed order
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) loss_local += __shfl_xor_sync(0xffffffffu, loss_local, off);
  if ((threadIdx.x & 31) == 0) warp_loss[threadIdx.x >> 5] = loss_local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < NT_FB / 32; ++w) s += warp_loss[w];
    loss_part[blockIdx.x] = s;
  }
}

// ------------------------------------------------------------------------------------------------ AE_Dropout_BN
// reference baler/modules/models.py:256-313 in train mode:
//   encoder 4 x (Linear -> Dropout(p = .5,.4,.3,.2) -> LeakyReLU)   [activation also on the latent]
//   decoder 3 x (Linear -> LeakyReLU -> BatchNorm1d) + Linear -> BatchNorm1d -> ReLU
// BatchNorm in train mode uses the statistics of the WHOLE batch (biased variance, eps 1e-5) and updates the
// running statistics with momentum 0.1 and the unbiased variance.  The batch is spread over CTAs (4 rows each), so
// the kernel is launched cooperatively and meets at a grid-wide barrier at each of the 4 BatchNorms in the forward
// and in the backward pass; per-CTA partial sums are combined in a fixed order (reproducible).
struct DbnArgs {
  const float* x;
  int batch_rows;
  int mode;                   // 0: train forward + backward, 1: eval forward (no dropout, running statistics), loss only
  float* act_g;
  float* dz_g;
  float* loss_part;
  float* bn_part;             // [8 barriers][gridDim.x][2 * max_dim] partial sums
  float* rm;                  // running mean / var, bn_f_total floats each
  float* rv;
  long long* nbt;             // num_batches_tracked[4]
  float* bn_grad;             // split 0 of the gradient partial buffer (BN gamma / beta gradients land there)
  const unsigned char* mask[4];  // injected dropout keep-masks [batch][N_l] (parity tests) or nullptr (Philox)
  unsigned long long seed, step;
};

__device__ __forceinline__ bool dropout_keep(const DbnArgs& a, const int l, const int grow, const int j, const int N) {
  if (a.mask[l] != nullptr) return a.mask[l][(size_t)grow * N + j] != 0;
  return bb_philox_keep(a.seed, a.step, l, grow, j);
}

__global__ void __launch_bounds__(NT_FB)
train_dbn_kernel(const __grid_constant__ TrainDims d, const float* __restrict__ params, const float* __restrict__ wt,
                 const __grid_constant__ DbnArgs a) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) float smem[];
  float* act_s = smem;                             // a_stride * RT : layer inputs A_0..A_7 and the reconstruction
  float* dz_s0 = act_s + d.a_stride * RT;
  float* dz_s1 = dz_s0 + d.max_dim * RT;
  float* red_s = dz_s1 + d.max_dim * RT;
  float* xhat_s = red_s + (d.max_dim > NT_FB ? d.max_dim : NT_FB) * RT;  // bn_f_total * RT : normalised BN inputs
  float* u_s = xhat_s + d.bn_f_total * RT;                               // bn_f_total * RT : BN inputs (sign for LeakyReLU')
  float* inv_s = u_s + d.bn_f_total * RT;                                // bn_f_total : 1 / sqrt(var + eps)
  float* tot_s = inv_s + ((d.bn_f_total + 3) & ~3);                      // 2 * max_dim : batch sums (16-byte aligned)
  __shared__ float warp_loss[NT_FB / 32];
  WStage ws;
  ws.buf[0] = tot_s + 2 * d.max_dim;
  ws.buf[1] = ws.buf[0] + d.max_mat;
  const bool train = a.mode == 0;
  ws.per_chain = train ? 2 * NL - 1 : NL;
  ws.total = ws.per_chain;
  ws.gp = 0;
  prefetch_pass(d, params, wt, 0, ws.buf[0]);
  cp_async_commit();

  const int B = a.batch_rows;
  const int row0 = blockIdx.x * RT;
  const int rows = max(0, min(RT, B - row0));
  const int F = d.dims[0];
  const float keep_scale[4] = {1.f / 0.5f, 1.f / 0.6f, 1.f / 0.7f, 1.f / 0.8f};
  for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
    int r, j;
    FastDiv(F).divmod(o, r, j);
    const float v = r < rows ? __ldg(a.x + (size_t)(row0 + r) * F + j) : 0.f;
    act_s[j * RT + r] = v;
    if (r < rows) a.act_g[(size_t)(row0 + r) * d.a_stride + j] = v;
  }
  __syncthreads();

  // ---------------- forward: encoder
  for (int l = 0; l < 4; ++l) {
    const int K = d.dims[l], N = d.dims[l + 1];
    const int KP = gemv8(act_s + d.a_off[l] * RT, acquire_pass(d, params, wt, ws), K, N, red_s);
    const float* bias = params + d.b_off[l];
    float* out_s = act_s + d.a_off[l + 1] * RT;
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      int r, j;
      FastDiv(N).divmod(o, r, j);
      float v = red_sum(red_s, KP, N, r, j) + __ldg(bias + j);
      if (train && r < rows) v = dropout_keep(a, l, row0 + r, j, N) ? v * keep_scale[l] : 0.f;
      v = act_fwd(v, BB_ACT_LEAKY);
      out_s[j * RT + r] = v;
      if (r < rows) a.act_g[(size_t)(row0 + r) * d.a_stride + d.a_off[l + 1] + j] = v;
    }
    __syncthreads();
  }
  // ---------------- forward: decoder with BatchNorm
  const int n_cta = gridDim.x;
  for (int i = 0; i < 4; ++i) {
    const int l = 4 + i, K = d.dims[l], N = d.dims[l + 1], fo = d.bn_f_off[i];
    const int KP = gemv8(act_s + d.a_off[l] * RT, acquire_pass(d, params, wt, ws), K, N, red_s);
    const float* bias = params + d.b_off[l];
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      int r, j;
      FastDiv(N).divmod(o, r, j);
      float v = red_sum(red_s, KP, N, r, j) + __ldg(bias + j);
      if (i < 3) v = act_fwd(v, BB_ACT_LEAKY);
      u_s[(fo + j) * RT + r] = r < rows ? v : 0.f;
    }
    __syncthreads();
    const float* gam = params + d.bn_g_off[i];
    const float* bet = params + d.bn_b_off[i];
    if (train) {
      float* part = a.bn_part + ((size_t)i * n_cta + blockIdx.x) * 2 * d.max_dim;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int r = 0; r < RT; ++r) { const float u = u_s[(fo + j) * RT + r]; s1 += u; s2 = fmaf(u, u, s2); }
        part[j] = s1; part[N + j] = s2;
      }
      __threadfence();
      grid.sync();
      const float* all = a.bn_part + (size_t)i * n_cta * 2 * d.max_dim;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        double S1 = 0.0, S2 = 0.0;
        for (int c = 0; c < n_cta; ++c) { S1 += (double)__ldcg(all + (size_t)c * 2 * d.max_dim + j); S2 += (double)__ldcg(all + (size_t)c * 2 * d.max_dim + N + j); }
        const double mean = S1 / B;
        double var = S2 / B - mean * mean;  // biased batch variance
        var = var > 0.0 ? var : 0.0;
        tot_s[j] = (float)mean;
        inv_s[fo + j] = (float)(1.0 / sqrt(var + 1e-5));
        if (blockIdx.x == 0) {  // running statistics: momentum 0.1, unbiased variance
          a.rm[fo + j] = 0.9f * a.rm[fo + j] + 0.1f * (float)mean;
          a.rv[fo + j] = 0.9f * a.rv[fo + j] + 0.1f * (float)(var * B / (B > 1 ? B - 1 : 1));
          if (j == 0) a.nbt[i] += 1;
        }
      }
    } else {
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        tot_s[j] = a.rm[fo + j];
        inv_s[fo + j] = rsqrtf(a.rv[fo + j] + 1e-5f);
      }
    }
    __syncthreads();
    float* out_s = act_s + d.a_off[l + 1] * RT;
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      int r, j;
      FastDiv(N).divmod(o, r, j);
      const float xh = (u_s[(fo + j) * RT + r] - tot_s[j]) * inv_s[fo + j];
      float h = fmaf(xh, __ldg(gam + j), __ldg(bet + j));
      if (i == 3) h = fmaxf(h, 0.f);
      xhat_s[(fo + j) * RT + r] = xh;
      out_s[j * RT + r] = h;
      if (r < rows && l + 1 < NL) a.act_g[(size_t)(row0 + r) * d.a_stride + d.a_off[l + 1] + j] = h;
    }
    __syncthreads();
  }
  // ---------------- loss and the seed gradient
  float loss_local = 0.f;
  float* dz_cur = dz_s0;
  float* dz_nxt = dz_s1;
  {
    const float* out_s = act_s + d.a_off[NL] * RT;
    for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
      int r, j;
      FastDiv(F).divmod(o, r, j);
      float g = 0.f;
      if (r < rows) {
        const float rec = out_s[j * RT + r];
        const float diff = rec - act_s[j * RT + r];
        loss_local += diff * diff / F;
        g = rec > 0.f ? 2.f * diff / F : 0.f;  // through the final ReLU
      }
      dz_cur[j * RT + r] = g;
    }
    __syncthreads();
  }
  if (train) {
    // ---------------- backward: decoder
    for (int i = 3; i >= 0; --i) {
      const int l = 4 + i, K = d.dims[l], N = d.dims[l + 1], fo = d.bn_f_off[i];
      float* part = a.bn_part + ((size_t)(4 + 3 - i) * n_cta + blockIdx.x) * 2 * d.max_dim;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        float t1 = 0.f, t2 = 0.f;
#pragma unroll
        for (int r = 0; r < RT; ++r) { const float g = dz_cur[j * RT + r]; t1 += g; t2 = fmaf(g, xhat_s[(fo + j) * RT + r], t2); }
        part[j] = t1; part[N + j] = t2;
      }
      __threadfence();
      grid.sync();
      const float* all = a.bn_part + (size_t)(4 + 3 - i) * n_cta * 2 * d.max_dim;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        double T1 = 0.0, T2 = 0.0;
        for (int c = 0; c < n_cta; ++c) { T1 += (double)__ldcg(all + (size_t)c * 2 * d.max_dim + j); T2 += (double)__ldcg(all + (size_t)c * 2 * d.max_dim + N + j); }
        tot_s[j] = (float)T1; tot_s[d.max_dim + j] = (float)T2;
        if (blockIdx.x == 0) { a.bn_grad[d.bn_b_off[i] + j] = (float)T1; a.bn_grad[d.bn_g_off[i] + j] = (float)T2; }
      }
      __syncthreads();
      const float* gam = params + d.bn_g_off[i];
      const float invB = 1.f / B;
      for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
        int r, j;
        FastDiv(N).divmod(o, r, j);
        const float g = __ldg(gam + j);
        // dx = inv / B * (B dxh - sum(dxh) - xhat sum(dxh xhat)), dxh = dy * gamma
        float dx = inv_s[fo + j] * g * (dz_cur[j * RT + r] - invB * tot_s[j] - xhat_s[(fo + j) * RT + r] * invB * tot_s[d.max_dim + j]);
        if (i < 3) dx *= u_s[(fo + j) * RT + r] > 0.f ? 1.f : BB_LEAKY;
        if (r >= rows) dx = 0.f;
        dz_nxt[j * RT + r] = dx;
        if (r < rows) a.dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[l] + j] = dx;
      }
      __syncthreads();
      {  // dX = dZ W_l  (gradient w.r.t. the input of Linear l = output of the previous block)
        const int KP = gemv8(dz_nxt, acquire_pass(d, params, wt, ws), N, K, red_s);
        for (int o = threadIdx.x; o < RT * K; o += NT_FB) {
          int r, j;
          FastDiv(K).divmod(o, r, j);
          dz_cur[j * RT + r] = red_sum(red_s, KP, K, r, j);
        }
        __syncthreads();
      }
    }
    // ---------------- backward: encoder (dz_cur = gradient w.r.t. the output of encoder layer l)
    for (int l = 3; l >= 0; --l) {
      const int K = d.dims[l], N = d.dims[l + 1];
      const float* a_out = act_s + d.a_off[l + 1] * RT;
      for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
        int r, j;
        FastDiv(N).divmod(o, r, j);
        float g = 0.f;
        if (r < rows) {
          g = dz_cur[j * RT + r] * (a_out[j * RT + r] > 0.f ? 1.f : BB_LEAKY);
          g = dropout_keep(a, l, row0 + r, j, N) ? g * keep_scale[l] : 0.f;
          a.dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[l] + j] = g;
        }
        dz_nxt[j * RT + r] = g;
      }
      __syncthreads();
      if (l >= 1) {
        const int KP = gemv8(dz_nxt, acquire_pass(d, params, wt, ws), N, K, red_s);
        for (int o = threadIdx.x; o < RT * K; o += NT_FB) {
          int r, j;
          FastDiv(K).divmod(o, r, j);
          dz_cur[j * RT + r] = red_sum(red_s, KP, K, r, j);
        }
        __syncthreads();
      }
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) loss_local += __shfl_xor_sync(0xffffffffu, loss_local, off);
  if ((threadIdx.x & 31) == 0) warp_loss[threadIdx.x >> 5] = loss_local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < NT_FB / 32; ++w) s += warp_loss[w];
    a.loss_part[blockIdx.x] = s;
  }
}

// partial[split][w_off[l] + n*K + k] = sum_{r in split} dZ_l[r][n] * A_l[r][k]   (+ second chain)
__global__ void __launch_bounds__(NT)
train_dw_kernel(const __grid_constant__ TrainDims d, const DwTile* __restrict__ tiles, const float* __restrict__ act_g,
                const float* __restrict__ dz_g, const size_t chain_act_stride, const size_t chain_dz_stride,
                const int n_chains, const int batch_rows, float* __restrict__ partial) {
  __shared__ __align__(16) float dz_s[DW_T][DW_LD];
  __shared__ __align__(16) float a_s[DW_T][DW_LD];
  pdl_launch_dependents();
  pdl_wait();  // activations and dZ come from the forward / backward kernel
  const DwTile tile = tiles[blockIdx.x];
  const int l = tile.l, N = d.dims[l + 1], K = d.dims[l];
  const int r0 = blockIdx.y * DW_T;
  const int rows = min(DW_T, batch_rows - r0);
  const int tn = threadIdx.x >> 4, tk = threadIdx.x & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bsum = 0.f;
  for (int c = 0; c < n_chains; ++c) {
    const float* dz = dz_g + c * chain_dz_stride + d.z_off[l];
    const float* a = act_g + c * chain_act_stride + d.a_off[l];
    if (c) __syncthreads();
    for (int e = threadIdx.x; e < DW_T * DW_T; e += NT) {
      const int rr = e >> 6, cc = e & 63;
      const bool rv = rr < rows;
      dz_s[rr][cc] = (rv && tile.n0 + cc < N) ? __ldg(dz + (size_t)(r0 + rr) * d.z_stride + tile.n0 + cc) : 0.f;
      a_s[rr][cc] = (rv && tile.k0 + cc < K) ? __ldg(a + (size_t)(r0 + rr) * d.a_stride + tile.k0 + cc) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < DW_T; ++rr) {
      const float4 dv = *reinterpret_cast<const float4*>(&dz_s[rr][tn * 4]);
      const float4 av = *reinterpret_cast<const float4*>(&a_s[rr][tk * 4]);
      const float dd[4] = {dv.x, dv.y, dv.z, dv.w}, aa[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dd[i], aa[j], acc[i][j]);
    }
    if (tile.k0 == 0 && threadIdx.x < DW_T)
      for (int rr = 0; rr < DW_T; ++rr) bsum += dz_s[rr][threadIdx.x];
  }
  float* out = partial + (size_t)blockIdx.y * d.n_params;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = tile.n0 + tn * 4 + i;
    if (n >= N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = tile.k0 + tk * 4 + j;
      if (k < K) out[d.w_off[l] + n * K + k] = acc[i][j];
    }
  }
  if (tile.k0 == 0 && threadIdx.x < DW_T && tile.n0 + threadIdx.x < N) out[d.b_off[l] + tile.n0 + threadIdx.x] = bsum;
}

// mode 0: grads = sum of partials, then Adam.  mode 1: grads = sum of partials only (+ loss slot).
// mode 2: Adam from grads (after the caller's all-reduce).
__global__ void __launch_bounds__(NT)
train_adam_kernel(const int n_params, const int mode, const float* __restrict__ partial, const int n_splits,
                  float* __restrict__ grads, float* __restrict__ params, float* __restrict__ wt,
                  const int* __restrict__ wt_index, float* __restrict__ m, float* __restrict__ v, const float lr_bc1,
                  const float inv_sqrt_bc2, const float beta1, const float beta2, const float eps,
                  const float* __restrict__ loss_part, const int n_loss_parts, double* __restrict__ loss_accum) {
  pdl_launch_dependents();
  pdl_wait();  // gradient partials come from the dW kernel
  const int p = blockIdx.x * NT + threadIdx.x;
  if (p < n_params) {
    float g;
    if (mode == 2) {
      g = grads[p];
    } else {
      g = 0.f;
      for (int s = 0; s < n_splits; ++s) g += __ldg(partial + (size_t)s * n_params + p);
      grads[p] = g;
    }
    if (mode != 1) {
      const float mm = m[p] + (g - m[p]) * (1.f - beta1);      // exp_avg.lerp_(g, 1 - beta1)
      const float vv = beta2 * v[p] + (1.f - beta2) * g * g;   // exp_avg_sq.mul_(b2).addcmul_(g, g, 1 - b2)
      m[p] = mm;
      v[p] = vv;
      const float denom = sqrtf(vv) * inv_sqrt_bc2 + eps;
      const float np = params[p] - lr_bc1 * (mm / denom);
      params[p] = np;
      const int wi = wt_index[p];
      if (wi >= 0) wt[wi] = np;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (mode != 2) {
      float s = 0.f;
      for (int i = 0; i < n_loss_parts; ++i) s += loss_part[i];
      grads[n_params] = s;  // loss rides in the last slot so one all-reduce covers it
    }
    if (mode != 1 && loss_accum) *loss_accum += (double)grads[n_params];
  }
}

}  // namespace

struct bb_trainer {
  bb_ctx* ctx = nullptr;
  TrainDims d;
  int max_batch = 0, n_tiles = 0, wt_floats = 0;
  long long step = 0;
  int last_rows = 0;  // rows of the most recent forward pass (activation extraction)
  float *params = nullptr, *wt = nullptr, *grads = nullptr, *m = nullptr, *v = nullptr;
  float *act_g = nullptr, *dz_g = nullptr, *partial = nullptr, *loss_part = nullptr;
  int* wt_index = nullptr;
  DwTile* tiles = nullptr;
  double* loss_accum = nullptr;  // internal accumulator used by bb_trainer_epoch / validate
  size_t smem_bytes = 0;
  // AE_Dropout_BN
  int kind = 0;                  // 0: AE / CFD_dense_AE, 1: AE_Dropout_BN
  float *bn_part = nullptr, *rm = nullptr, *rv = nullptr;
  long long* nbt = nullptr;
  const unsigned char* mask_dev[4] = {nullptr, nullptr, nullptr, nullptr};
  unsigned long long seed = 0;
  size_t dbn_smem = 0;
  int dbn_max_ctas = 0;
  // tensor-core path (bb_train_tc.cu): the default for the plain AE with the MSE loss.  Both paths share params / m / v /
  // grads; each keeps derived weight copies (fp32 transposed `wt` here, packed fp16 images there) that go stale when the
  // other one moves the parameters and are rebuilt on the next switch.
  TcTrainer* tc = nullptr;
  int precision = BB_PREC_AUTO;      // BB_PREC_FP32 forces the fp32 kernels
  bool wt_fresh = true, tc_fresh = true;
  bool last_tc = false;              // which path ran the most recent forward pass (activation extraction)
  // float64 path (bb_train_f64.cu, BB_PREC_FP64): its own float64 master parameters, Adam state and scratch, made by
  // bb_trainer_set_precision from the float64 weights bb_trainer_create received (kept here until then)
  F64Trainer* f64 = nullptr;
  std::vector<double> params_host;
  std::vector<double> bn_stats_host;  // AE_Dropout_BN: float64 running_mean then running_var (bn_f_total each)
  long long nbt_host[4] = {0, 0, 0, 0};
  bool started = false;              // a step or an epoch has run (the precision of a float64 run is fixed from then on)
  HostWindow* win = nullptr;         // device window of bb_trainer_epoch_host / _validate_host (kept between calls)
};

namespace {

int launch_fwd_bwd(bb_trainer* t, const float* x, int rows, int backward, const bb_train_hyper* h, cudaStream_t s) {
  const int grid = (rows + RT - 1) / RT;
  t->last_rows = rows;
  const int world = h && h->world_size > 0 ? h->world_size : 1;
  const float inv_rows = 1.f / ((float)rows * world);
  return (int)pdl_launch(train_fwd_bwd_kernel, dim3(grid), dim3(NT_FB), t->smem_bytes, s, t->d, t->params, t->wt, x, rows, t->act_g,
                         t->dz_g, (size_t)t->max_batch * t->d.a_stride, (size_t)t->max_batch * t->d.z_stride, backward,
                         h ? h->l1 : 0, h ? (float)h->reg_param : 0.f, inv_rows, t->loss_part);
}

int launch_dbn(bb_trainer* t, const float* x, int rows, int mode, cudaStream_t s) {
  const int grid = (rows + RT - 1) / RT;
  if (grid > t->dbn_max_ctas) return BB_ERR_UNSUPPORTED;  // cooperative launch: every CTA must be resident
  t->last_rows = rows;
  DbnArgs a;
  a.x = x; a.batch_rows = rows; a.mode = mode;
  a.act_g = t->act_g; a.dz_g = t->dz_g; a.loss_part = t->loss_part; a.bn_part = t->bn_part;
  a.rm = t->rm; a.rv = t->rv; a.nbt = t->nbt; a.bn_grad = t->partial;
  for (int i = 0; i < 4; ++i) a.mask[i] = t->mask_dev[i];
  a.seed = t->seed; a.step = (unsigned long long)t->step;
  void* args[] = {(void*)&t->d, (void*)&t->params, (void*)&t->wt, (void*)&a};
  return (int)cudaLaunchCooperativeKernel((const void*)train_dbn_kernel, dim3(grid), dim3(NT_FB), args, t->dbn_smem, s);
}

int create_common(bb_ctx* ctx, int n_features, int z_dim, const double* const* weights_host, const double* const* biases_host,
                  int max_batch, int kind, const double* const* bn_gamma, const double* const* bn_beta,
                  const double* const* bn_mean, const double* const* bn_var, const long long* bn_nbt, bb_trainer** out);

__global__ void __launch_bounds__(NT) refresh_wt_kernel(const int n_params, const float* __restrict__ params,
                                                        const int* __restrict__ wt_index, float* __restrict__ wt) {
  const int p = blockIdx.x * NT + threadIdx.x;
  if (p < n_params && wt_index[p] >= 0) wt[wt_index[p]] = params[p];
}

// which implementation serves this call; rebuilds that path's derived weight copy when the other path moved the parameters
bool use_tc(bb_trainer* t, const bb_train_hyper* h, cudaStream_t s, int* rc) {
  *rc = BB_OK;
  const bool tc = t->tc && t->precision != BB_PREC_FP32 && !(h && h->l1);
  if (tc && !t->tc_fresh) {
    *rc = bb_tc_train_repack(t->tc, s);
    t->tc_fresh = true;
  }
  if (!tc && !t->wt_fresh) {
    refresh_wt_kernel<<<(t->d.n_params + NT - 1) / NT, NT, 0, s>>>(t->d.n_params, t->params, t->wt_index, t->wt);
    *rc = (int)cudaGetLastError();
    t->wt_fresh = true;
  }
  return tc;
}

TcHyper tc_hyper(const bb_train_hyper* h) {
  TcHyper o;
  o.beta1 = (float)h->beta1; o.beta2 = (float)h->beta2; o.eps = (float)h->eps;
  o.lr = h->lr; o.b1d = h->beta1; o.b2d = h->beta2;
  return o;
}

}  // namespace

extern "C" {

int bb_trainer_create(bb_ctx* ctx, int n_features, int z_dim, const double* const* weights_host,
                      const double* const* biases_host, int max_batch, bb_trainer** out) {
  return create_common(ctx, n_features, z_dim, weights_host, biases_host, max_batch, 0, nullptr, nullptr, nullptr, nullptr,
                       nullptr, out);
}

int bb_trainer_create_dbn(bb_ctx* ctx, int n_features, int z_dim, const double* const* weights_host,
                          const double* const* biases_host, const double* const* bn_weight_host,
                          const double* const* bn_bias_host, const double* const* bn_mean_host,
                          const double* const* bn_var_host, const long long* bn_batches_tracked, int max_batch,
                          bb_trainer** out) {
  if (!bn_weight_host || !bn_bias_host || !bn_mean_host || !bn_var_host) return BB_ERR_INVALID;
  return create_common(ctx, n_features, z_dim, weights_host, biases_host, max_batch, 1, bn_weight_host, bn_bias_host,
                       bn_mean_host, bn_var_host, bn_batches_tracked, out);
}

int bb_trainer_set_dropout(bb_trainer* t, unsigned long long seed, const unsigned char* const* masks_dev) {
  if (!t || t->kind != 1) return BB_ERR_INVALID;
  t->seed = seed;
  for (int i = 0; i < 4; ++i) t->mask_dev[i] = masks_dev ? masks_dev[i] : nullptr;
  if (t->f64) {
    const int rc = bb_f64_train_set_dropout(t->f64, seed, masks_dev);
    if (rc != BB_OK) return rc;
  }
  if (t->tc) return bb_tc_train_set_dropout(t->tc, seed, masks_dev);
  return BB_OK;
}

int bb_trainer_set_dropout_mt19937(bb_trainer* t, const uint32_t* key_624, int pos) {
  if (!t || t->kind != 1 || !key_624) return BB_ERR_INVALID;
  if (t->precision != BB_PREC_FP64) return BB_ERR_UNSUPPORTED;
  return bb_f64_train_set_mt19937(t->f64, key_624, pos);
}

int bb_trainer_get_dropout_mt19937(bb_trainer* t, uint32_t* key_out_624, int* pos_out) {
  if (!t || t->kind != 1 || !key_out_624 || !pos_out) return BB_ERR_INVALID;
  if (t->precision != BB_PREC_FP64) return BB_ERR_UNSUPPORTED;
  return bb_f64_train_get_mt19937(t->f64, key_out_624, pos_out);
}

int bb_trainer_bn_running_dev_f64(bb_trainer* t, double** running_mean_dev, double** running_var_dev, int* n) {
  if (!t || t->kind != 1 || !running_mean_dev || !running_var_dev || !n) return BB_ERR_INVALID;
  if (t->precision != BB_PREC_FP64) return BB_ERR_UNSUPPORTED;
  *n = t->d.bn_f_total;
  return bb_f64_train_bn_running(t->f64, running_mean_dev, running_var_dev);
}

int bb_trainer_bn_running_dev(bb_trainer* t, float** running_mean_dev, float** running_var_dev, int* n) {
  if (!t || t->kind != 1 || !running_mean_dev || !running_var_dev || !n) return BB_ERR_INVALID;
  *running_mean_dev = t->rm; *running_var_dev = t->rv; *n = t->d.bn_f_total;
  return BB_OK;
}

int bb_trainer_get_bn(bb_trainer* t, double* const* bn_weight_host, double* const* bn_bias_host,
                      double* const* bn_mean_host, double* const* bn_var_host, long long* bn_batches_tracked) {
  if (!t || t->kind != 1 || !bn_weight_host || !bn_bias_host || !bn_mean_host || !bn_var_host || !bn_batches_tracked)
    return BB_ERR_INVALID;
  if (t->precision == BB_PREC_FP64) {  // the float64 master as it is
    std::vector<double> hp(t->d.n_params), hm(t->d.bn_f_total), hv(t->d.bn_f_total);
    int rc = bb_f64_train_get_params(t->f64, hp.data());
    if (rc == BB_OK) rc = bb_f64_train_get_bn_stats(t->f64, hm.data(), hv.data(), bn_batches_tracked);
    if (rc != BB_OK) return rc;
    for (int i = 0; i < 4; ++i) {
      const int n = t->d.dims[5 + i];
      memcpy(bn_weight_host[i], hp.data() + t->d.bn_g_off[i], sizeof(double) * n);
      memcpy(bn_bias_host[i], hp.data() + t->d.bn_b_off[i], sizeof(double) * n);
      memcpy(bn_mean_host[i], hm.data() + t->d.bn_f_off[i], sizeof(double) * n);
      memcpy(bn_var_host[i], hv.data() + t->d.bn_f_off[i], sizeof(double) * n);
    }
    return BB_OK;
  }
  std::vector<float> hp(t->d.n_params), hm(t->d.bn_f_total), hv(t->d.bn_f_total);
  BB_CUDA(cudaMemcpy(hp.data(), t->params, sizeof(float) * hp.size(), cudaMemcpyDeviceToHost));
  BB_CUDA(cudaMemcpy(hm.data(), t->rm, sizeof(float) * hm.size(), cudaMemcpyDeviceToHost));
  BB_CUDA(cudaMemcpy(hv.data(), t->rv, sizeof(float) * hv.size(), cudaMemcpyDeviceToHost));
  BB_CUDA(cudaMemcpy(bn_batches_tracked, t->nbt, sizeof(long long) * 4, cudaMemcpyDeviceToHost));
  for (int i = 0; i < 4; ++i) {
    const int n = t->d.dims[5 + i];
    for (int j = 0; j < n; ++j) {
      bn_weight_host[i][j] = (double)hp[t->d.bn_g_off[i] + j];
      bn_bias_host[i][j] = (double)hp[t->d.bn_b_off[i] + j];
      bn_mean_host[i][j] = (double)hm[t->d.bn_f_off[i] + j];
      bn_var_host[i][j] = (double)hv[t->d.bn_f_off[i] + j];
    }
  }
  return BB_OK;
}

}  // extern "C"

namespace {
int create_common(bb_ctx* ctx, int n_features, int z_dim, const double* const* weights_host, const double* const* biases_host,
                  int max_batch, int kind, const double* const* bn_gamma, const double* const* bn_beta,
                  const double* const* bn_mean, const double* const* bn_var, const long long* bn_nbt, bb_trainer** out) {
  if (!ctx || !out || n_features < 1 || z_dim < 1 || max_batch < 1 || !weights_host || !biases_host) return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(ctx->device));
  bb_trainer* t = new (std::nothrow) bb_trainer();
  if (!t) return BB_ERR_NOMEM;
  t->ctx = ctx;
  t->max_batch = max_batch;
  TrainDims& d = t->d;
  const int dims[NL + 1] = {n_features, 200, 100, 50, z_dim, 50, 100, 200, n_features};
  const int acts[NL] = {BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_NONE, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_LEAKY, BB_ACT_NONE};
  t->kind = kind;
  int p = 0, wtp = 0, a = 0, z = 0, mx = 0;
  for (int l = 0; l <= NL; ++l) {
    d.dims[l] = dims[l];
    d.a_off[l] = a;
    a += dims[l];
    mx = dims[l] > mx ? dims[l] : mx;
  }
  for (int l = 0; l < NL; ++l) {
    d.act[l] = acts[l];
    d.w_off[l] = p; p += dims[l] * dims[l + 1];
    d.b_off[l] = p; p += dims[l + 1];
    d.wt_off[l] = wtp; wtp += dims[l] * dims[l + 1];
    d.z_off[l] = z; z += dims[l + 1];
  }
  d.n_linear = p;
  d.bn_f_total = 0;
  for (int i = 0; i < 4; ++i) {
    d.bn_f_off[i] = d.bn_f_total;
    d.bn_g_off[i] = d.bn_b_off[i] = 0;
    if (kind == 1) {
      d.bn_g_off[i] = p; p += dims[5 + i];
      d.bn_b_off[i] = p; p += dims[5 + i];
    }
    d.bn_f_total += dims[5 + i];
  }
  d.a_stride = a; d.z_stride = z; d.n_params = p; d.max_dim = mx;
  int mm = 0;
  for (int l = 0; l < NL; ++l) mm = dims[l] * dims[l + 1] > mm ? dims[l] * dims[l + 1] : mm;
  d.max_mat = (mm + 8 + 3) & ~3;
  t->wt_floats = wtp;
  t->smem_bytes = ((size_t)(d.a_stride + 2 * mx + (mx > NT_FB ? mx : NT_FB)) * RT + 2 * (size_t)d.max_mat) * sizeof(float);
  if (t->smem_bytes > ctx->smem_optin) { delete t; return BB_ERR_UNSUPPORTED; }

  std::vector<float> hp(p, 0.f), hwt(wtp);
  std::vector<int> hidx(p, -1);
  std::vector<DwTile> tiles;
  for (int l = 0; l < NL; ++l) {
    const int K = dims[l], N = dims[l + 1];
    if (!weights_host[l] || !biases_host[l]) { delete t; return BB_ERR_INVALID; }
    for (int n = 0; n < N; ++n) {
      for (int k = 0; k < K; ++k) {
        const float w = (float)weights_host[l][(size_t)n * K + k];
        hp[d.w_off[l] + n * K + k] = w;
        hwt[d.wt_off[l] + k * N + n] = w;
        hidx[d.w_off[l] + n * K + k] = d.wt_off[l] + k * N + n;
      }
      hp[d.b_off[l] + n] = (float)biases_host[l][n];
    }
    for (int n0 = 0; n0 < N; n0 += DW_T)
      for (int k0 = 0; k0 < K; k0 += DW_T) tiles.push_back({l, n0, k0});
  }
  std::vector<float> hrm(d.bn_f_total, 0.f), hrv(d.bn_f_total, 1.f);
  long long hnbt[4] = {0, 0, 0, 0};
  if (kind == 1) {
    for (int i = 0; i < 4; ++i) {
      if (!bn_gamma[i] || !bn_beta[i] || !bn_mean[i] || !bn_var[i]) { delete t; return BB_ERR_INVALID; }
      for (int j = 0; j < dims[5 + i]; ++j) {
        hp[d.bn_g_off[i] + j] = (float)bn_gamma[i][j];
        hp[d.bn_b_off[i] + j] = (float)bn_beta[i][j];
        hrm[d.bn_f_off[i] + j] = (float)bn_mean[i][j];
        hrv[d.bn_f_off[i] + j] = (float)bn_var[i][j];
      }
      hnbt[i] = bn_nbt ? bn_nbt[i] : 0;
    }
  }
  // float64 copies of what create received, for bb_trainer_set_precision(BB_PREC_FP64)
  t->params_host.assign(p, 0.0);
  for (int l = 0; l < NL; ++l) {
    const int K = dims[l], N = dims[l + 1];
    for (int i = 0; i < N * K; ++i) t->params_host[d.w_off[l] + i] = weights_host[l][i];
    for (int n = 0; n < N; ++n) t->params_host[d.b_off[l] + n] = biases_host[l][n];
  }
  if (kind == 1) {
    t->bn_stats_host.assign(2 * (size_t)d.bn_f_total, 0.0);
    for (int i = 0; i < 4; ++i) {
      for (int j = 0; j < dims[5 + i]; ++j) {
        t->params_host[d.bn_g_off[i] + j] = bn_gamma[i][j];
        t->params_host[d.bn_b_off[i] + j] = bn_beta[i][j];
        t->bn_stats_host[d.bn_f_off[i] + j] = bn_mean[i][j];
        t->bn_stats_host[d.bn_f_total + d.bn_f_off[i] + j] = bn_var[i][j];
      }
      t->nbt_host[i] = hnbt[i];
    }
  }
  t->n_tiles = (int)tiles.size();
  const int max_splits = (max_batch + DW_T - 1) / DW_T;
  const int max_ctas = (max_batch + RT - 1) / RT;
  int rc = BB_OK;
  auto alloc = [&](void** ptr, size_t bytes) { if (rc == BB_OK) rc = (int)cudaMalloc(ptr, bytes); };
  alloc((void**)&t->params, sizeof(float) * (p + 8));
  alloc((void**)&t->wt, sizeof(float) * (wtp + 8));
  alloc((void**)&t->grads, sizeof(float) * (p + 1));
  alloc((void**)&t->m, sizeof(float) * p);
  alloc((void**)&t->v, sizeof(float) * p);
  alloc((void**)&t->act_g, sizeof(float) * 2 * (size_t)max_batch * d.a_stride);
  alloc((void**)&t->dz_g, sizeof(float) * 2 * (size_t)max_batch * d.z_stride);
  alloc((void**)&t->partial, sizeof(float) * (size_t)max_splits * p);
  alloc((void**)&t->loss_part, sizeof(float) * max_ctas);
  alloc((void**)&t->wt_index, sizeof(int) * p);
  alloc((void**)&t->tiles, sizeof(DwTile) * tiles.size());
  alloc((void**)&t->loss_accum, sizeof(double));
  if (kind == 1) {
    alloc((void**)&t->bn_part, sizeof(float) * 8 * (size_t)max_ctas * 2 * mx);
    alloc((void**)&t->rm, sizeof(float) * d.bn_f_total);
    alloc((void**)&t->rv, sizeof(float) * d.bn_f_total);
    alloc((void**)&t->nbt, sizeof(long long) * 4);
  }
  if (rc == BB_OK) rc = (int)cudaMemcpy(t->params, hp.data(), sizeof(float) * p, cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemcpy(t->wt, hwt.data(), sizeof(float) * wtp, cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemcpy(t->wt_index, hidx.data(), sizeof(int) * p, cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemcpy(t->tiles, tiles.data(), sizeof(DwTile) * tiles.size(), cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemset(t->m, 0, sizeof(float) * p);
  if (rc == BB_OK) rc = (int)cudaMemset(t->v, 0, sizeof(float) * p);
  if (rc == BB_OK) rc = (int)cudaMemset(t->grads, 0, sizeof(float) * (p + 1));
  if (rc == BB_OK) rc = (int)cudaMemset(t->loss_accum, 0, sizeof(double));
  if (rc == BB_OK) rc = (int)cudaMemset(t->partial, 0, sizeof(float) * (size_t)max_splits * p);  // BN slots of splits > 0 stay zero
  if (rc == BB_OK && kind == 1) {
    rc = (int)cudaMemcpy(t->rm, hrm.data(), sizeof(float) * hrm.size(), cudaMemcpyHostToDevice);
    if (rc == BB_OK) rc = (int)cudaMemcpy(t->rv, hrv.data(), sizeof(float) * hrv.size(), cudaMemcpyHostToDevice);
    if (rc == BB_OK) rc = (int)cudaMemcpy(t->nbt, hnbt, sizeof(hnbt), cudaMemcpyHostToDevice);
    t->dbn_smem = t->smem_bytes + ((size_t)2 * d.bn_f_total * RT + d.bn_f_total + 4 + 2 * mx) * sizeof(float);
    if (t->dbn_smem > ctx->smem_optin) rc = BB_ERR_UNSUPPORTED;
    if (rc == BB_OK) rc = (int)cudaFuncSetAttribute(train_dbn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)t->dbn_smem);
    int per_sm = 0;
    if (rc == BB_OK) rc = (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, train_dbn_kernel, NT_FB, t->dbn_smem);
    t->dbn_max_ctas = per_sm * ctx->sm_count;
  }
  if (rc == BB_OK) rc = (int)cudaFuncSetAttribute(train_fwd_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)t->smem_bytes);
  if (rc == BB_OK) {
    // tensor-core path; shapes it does not take (BB_ERR_UNSUPPORTED) stay on the fp32 kernels
    int tacts[NL];
    for (int l = 0; l < NL; ++l) tacts[l] = acts[l];
    if (kind == 1) tacts[3] = BB_ACT_LEAKY;  // AE_Dropout_BN activates the latent too (models.py:273-275)
    const int trc = bb_tc_train_create(ctx, dims, tacts, max_batch, t->params, t->m, t->v, t->grads, kind, d.bn_g_off, d.bn_b_off,
                                       d.n_params, &t->tc);
    if (trc == BB_OK) {
      if (kind == 1) rc = bb_tc_train_set_bn(t->tc, t->rm, t->rv, t->nbt);
      if (rc == BB_OK) rc = bb_tc_train_repack(t->tc, nullptr);
    } else if (trc != BB_ERR_UNSUPPORTED) {
      rc = trc;
    }
    if (rc == BB_OK) rc = (int)cudaDeviceSynchronize();
  }
  if (rc != BB_OK) { bb_trainer_destroy(t); return rc; }
  *out = t;
  return BB_OK;
}
}  // namespace

extern "C" {

int bb_trainer_destroy(bb_trainer* t) {
  if (!t) return BB_OK;
  void* ptrs[] = {t->params, t->wt, t->grads, t->m, t->v, t->act_g, t->dz_g, t->partial, t->loss_part, t->wt_index, t->tiles, t->loss_accum,
                  t->bn_part, t->rm, t->rv, t->nbt};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  bb_tc_train_destroy(t->tc);
  bb_f64_train_destroy(t->f64);
  bb_host_window_free(t->win);
  delete t;
  return BB_OK;
}

int bb_trainer_set_precision(bb_trainer* t, int precision) {
  if (!t) return BB_ERR_INVALID;
  if (precision == BB_PREC_FP64) {
    if (t->started) return BB_ERR_INVALID;
    if (!t->f64) {
      F64TrainLayout fl;
      const TrainDims& d = t->d;
      memcpy(fl.dims, d.dims, sizeof(fl.dims));
      memcpy(fl.act, d.act, sizeof(fl.act));
      memcpy(fl.w_off, d.w_off, sizeof(fl.w_off));
      memcpy(fl.b_off, d.b_off, sizeof(fl.b_off));
      memcpy(fl.wt_off, d.wt_off, sizeof(fl.wt_off));
      memcpy(fl.a_off, d.a_off, sizeof(fl.a_off));
      memcpy(fl.z_off, d.z_off, sizeof(fl.z_off));
      fl.a_stride = d.a_stride; fl.z_stride = d.z_stride; fl.n_params = d.n_params; fl.max_dim = d.max_dim;
      fl.kind = t->kind;
      memcpy(fl.bn_g_off, d.bn_g_off, sizeof(fl.bn_g_off));
      memcpy(fl.bn_b_off, d.bn_b_off, sizeof(fl.bn_b_off));
      memcpy(fl.bn_f_off, d.bn_f_off, sizeof(fl.bn_f_off));
      fl.bn_f_total = d.bn_f_total;
      if (t->kind == 1) fl.act[3] = BB_ACT_LEAKY;  // AE_Dropout_BN activates the latent too (models.py:273-275)
      BB_CUDA(cudaSetDevice(t->ctx->device));
      int rc = bb_f64_train_create(t->ctx, fl, t->params_host.data(), t->kind == 1 ? t->bn_stats_host.data() : nullptr,
                                   t->nbt_host, t->max_batch, &t->f64);
      if (rc == BB_OK && t->kind == 1) rc = bb_f64_train_set_dropout(t->f64, t->seed, t->mask_dev);
      if (rc != BB_OK) {
        bb_f64_train_destroy(t->f64);
        t->f64 = nullptr;
        return rc;
      }
    }
    t->precision = BB_PREC_FP64;
    return BB_OK;
  }
  if (precision < BB_PREC_AUTO || precision > BB_PREC_SPLIT16) return BB_ERR_INVALID;
  if (t->precision == BB_PREC_FP64 && t->started) return BB_ERR_INVALID;
  if (precision == BB_PREC_SPLIT16 && !t->tc) return BB_ERR_UNSUPPORTED;
  t->precision = precision;
  return BB_OK;
}

int bb_trainer_precision(const bb_trainer* t) {
  if (!t) return BB_ERR_INVALID;
  if (t->precision == BB_PREC_FP64) return BB_PREC_FP64;
  return t->tc && t->precision != BB_PREC_FP32 ? BB_PREC_SPLIT16 : BB_PREC_FP32;
}

int bb_trainer_range_flag(bb_trainer* t, int reset, int* out) {
  if (!t || !out) return BB_ERR_INVALID;
  *out = 0;
  if (t->precision == BB_PREC_FP64) return BB_OK;
  return t->tc ? bb_tc_train_range_flag(t->tc, reset, out) : BB_OK;
}

int bb_trainer_debug_layer(bb_trainer* t, int which, int layer, int rows, float* out_host, int capacity_floats) {
  if (!t || !t->tc) return BB_ERR_UNSUPPORTED;
  return bb_tc_train_debug_layer(t->tc, which, layer, rows, out_host, capacity_floats);
}

int bb_trainer_dp_export(bb_trainer* t, int world_size, unsigned char* handle_out_64) {
  if (!t || !t->tc || t->precision == BB_PREC_FP64) return BB_ERR_UNSUPPORTED;
  return bb_tc_train_dp_export(t->tc, world_size, handle_out_64);
}

int bb_trainer_dp_connect(bb_trainer* t, int rank, int world_size, const unsigned char* handles) {
  if (!t || !t->tc || t->precision == BB_PREC_FP64) return BB_ERR_UNSUPPORTED;
  return bb_tc_train_dp_connect(t->tc, rank, world_size, handles);
}

int bb_trainer_profile(bb_trainer* t, int step, long long* out_128) {
  if (!t || !t->tc) return BB_ERR_UNSUPPORTED;
  return bb_tc_train_profile(t->tc, step, out_128);
}

int bb_trainer_param_count(const bb_trainer* t) { return t ? t->d.n_params : 0; }
float* bb_trainer_params_dev(bb_trainer* t) { return t ? t->params : nullptr; }
float* bb_trainer_grads_dev(bb_trainer* t) { return t ? t->grads : nullptr; }
double* bb_trainer_params_dev_f64(bb_trainer* t) { return t && t->precision == BB_PREC_FP64 ? bb_f64_train_params(t->f64) : nullptr; }
double* bb_trainer_grads_dev_f64(bb_trainer* t) { return t && t->precision == BB_PREC_FP64 ? bb_f64_train_grads(t->f64) : nullptr; }

int bb_trainer_get_params(bb_trainer* t, double* const* weights_host, double* const* biases_host) {
  if (!t || !weights_host || !biases_host) return BB_ERR_INVALID;
  if (t->precision == BB_PREC_FP64) {  // the float64 master as it is
    std::vector<double> hp(t->d.n_params);
    const int rc = bb_f64_train_get_params(t->f64, hp.data());
    if (rc != BB_OK) return rc;
    for (int l = 0; l < NL; ++l) {
      const int K = t->d.dims[l], N = t->d.dims[l + 1];
      memcpy(weights_host[l], hp.data() + t->d.w_off[l], sizeof(double) * N * K);
      memcpy(biases_host[l], hp.data() + t->d.b_off[l], sizeof(double) * N);
    }
    return BB_OK;
  }
  std::vector<float> hp(t->d.n_params);
  BB_CUDA(cudaMemcpy(hp.data(), t->params, sizeof(float) * hp.size(), cudaMemcpyDeviceToHost));
  for (int l = 0; l < NL; ++l) {
    const int K = t->d.dims[l], N = t->d.dims[l + 1];
    for (int i = 0; i < N * K; ++i) weights_host[l][i] = (double)hp[t->d.w_off[l] + i];
    for (int n = 0; n < N; ++n) biases_host[l][n] = (double)hp[t->d.b_off[l] + n];
  }
  return BB_OK;
}

}  // extern "C"

namespace {
// BB_PREC_FP64: the float64 step of bb_train_f64.cu on a float32 table (widened exactly) or a float64 one
int step_f64(bb_trainer* t, const void* x, int x_is_f64, int rows, const bb_train_hyper* h, int phase, double* loss_accum,
             cudaStream_t s) {
  if (!t || !h || !x || rows < 1 || rows > t->max_batch || phase < 0 || phase > 2) return BB_ERR_INVALID;
  if (t->precision != BB_PREC_FP64) return BB_ERR_INVALID;
  t->started = true;
  const long long step = phase != 1 ? t->step + 1 : t->step;
  const int rc = bb_f64_train_step(t->f64, x, x_is_f64, rows, h, phase, step, loss_accum, s);
  if (rc == BB_OK) t->step = step;
  return rc;
}

// Arguments of an epoch on a table of float32 (x_is_f64 = 0) or float64 rows that the entry points refuse, else BB_OK
int check_epoch(bb_trainer* t, int x_is_f64, int batch, const bb_train_hyper* h) {
  if (x_is_f64 && t->precision != BB_PREC_FP64) return BB_ERR_INVALID;
  if (t->precision == BB_PREC_FP64) {
    if (batch > t->max_batch) return BB_ERR_INVALID;
    return h->world_size > 1 ? BB_ERR_UNSUPPORTED : BB_OK;  // data parallel: phases 1 and 2 around the caller's all-reduce
  }
  t->started = true;
  if (h->world_size <= 1 && batch > t->max_batch) return BB_ERR_INVALID;
  const int dp_world = t->tc ? bb_tc_train_dp_world(t->tc) : 1;
  if (h->world_size > 1 && h->world_size != dp_world) return BB_ERR_INVALID;  // data parallel needs bb_trainer_dp_connect
  if (h->world_size > 1 && (batch + dp_world - 1) / dp_world > t->max_batch) return BB_ERR_INVALID;
  return BB_OK;
}

// The training steps of the batches of rows [0, n_rows) of x in order (the last one may be ragged), their losses added to
// t->loss_accum.  The body of an epoch over a device table, and of every window of a streamed host table: windows hold
// whole batches and the step counter runs on, so both run the same steps.
int train_rows(bb_trainer* t, const void* x, int x_is_f64, int64_t n_rows, int batch, const bb_train_hyper* h, cudaStream_t s) {
  const size_t row_bytes = (size_t)t->d.dims[0] * (x_is_f64 ? sizeof(double) : sizeof(float));
  if (t->precision == BB_PREC_FP64) {
    for (int64_t r0 = 0; r0 < n_rows; r0 += batch) {
      const int rows = (int)(n_rows - r0 < batch ? n_rows - r0 : batch);
      const int rc = step_f64(t, (const char*)x + (size_t)r0 * row_bytes, x_is_f64, rows, h, 0, t->loss_accum, s);
      if (rc != BB_OK) return rc;
    }
    return BB_OK;
  }
  int urc;
  if (use_tc(t, h, s, &urc)) {
    // the whole epoch (window) is one persistent kernel: no launch and no host round trip between steps
    if (urc != BB_OK) return urc;
    const TcHyper th = tc_hyper(h);
    const int64_t n_batches = (n_rows + batch - 1) / batch;
    t->wt_fresh = false;
    t->last_tc = true;
    t->last_rows = (int)(n_rows - (n_batches - 1) * batch);
    bb_tc_train_set_mode(t->tc, 1, (unsigned long long)t->step);
    const int rc = bb_tc_train_run(t->tc, (const float*)x, n_rows, batch, TC_P1 | TC_DW | TC_ADAM, &th, t->step + 1,
                                   t->loss_accum, h->world_size > 1 ? 1 : 0, s);
    if (rc != BB_OK) return rc;
    t->step += n_batches;
    return BB_OK;
  }
  if (urc != BB_OK) return urc;
  if (h->world_size > 1) return BB_ERR_UNSUPPORTED;  // the fused exchange lives in the tensor-core kernel
  for (int64_t r0 = 0; r0 < n_rows; r0 += batch) {
    const int rows = (int)(n_rows - r0 < batch ? n_rows - r0 : batch);
    const int rc = bb_trainer_step(t, (const float*)x + (size_t)r0 * t->d.dims[0], rows, h, 0, t->loss_accum, s);
    if (rc != BB_OK) return rc;
  }
  return BB_OK;
}

// The eval-mode forward passes of the batches of rows [0, n_rows) of x, their losses added to t->loss_accum (validate;
// windows as in train_rows)
int eval_rows(bb_trainer* t, const void* x, int x_is_f64, int64_t n_rows, int batch, cudaStream_t s) {
  if (t->precision == BB_PREC_FP64) {
    const size_t row_bytes = (size_t)t->d.dims[0] * (x_is_f64 ? sizeof(double) : sizeof(float));
    for (int64_t r0 = 0; r0 < n_rows; r0 += batch) {
      const int rows = (int)(n_rows - r0 < batch ? n_rows - r0 : batch);
      const int rc = bb_f64_train_eval(t->f64, (const char*)x + (size_t)r0 * row_bytes, x_is_f64, rows, t->loss_accum, s);
      if (rc != BB_OK) return rc;
    }
    return BB_OK;
  }
  const float* xf = (const float*)x;
  int urc;
  const bool tc = use_tc(t, nullptr, s, &urc);
  if (urc != BB_OK) return urc;
  if (tc) {
    TcHyper th;
    memset(&th, 0, sizeof(th));
    th.b1d = th.b2d = 0.5;
    const int64_t n_batches = (n_rows + batch - 1) / batch;
    t->last_tc = true;
    t->last_rows = (int)(n_rows - (n_batches - 1) * batch);
    bb_tc_train_set_mode(t->tc, 0, 0ull);
    return bb_tc_train_run(t->tc, xf, n_rows, batch, TC_FWD_ONLY, &th, 1, t->loss_accum, 0, s);
  }
  for (int64_t r0 = 0; r0 < n_rows; r0 += batch) {
    const int rows = (int)(n_rows - r0 < batch ? n_rows - r0 : batch);
    t->last_tc = false;
    int rc = t->kind == 1 ? launch_dbn(t, xf + (size_t)r0 * t->d.dims[0], rows, 1, s)
                          : launch_fwd_bwd(t, xf + (size_t)r0 * t->d.dims[0], rows, 0, nullptr, s);
    if (rc != BB_OK) return rc;
    // mode 1 with zero splits: only folds the loss partials into the gradient's loss slot ...
    train_adam_kernel<<<1, NT, 0, s>>>(0, 1, t->partial, 0, t->grads + t->d.n_params, nullptr, nullptr, nullptr, nullptr,
                                       nullptr, 0.f, 0.f, 0.f, 0.f, 0.f, t->loss_part, (rows + RT - 1) / RT, nullptr);
    // ... and mode 2 with zero parameters adds that slot to the accumulator
    train_adam_kernel<<<1, NT, 0, s>>>(0, 2, nullptr, 0, t->grads + t->d.n_params, nullptr, nullptr, nullptr, nullptr,
                                       nullptr, 0.f, 0.f, 0.f, 0.f, 0.f, nullptr, 0, t->loss_accum);
    BB_CUDA(cudaGetLastError());
  }
  return BB_OK;
}

// epoch loss = the summed batch losses over the number of batches (training.py:99); synchronises s
int finish_epoch(bb_trainer* t, int64_t n_rows, int batch, double* epoch_loss_host, cudaStream_t s) {
  double total = 0.0;
  BB_CUDA(cudaMemcpyAsync(&total, t->loss_accum, sizeof(double), cudaMemcpyDeviceToHost, s));
  BB_CUDA(cudaStreamSynchronize(s));
  *epoch_loss_host = total / (double)((n_rows + batch - 1) / batch);
  return BB_OK;
}

int epoch_dev(bb_trainer* t, const void* x, int x_is_f64, int64_t n_rows, int batch, const bb_train_hyper* h,
              double* epoch_loss_host, cudaStream_t s) {
  if (!t || !h || !x || n_rows < 1 || batch < 1 || !epoch_loss_host) return BB_ERR_INVALID;
  int rc = check_epoch(t, x_is_f64, batch, h);
  if (rc != BB_OK) return rc;
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  rc = train_rows(t, x, x_is_f64, n_rows, batch, h, s);
  return rc != BB_OK ? rc : finish_epoch(t, n_rows, batch, epoch_loss_host, s);
}

int validate_dev(bb_trainer* t, const void* x, int x_is_f64, int64_t n_rows, int batch, double* epoch_loss_host,
                 cudaStream_t s) {
  if (!t || !x || n_rows < 1 || batch < 1 || batch > t->max_batch || !epoch_loss_host) return BB_ERR_INVALID;
  if (x_is_f64 && t->precision != BB_PREC_FP64) return BB_ERR_INVALID;
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  const int rc = eval_rows(t, x, x_is_f64, n_rows, batch, s);
  return rc != BB_OK ? rc : finish_epoch(t, n_rows, batch, epoch_loss_host, s);
}

// bytes per row of a host table of x_dtype for this trainer (0: a dtype it does not take); checks the window
size_t host_row_bytes(bb_trainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch, int64_t window_rows) {
  if (!x_host || n_rows < 1 || batch < 1 || window_rows < batch || window_rows % batch) return 0;
  if (x_dtype == BB_F32) return (size_t)t->d.dims[0] * sizeof(float);
  if (x_dtype == BB_F64 && t->precision == BB_PREC_FP64) return (size_t)t->d.dims[0] * sizeof(double);
  return 0;
}
}  // namespace

extern "C" {

int bb_trainer_step_f64(bb_trainer* t, const double* x_dev, int batch_rows, const bb_train_hyper* h, int phase,
                        double* loss_accum_dev, bb_stream_t stream) {
  return step_f64(t, x_dev, 1, batch_rows, h, phase, loss_accum_dev, (cudaStream_t)stream);
}

int bb_trainer_epoch_f64(bb_trainer* t, const double* x_dev, int64_t n_rows, int batch, const bb_train_hyper* h,
                         double* epoch_loss_host, bb_stream_t stream) {
  return epoch_dev(t, x_dev, 1, n_rows, batch, h, epoch_loss_host, (cudaStream_t)stream);
}

int bb_trainer_validate_f64(bb_trainer* t, const double* x_dev, int64_t n_rows, int batch, double* epoch_loss_host,
                            bb_stream_t stream) {
  return validate_dev(t, x_dev, 1, n_rows, batch, epoch_loss_host, (cudaStream_t)stream);
}

int bb_trainer_step(bb_trainer* t, const float* x_dev, int batch_rows, const bb_train_hyper* h, int phase,
                    double* loss_accum_dev, bb_stream_t stream) {
  if (!t || !h || !x_dev || batch_rows < 1 || batch_rows > t->max_batch || phase < 0 || phase > 2) return BB_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  if (t->precision == BB_PREC_FP64) return step_f64(t, x_dev, 0, batch_rows, h, phase, loss_accum_dev, s);
  t->started = true;
  int urc;
  if (use_tc(t, h, s, &urc)) {
    if (urc != BB_OK) return urc;
    const TcHyper th = tc_hyper(h);
    t->wt_fresh = t->wt_fresh && phase == 1;
    if (phase != 2) { t->last_rows = batch_rows; t->last_tc = true; }
    if (phase == 2) {
      t->step += 1;
      return bb_tc_train_adam_flat(t->tc, &th, t->step, loss_accum_dev, s);
    }
    const int flags = TC_P1 | TC_DW | TC_GRADS | (phase == 0 ? TC_ADAM : 0);
    bb_tc_train_set_mode(t->tc, 1, (unsigned long long)t->step);
    if (phase == 0) t->step += 1;
    return bb_tc_train_run(t->tc, x_dev, batch_rows, batch_rows, flags, &th, t->step, loss_accum_dev, 0, s);
  }
  if (urc != BB_OK) return urc;
  if (phase != 1) t->tc_fresh = false;
  if (phase != 2) t->last_tc = false;
  const int p = t->d.n_params;
  const int n_splits = (batch_rows + DW_T - 1) / DW_T;
  const int n_ctas = (batch_rows + RT - 1) / RT;
  if (phase != 2) {
    // AE_Dropout_BN: MSE only.  world_size > 1 is data parallel with per-rank BatchNorm statistics (each rank normalises
    // its slice of the global batch, what torch DistributedDataParallel does with this model); gradients are summed.
    if (t->kind == 1 && h->l1) return BB_ERR_UNSUPPORTED;
    int rc = t->kind == 1 ? launch_dbn(t, x_dev, batch_rows, 0, s) : launch_fwd_bwd(t, x_dev, batch_rows, 1, h, s);
    if (rc != BB_OK) return rc;
    BB_CUDA(pdl_launch(train_dw_kernel, dim3(t->n_tiles, n_splits), dim3(NT), 0, s, t->d, t->tiles, t->act_g, t->dz_g,
                       (size_t)t->max_batch * t->d.a_stride, (size_t)t->max_batch * t->d.z_stride, h->l1 ? 2 : 1, batch_rows,
                       t->partial));
  }
  float lr_bc1 = 0.f, inv_sqrt_bc2 = 0.f;
  if (phase != 1) {
    t->step += 1;
    const double bc1 = 1.0 - std::pow(h->beta1, (double)t->step);
    const double bc2 = 1.0 - std::pow(h->beta2, (double)t->step);
    lr_bc1 = (float)(h->lr / bc1);
    inv_sqrt_bc2 = (float)(1.0 / std::sqrt(bc2));
  }
  return (int)pdl_launch(train_adam_kernel, dim3((p + NT - 1) / NT), dim3(NT), 0, s, p, phase, t->partial, n_splits, t->grads,
                         t->params, t->wt, t->wt_index, t->m, t->v, lr_bc1, inv_sqrt_bc2, (float)h->beta1, (float)h->beta2,
                         (float)h->eps, t->loss_part, n_ctas, loss_accum_dev);
}

int bb_trainer_epoch(bb_trainer* t, const float* x_dev, int64_t n_rows, int batch, const bb_train_hyper* h,
                     double* epoch_loss_host, bb_stream_t stream) {
  return epoch_dev(t, x_dev, 0, n_rows, batch, h, epoch_loss_host, (cudaStream_t)stream);
}

int bb_trainer_validate(bb_trainer* t, const float* x_dev, int64_t n_rows, int batch, double* epoch_loss_host,
                        bb_stream_t stream) {
  return validate_dev(t, x_dev, 0, n_rows, batch, epoch_loss_host, (cudaStream_t)stream);
}

int bb_trainer_epoch_host(bb_trainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch, const bb_train_hyper* h,
                          int64_t window_rows, double* epoch_loss_host, bb_stream_t stream) {
  if (!t || !h || !epoch_loss_host) return BB_ERR_INVALID;
  const size_t row_bytes = host_row_bytes(t, x_host, x_dtype, n_rows, batch, window_rows);
  if (!row_bytes) return BB_ERR_INVALID;
  const int x_is_f64 = x_dtype == BB_F64;
  int rc = check_epoch(t, x_is_f64, batch, h);
  if (rc != BB_OK) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  BB_CUDA(cudaSetDevice(t->ctx->device));
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  rc = bb_host_window_run(&t->win, x_host, row_bytes, n_rows, window_rows, s, [&](const void* x, int64_t rows) {
    return train_rows(t, x, x_is_f64, rows, batch, h, s);
  });
  return rc != BB_OK ? rc : finish_epoch(t, n_rows, batch, epoch_loss_host, s);
}

int bb_trainer_validate_host(bb_trainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch, int64_t window_rows,
                             double* epoch_loss_host, bb_stream_t stream) {
  if (!t || !epoch_loss_host || batch > t->max_batch) return BB_ERR_INVALID;
  const size_t row_bytes = host_row_bytes(t, x_host, x_dtype, n_rows, batch, window_rows);
  if (!row_bytes) return BB_ERR_INVALID;
  const int x_is_f64 = x_dtype == BB_F64;
  cudaStream_t s = (cudaStream_t)stream;
  BB_CUDA(cudaSetDevice(t->ctx->device));
  BB_CUDA(cudaMemsetAsync(t->loss_accum, 0, sizeof(double), s));
  const int rc = bb_host_window_run(&t->win, x_host, row_bytes, n_rows, window_rows, s, [&](const void* x, int64_t rows) {
    return eval_rows(t, x, x_is_f64, rows, batch, s);
  });
  return rc != BB_OK ? rc : finish_epoch(t, n_rows, batch, epoch_loss_host, s);
}

int bb_trainer_activation_means(bb_trainer* t, double* out) {
  if (!t || !out) return BB_ERR_INVALID;
  if (t->precision == BB_PREC_FP64) return bb_f64_train_activation_means(t->f64, out);
  if (t->last_tc) return bb_tc_train_activation_means(t->tc, t->last_rows, out);
  const int rows = t->last_rows, stride = t->d.a_stride;
  std::vector<float> h((size_t)rows * stride);
  if (rows) BB_CUDA(cudaMemcpy(h.data(), t->act_g, h.size() * sizeof(float), cudaMemcpyDeviceToHost));
  const int layers[6] = {1, 2, 3, 5, 6, 7};  // A_l = LeakyReLU(output of Linear l-1)
  for (int i = 0; i < 6; ++i) {
    const int l = layers[i], n = t->d.dims[l];
    for (int j = 0; j < 200; ++j) {
      double s = NAN;
      if (j < n && rows) {
        s = 0.0;
        for (int r = 0; r < rows; ++r) s += (double)h[(size_t)r * stride + t->d.a_off[l] + j];
        s /= rows;
      }
      out[i * 200 + j] = s;
    }
  }
  return BB_OK;
}

}  // extern "C"

namespace {
__global__ void __launch_bounds__(1024) mse_sum_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                       const int64_t n, double* __restrict__ out) {
  __shared__ double part[32];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += 1024) {
    const float d = a[i] - b[i];
    s += (double)d * d;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int w = 0; w < 32; ++w) tot += part[w];
    *out += tot;
  }
}
}  // namespace

extern "C" int bb_mse_sum_f32(bb_ctx* ctx, const float* a_dev, const float* b_dev, int64_t n, double* out_dev,
                              bb_stream_t stream) {
  if (!ctx || !out_dev || n < 0 || ((!a_dev || !b_dev) && n)) return BB_ERR_INVALID;
  mse_sum_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(a_dev, b_dev, n, out_dev);
  return (int)cudaGetLastError();
}
