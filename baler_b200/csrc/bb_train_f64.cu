// Training step of the dense autoencoder in float64 (DFMA on CUDA cores): BB_PREC_FP64 of bb_trainer.
//
// The reference trains its float64 AE in float64 on torch (training.py:230 makes a float64 tensor of the normalised
// table; fit, training.py:64-97, with Adam, training.py:266).  This is the three-launch step of bb_train.cu with every
// value in float64, so a run reproduces the reference's training to rounding (~1e-14 over the horizons of the tests):
//   1. train_fwd_bwd_f64_kernel  one CTA (512 threads) per RT = 4 rows of the batch: 8 layers forward, the loss (sum-MSE
//      / n_cols, + reg * L1 chain when h->l1), 7 layers backward, every activation of its rows transposed in shared
//      memory (act[feature][RT]).  It leaves the layer inputs A_l and the pre-activation gradients dZ_l (row-major
//      [B][dim]) in global scratch and one loss partial per CTA.
//   2. train_dw_f64_kernel       dW_l = dZ_l^T A_l as 64 x 64 output tiles x 64-row splits, written as per-split partial
//      sums (no atomics: fixed summation order, reproducible).
//   3. train_adam_f64_kernel     sums the split partials into the flat gradient (+ the batch loss in its last slot),
//      applies torch's Adam in the operation order of torch.optim.Adam (single-tensor) and refreshes the transposed weights.
// The launches are chained with programmatic dependent launch; a step does not synchronise with the host.
//
// Weights.  The fp32 kernel double-buffers whole matrices in shared memory; in float64 one 200 x 100 matrix is 160 KB,
// so two do not fit.  Every pass instead streams its matrix (W^T [K][N] forward, W [N][K] backward: rows of the
// reduction dimension) in chunks of KC = 16 rows through a two-stage cp.async ring, the next chunk (of this pass or of
// the next one) landing while the current one is multiplied, as chain_f64_kernel does.
// Budget per CTA at RT = 4 for the CMS shape (24 columns, z = 15): activations 763 x 4 x 8 B = 24 KB, dZ 2 x 6.4 KB,
// reduction 16 KB, ring 2 x (16 x 200 + 2) x 8 B = 51 KB: 105 KB.
//
// Arithmetic.  Dot products are DFMA chains; a narrow output splits its reduction over KP thread groups (KP a power of
// two dividing KC, each group owning KC / KP consecutive rows of every chunk) combined in a fixed order.  The bias add,
// LeakyReLU (slope 0.01 as __dmul_rn, F.leaky_relu in float64), the loss terms and Adam are single IEEE operations with
// no contraction.  Inputs arrive as float32 (widened exactly, what torch.tensor(..., float64) does) or float64.
#include <cmath>
#include <cstring>
#include <new>

#include <cooperative_groups.h>

#include "bb_train_f64.cuh"

namespace {

constexpr int NL = 8;
constexpr int RT = 4;        // rows per CTA of the forward / backward kernel
constexpr int NT_FB = 512;   // threads of the forward / backward kernel
constexpr int NT = 256;      // dW and Adam kernels
constexpr int KC = 16;       // reduction rows of a streamed weight chunk
constexpr int DW_T = 64;     // dW output tile edge and rows per split
constexpr int DW_R = 32;     // rows of a split staged in shared memory at a time
constexpr int DW_LD = DW_T + 2;

struct Tile { int l, n0, k0; };

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

__device__ __forceinline__ void cp_async16(double* smem, const double* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ double act_fwd(double v, int act) {
  if (act == BB_ACT_LEAKY) return v > 0.0 ? v : __dmul_rn(0.01, v);
  if (act == BB_ACT_RELU) return v > 0.0 ? v : (v == v ? 0.0 : v);
  return v;
}

// Matrix of pass p (0..7 forward on W_l^T, 8..14 backward on W_l for l = 7..1): rows of `dout` doubles, `din` rows.
__device__ __forceinline__ const double* pass_src(const F64TrainLayout& d, const double* params, const double* wt, int p,
                                                  int& din, int& dout) {
  if (p < NL) { din = d.dims[p]; dout = d.dims[p + 1]; return wt + d.wt_off[p]; }
  const int l = 2 * NL - 1 - p;
  din = d.dims[l + 1]; dout = d.dims[l];
  return params + d.w_off[l];
}

// The weight stream of one launch: `total` passes (per_chain per chain), chunk n of the stream in ring stage n & 1.
struct Stream {
  double* ring;
  int stage_elems;
  int n;                // chunks consumed so far
  int next_p, next_i0;  // next chunk to issue: pass (stream position) and first row
  int total, per_chain;
};

// issue the next chunk of the stream into stage (s.n + 1) & 1 (an empty group once the stream is exhausted)
__device__ __forceinline__ void issue_next(const F64TrainLayout& d, const double* params, const double* wt, Stream& s, int stage) {
  if (s.next_p < s.total) {
    int din, dout;
    const double* src = pass_src(d, params, wt, s.next_p % s.per_chain, din, dout);
    src += (size_t)s.next_i0 * dout;
    const double* a = reinterpret_cast<const double*>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)15);
    const int rows = min(KC, din - s.next_i0);
    const int n16 = ((int)(src - a) + rows * dout + 1) >> 1;
    double* dst = s.ring + stage * s.stage_elems;
    for (int i = threadIdx.x; i < n16; i += NT_FB) cp_async16(dst + 2 * i, a + 2 * i);
    s.next_i0 += KC;
    if (s.next_i0 >= din) { s.next_i0 = 0; ++s.next_p; }
  }
  cp_async_commit();
}

// red_s[kp][r][j] = partial sums of out[r][j] = sum_i in_s[i][r] * M[i][j] over the KP row groups, M = the matrix at
// `src` (din x dout) streamed chunk by chunk.  Ends with __syncthreads.  Returns KP.
__device__ __forceinline__ int gemv_f64(const F64TrainLayout& d, const double* params, const double* wt, Stream& s,
                                        const double* src, const double* __restrict__ in_s, const int din, const int dout,
                                        double* __restrict__ red_s) {
  int KP = 1;
  while (KP < KC && 2 * KP * dout <= NT_FB) KP *= 2;
  const int R = KC / KP;
  const int kp = threadIdx.x / dout, j = threadIdx.x - kp * dout;
  const bool active = kp < KP;
  double acc[RT];
#pragma unroll
  for (int r = 0; r < RT; ++r) acc[r] = 0.0;
  for (int i0 = 0; i0 < din; i0 += KC) {
    cp_async_wait_all();
    __syncthreads();  // chunk n landed for every thread; the other stage (chunk n - 1) is no longer read
    issue_next(d, params, wt, s, (s.n + 1) & 1);
    const double* cs = src + (size_t)i0 * dout;
    const double* w = s.ring + (s.n & 1) * s.stage_elems + ((reinterpret_cast<uintptr_t>(cs) & 15) >> 3);
    if (active) {
      const int ib = i0 + kp * R, ie = min(din, ib + R);
      for (int i = ib; i < ie; ++i) {
        const double wv = w[(i - i0) * dout + j];
        const double2 a01 = *reinterpret_cast<const double2*>(in_s + i * RT);
        const double2 a23 = *reinterpret_cast<const double2*>(in_s + i * RT + 2);
        acc[0] = fma(a01.x, wv, acc[0]);
        acc[1] = fma(a01.y, wv, acc[1]);
        acc[2] = fma(a23.x, wv, acc[2]);
        acc[3] = fma(a23.y, wv, acc[3]);
      }
    }
    ++s.n;
  }
  if (active) {
#pragma unroll
    for (int r = 0; r < RT; ++r) red_s[(kp * RT + r) * dout + j] = acc[r];
  }
  __syncthreads();
  return KP;
}

__device__ __forceinline__ double red_sum(const double* red_s, int KP, int dout, int r, int j) {
  double v = red_s[r * dout + j];
  for (int kp = 1; kp < KP; ++kp) v = __dadd_rn(v, red_s[(kp * RT + r) * dout + j]);
  return v;
}

// One chain forward + backward for RT rows (as run_chain of bb_train.cu):
//   chain 0: loss term sum((recon - x)^2) / C, seed gradient 2 (recon - x) / C
//   chain 1: loss term reg * sum_l mean|v_l|,  gradient reg / (B * N_l) injected at every layer output (ReLU chain)
template <int CHAIN>
__device__ void run_chain(const F64TrainLayout& d, const double* __restrict__ params, const double* __restrict__ wt,
                          double* __restrict__ act_g, double* __restrict__ dz_g, const int row0, const int rows,
                          const bool backward, const double reg_inv_rows, double* act_s, double* dz_s0, double* dz_s1,
                          double* red_s, double& loss_local, Stream& s) {
  for (int l = 0; l < NL; ++l) {
    int K, N;
    const double* src = pass_src(d, params, wt, l, K, N);
    const double* in_s = act_s + d.a_off[l] * RT;
    double* out_s = act_s + d.a_off[l + 1] * RT;
    const int KP = gemv_f64(d, params, wt, s, src, in_s, K, N, red_s);
    const double* bias = params + d.b_off[l];
    const int act = CHAIN == 0 ? d.act[l] : BB_ACT_RELU;
    const double l1_scale = CHAIN == 1 ? __ddiv_rn(reg_inv_rows, (double)N) : 0.0;
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      const int r = o / N, j = o - r * N;
      const double v = act_fwd(__dadd_rn(red_sum(red_s, KP, N, r, j), __ldg(bias + j)), act);
      out_s[j * RT + r] = v;
      if (r < rows && l + 1 < NL) act_g[(size_t)(row0 + r) * d.a_stride + d.a_off[l + 1] + j] = v;
      if (CHAIN == 1 && r < rows) loss_local = __dadd_rn(loss_local, __dmul_rn(l1_scale, fabs(v)));
    }
    __syncthreads();
  }
  const int F = d.dims[NL];
  double* dz_cur = dz_s0;
  double* dz_nxt = dz_s1;
  {
    const double* out_s = act_s + d.a_off[NL] * RT;
    const double* x_s = act_s;
    const double seed = CHAIN == 1 ? __ddiv_rn(reg_inv_rows, (double)F) : 0.0;
    for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
      const int r = o / F, j = o - r * F;
      double g = 0.0;
      if (r < rows) {
        if (CHAIN == 0) {
          const double diff = __dsub_rn(out_s[j * RT + r], x_s[j * RT + r]);
          loss_local = __dadd_rn(loss_local, __ddiv_rn(__dmul_rn(diff, diff), (double)F));
          g = __ddiv_rn(__dmul_rn(2.0, diff), (double)F);
        } else {
          g = out_s[j * RT + r] > 0.0 ? seed : 0.0;
        }
        if (backward) dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[NL - 1] + j] = g;
      }
      dz_cur[j * RT + r] = g;
    }
    __syncthreads();
  }
  if (!backward) return;
  for (int l = NL - 1; l >= 1; --l) {
    int N, K;
    const double* src = pass_src(d, params, wt, 2 * NL - 1 - l, N, K);  // W_l [N][K]: reduce over N
    const int KP = gemv_f64(d, params, wt, s, src, dz_cur, N, K, red_s);
    const double* a_s = act_s + d.a_off[l] * RT;  // output of layer l - 1 (post-activation)
    const int act = CHAIN == 0 ? d.act[l - 1] : BB_ACT_RELU;
    const double seed = CHAIN == 1 ? __ddiv_rn(reg_inv_rows, (double)K) : 0.0;
    for (int o = threadIdx.x; o < RT * K; o += NT_FB) {
      const int r = o / K, j = o - r * K;
      double g = red_sum(red_s, KP, K, r, j);
      if (CHAIN == 1) g = __dadd_rn(g, seed);
      const double a = a_s[j * RT + r];
      if (act == BB_ACT_LEAKY) g = a > 0.0 ? g : __dmul_rn(g, 0.01);
      else if (act == BB_ACT_RELU) g = a > 0.0 ? g : 0.0;
      if (r >= rows) g = 0.0;
      dz_nxt[j * RT + r] = g;
      if (r < rows) dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[l - 1] + j] = g;
    }
    __syncthreads();
    double* t = dz_cur; dz_cur = dz_nxt; dz_nxt = t;
  }
}

// scratch per chain c: act_g + c * chain_act_stride, dz_g + c * chain_dz_stride
__global__ void __launch_bounds__(NT_FB)
train_fwd_bwd_f64_kernel(const __grid_constant__ F64TrainLayout d, const double* __restrict__ params,
                         const double* __restrict__ wt, const void* __restrict__ x, const int x_is_f64,
                         const int batch_rows, double* __restrict__ act_g, double* __restrict__ dz_g,
                         const size_t chain_act_stride, const size_t chain_dz_stride, const int backward, const int l1,
                         const double reg_inv_rows, double* __restrict__ loss_part) {
  extern __shared__ __align__(16) double smem[];
  __shared__ double warp_loss[NT_FB / 32];
  pdl_launch_dependents();
  pdl_wait();  // parameters come from the previous step's Adam kernel
  double* act_s = smem;                       // a_stride * RT
  double* dz_s0 = act_s + d.a_stride * RT;    // max_dim * RT
  double* dz_s1 = dz_s0 + d.max_dim * RT;
  double* red_s = dz_s1 + d.max_dim * RT;     // max(max_dim, NT_FB) * RT
  Stream s;
  s.ring = red_s + (d.max_dim > NT_FB ? d.max_dim : NT_FB) * RT;
  s.stage_elems = (KC * d.max_dim + 2 + 1) & ~1;
  s.n = 0;
  s.next_p = 0; s.next_i0 = 0;
  s.per_chain = backward ? 2 * NL - 1 : NL;
  s.total = s.per_chain * (l1 ? 2 : 1);
  issue_next(d, params, wt, s, 0);

  const int row0 = blockIdx.x * RT;
  const int rows = min(RT, batch_rows - row0);
  const int F = d.dims[0];
  for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
    const int r = o / F, j = o - r * F;
    double v = 0.0;
    if (r < rows) {
      const size_t e = (size_t)(row0 + r) * F + j;
      v = x_is_f64 ? __ldg(reinterpret_cast<const double*>(x) + e) : (double)__ldg(reinterpret_cast<const float*>(x) + e);
      act_g[(size_t)(row0 + r) * d.a_stride + j] = v;  // A_0 keeps the dW kernel uniform
    }
    act_s[j * RT + r] = v;
  }
  __syncthreads();
  double loss_local = 0.0;
  run_chain<0>(d, params, wt, act_g, dz_g, row0, rows, backward != 0, 0.0, act_s, dz_s0, dz_s1, red_s, loss_local, s);
  if (l1) {
    __syncthreads();
    for (int o = threadIdx.x; o < RT * F; o += NT_FB) {  // A_0 of the second chain is x as well
      const int r = o / F, j = o - r * F;
      if (r < rows) act_g[chain_act_stride + (size_t)(row0 + r) * d.a_stride + j] = act_s[j * RT + r];
    }
    run_chain<1>(d, params, wt, act_g + chain_act_stride, dz_g + chain_dz_stride, row0, rows, backward != 0, reg_inv_rows,
                 act_s, dz_s0, dz_s1, red_s, loss_local, s);
  }
  cp_async_wait_all();
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) loss_local = __dadd_rn(loss_local, __shfl_xor_sync(0xffffffffu, loss_local, off));
  if ((threadIdx.x & 31) == 0) warp_loss[threadIdx.x >> 5] = loss_local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int w = 0; w < NT_FB / 32; ++w) v = __dadd_rn(v, warp_loss[w]);
    loss_part[blockIdx.x] = v;
  }
}

// ------------------------------------------------------------------------------------------------ AE_Dropout_BN
// reference baler/modules/models.py:256-313 in float64, in torch's arithmetic:
//   encoder 4 x (Linear -> Dropout(p = .5,.4,.3,.2) -> LeakyReLU)   [activation also on the latent]
//   decoder 3 x (Linear -> LeakyReLU -> BatchNorm1d) + Linear -> BatchNorm1d -> ReLU
// Dropout multiplies by the noise torch builds, bernoulli / (1 - p): 0 or the rounded float64 1 / (1 - p), in the
// forward and the backward pass.  BatchNorm in train mode normalises with the statistics of the whole batch (biased
// variance, eps 1e-5) and updates the float64 running statistics as torch does (momentum 0.1, unbiased variance).
// The batch is spread over CTAs of RT rows, so the kernel is launched cooperatively; the statistics are two passes
// (the mean, then the sum of squared deviations: no E[x^2] - mean^2 cancellation), each a per-CTA partial sum combined
// in CTA order after a grid-wide barrier, so a run is reproducible.  The backward pass needs one more barrier per
// BatchNorm for the batch sums of dy and dy * xhat; gamma / beta gradients are those totals.
struct F64DbnArgs {
  const void* x;
  int x_is_f64, batch_rows;
  int mode;                      // 0: train forward + backward, 1: eval forward (no dropout, running statistics), loss only
  double* act_g;
  double* dz_g;
  double* loss_part;
  double* bn_part;               // [12 slots][gridDim.x][2 * max_dim] partial sums
  double* rm;                    // running mean / var, bn_f_total each
  double* rv;
  long long* nbt;                // num_batches_tracked[4]
  double* bn_grad;               // split 0 of the gradient partials (the BatchNorm gamma / beta gradients land there)
  const unsigned char* mask[4];  // keep-masks [batch][N_l] (injected, or drawn from torch's stream) or nullptr (Philox)
  unsigned long long seed, step;
  double keep_scale[4];          // 1 / (1 - p) rounded, what noise.div_(1 - p) leaves in a kept element
};

__device__ __forceinline__ bool dbn_keep(const F64DbnArgs& a, int l, int grow, int j, int N) {
  if (a.mask[l] != nullptr) return a.mask[l][(size_t)grow * N + j] != 0;
  return bb_philox_keep(a.seed, a.step, l, grow, j);
}

// sum over the CTAs, in CTA order, of entry j of this barrier slot's partials
__device__ __forceinline__ double cta_total(const double* slot, int n_cta, int stride, int j) {
  double s = 0.0;
  for (int c = 0; c < n_cta; ++c) s = __dadd_rn(s, __ldcg(slot + (size_t)c * stride + j));
  return s;
}

__global__ void __launch_bounds__(NT_FB)
train_dbn_f64_kernel(const __grid_constant__ F64TrainLayout d, const double* __restrict__ params,
                     const double* __restrict__ wt, const __grid_constant__ F64DbnArgs a) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) double smem[];
  __shared__ double warp_loss[NT_FB / 32];
  double* act_s = smem;                                            // a_stride * RT
  double* dz_s0 = act_s + d.a_stride * RT;                         // max_dim * RT
  double* dz_s1 = dz_s0 + d.max_dim * RT;
  double* red_s = dz_s1 + d.max_dim * RT;                          // max(max_dim, NT_FB) * RT
  double* xhat_s = red_s + (d.max_dim > NT_FB ? d.max_dim : NT_FB) * RT;  // bn_f_total * RT: normalised BN inputs
  double* u_s = xhat_s + d.bn_f_total * RT;                        // bn_f_total * RT: BN inputs
  double* inv_s = u_s + d.bn_f_total * RT;                         // bn_f_total (+1): 1 / sqrt(var + eps)
  double* tot_s = inv_s + ((d.bn_f_total + 1) & ~1);               // 2 * max_dim: batch mean / batch sums
  const bool train = a.mode == 0;
  Stream s;
  s.ring = tot_s + 2 * d.max_dim;
  s.stage_elems = (KC * d.max_dim + 2 + 1) & ~1;
  s.n = 0;
  s.next_p = 0; s.next_i0 = 0;
  s.per_chain = train ? 2 * NL - 1 : NL;
  s.total = s.per_chain;
  issue_next(d, params, wt, s, 0);

  const int B = a.batch_rows;
  const int n_cta = gridDim.x;
  const int slot = 2 * d.max_dim;
  const int row0 = blockIdx.x * RT;
  const int rows = min(RT, B - row0);
  const int F = d.dims[0];
  for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
    const int r = o / F, j = o - r * F;
    double v = 0.0;
    if (r < rows) {
      const size_t e = (size_t)(row0 + r) * F + j;
      v = a.x_is_f64 ? __ldg(reinterpret_cast<const double*>(a.x) + e) : (double)__ldg(reinterpret_cast<const float*>(a.x) + e);
      a.act_g[(size_t)(row0 + r) * d.a_stride + j] = v;
    }
    act_s[j * RT + r] = v;
  }
  __syncthreads();

  // ---------------- forward: encoder
  for (int l = 0; l < 4; ++l) {
    int K, N;
    const double* src = pass_src(d, params, wt, l, K, N);
    const int KP = gemv_f64(d, params, wt, s, src, act_s + d.a_off[l] * RT, K, N, red_s);
    const double* bias = params + d.b_off[l];
    double* out_s = act_s + d.a_off[l + 1] * RT;
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      const int r = o / N, j = o - r * N;
      double v = __dadd_rn(red_sum(red_s, KP, N, r, j), __ldg(bias + j));
      if (train && r < rows) v = __dmul_rn(v, dbn_keep(a, l, row0 + r, j, N) ? a.keep_scale[l] : 0.0);
      v = act_fwd(v, BB_ACT_LEAKY);
      out_s[j * RT + r] = v;
      if (r < rows) a.act_g[(size_t)(row0 + r) * d.a_stride + d.a_off[l + 1] + j] = v;
    }
    __syncthreads();
  }
  // ---------------- forward: decoder with BatchNorm
  for (int i = 0; i < 4; ++i) {
    const int l = 4 + i, fo = d.bn_f_off[i];
    int K, N;
    const double* src = pass_src(d, params, wt, l, K, N);
    const int KP = gemv_f64(d, params, wt, s, src, act_s + d.a_off[l] * RT, K, N, red_s);
    const double* bias = params + d.b_off[l];
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      const int r = o / N, j = o - r * N;
      double v = __dadd_rn(red_sum(red_s, KP, N, r, j), __ldg(bias + j));
      if (i < 3) v = act_fwd(v, BB_ACT_LEAKY);
      u_s[(fo + j) * RT + r] = r < rows ? v : 0.0;
    }
    __syncthreads();
    if (train) {
      double* part = a.bn_part + ((size_t)(2 * i) * n_cta + blockIdx.x) * slot;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        double s1 = 0.0;
        for (int r = 0; r < rows; ++r) s1 = __dadd_rn(s1, u_s[(fo + j) * RT + r]);
        part[j] = s1;
      }
      __threadfence();
      grid.sync();
      const double* all = a.bn_part + (size_t)(2 * i) * n_cta * slot;
      for (int j = threadIdx.x; j < N; j += NT_FB) tot_s[j] = __ddiv_rn(cta_total(all, n_cta, slot, j), (double)B);
      __syncthreads();
      part = a.bn_part + ((size_t)(2 * i + 1) * n_cta + blockIdx.x) * slot;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        double s2 = 0.0;
        for (int r = 0; r < rows; ++r) {
          const double dv = __dsub_rn(u_s[(fo + j) * RT + r], tot_s[j]);
          s2 = __dadd_rn(s2, __dmul_rn(dv, dv));
        }
        part[j] = s2;
      }
      __threadfence();
      grid.sync();
      all = a.bn_part + (size_t)(2 * i + 1) * n_cta * slot;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        const double m2 = cta_total(all, n_cta, slot, j);
        inv_s[fo + j] = __ddiv_rn(1.0, __dsqrt_rn(__dadd_rn(__ddiv_rn(m2, (double)B), 1e-5)));
        if (blockIdx.x == 0) {  // running statistics: momentum * batch + (1 - momentum) * running, unbiased variance
          const double unbiased = __ddiv_rn(m2, (double)(B > 1 ? B - 1 : 1));
          a.rm[fo + j] = __dadd_rn(__dmul_rn(0.1, tot_s[j]), __dmul_rn(1.0 - 0.1, a.rm[fo + j]));
          a.rv[fo + j] = __dadd_rn(__dmul_rn(0.1, unbiased), __dmul_rn(1.0 - 0.1, a.rv[fo + j]));
          if (j == 0) a.nbt[i] += 1;
        }
      }
    } else {
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        tot_s[j] = a.rm[fo + j];
        inv_s[fo + j] = __ddiv_rn(1.0, __dsqrt_rn(__dadd_rn(a.rv[fo + j], 1e-5)));
      }
    }
    __syncthreads();
    const double* gam = params + d.bn_g_off[i];
    const double* bet = params + d.bn_b_off[i];
    double* out_s = act_s + d.a_off[l + 1] * RT;
    for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
      const int r = o / N, j = o - r * N;
      const double xh = __dmul_rn(__dsub_rn(u_s[(fo + j) * RT + r], tot_s[j]), inv_s[fo + j]);
      double h = __dadd_rn(__dmul_rn(xh, __ldg(gam + j)), __ldg(bet + j));
      if (i == 3) h = act_fwd(h, BB_ACT_RELU);
      xhat_s[(fo + j) * RT + r] = xh;
      out_s[j * RT + r] = h;
      if (r < rows && l + 1 < NL) a.act_g[(size_t)(row0 + r) * d.a_stride + d.a_off[l + 1] + j] = h;
    }
    __syncthreads();
  }
  // ---------------- loss and the seed gradient (through the final ReLU)
  double loss_local = 0.0;
  double* dz_cur = dz_s0;
  double* dz_nxt = dz_s1;
  {
    const double* out_s = act_s + d.a_off[NL] * RT;
    for (int o = threadIdx.x; o < RT * F; o += NT_FB) {
      const int r = o / F, j = o - r * F;
      double g = 0.0;
      if (r < rows) {
        const double rec = out_s[j * RT + r];
        const double diff = __dsub_rn(rec, act_s[j * RT + r]);
        loss_local = __dadd_rn(loss_local, __ddiv_rn(__dmul_rn(diff, diff), (double)F));
        g = rec > 0.0 ? __ddiv_rn(__dmul_rn(2.0, diff), (double)F) : 0.0;
      }
      dz_cur[j * RT + r] = g;
    }
    __syncthreads();
  }
  if (train) {
    // ---------------- backward: decoder (dz_cur = gradient w.r.t. the BatchNorm output)
    for (int i = 3; i >= 0; --i) {
      const int l = 4 + i, fo = d.bn_f_off[i];
      const int N = d.dims[l + 1];
      double* part = a.bn_part + ((size_t)(8 + 3 - i) * n_cta + blockIdx.x) * slot;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        double t1 = 0.0, t2 = 0.0;
        for (int r = 0; r < rows; ++r) {
          const double g = dz_cur[j * RT + r];
          t1 = __dadd_rn(t1, g);
          t2 = __dadd_rn(t2, __dmul_rn(g, xhat_s[(fo + j) * RT + r]));
        }
        part[j] = t1; part[N + j] = t2;
      }
      __threadfence();
      grid.sync();
      const double* all = a.bn_part + (size_t)(8 + 3 - i) * n_cta * slot;
      for (int j = threadIdx.x; j < N; j += NT_FB) {
        const double T1 = cta_total(all, n_cta, slot, j), T2 = cta_total(all, n_cta, slot, N + j);
        tot_s[j] = __ddiv_rn(T1, (double)B);
        tot_s[d.max_dim + j] = __ddiv_rn(T2, (double)B);
        if (blockIdx.x == 0) { a.bn_grad[d.bn_b_off[i] + j] = T1; a.bn_grad[d.bn_g_off[i] + j] = T2; }
      }
      __syncthreads();
      const double* gam = params + d.bn_g_off[i];
      for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
        const int r = o / N, j = o - r * N;
        // torch's batch-norm backward: dx = (dy - mean(dy) - xhat * mean(dy * xhat)) * invstd * gamma
        double dx = __dsub_rn(__dsub_rn(dz_cur[j * RT + r], tot_s[j]), __dmul_rn(xhat_s[(fo + j) * RT + r], tot_s[d.max_dim + j]));
        dx = __dmul_rn(__dmul_rn(dx, inv_s[fo + j]), __ldg(gam + j));
        if (i < 3 && !(u_s[(fo + j) * RT + r] > 0.0)) dx = __dmul_rn(dx, 0.01);
        if (r >= rows) dx = 0.0;
        dz_nxt[j * RT + r] = dx;
        if (r < rows) a.dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[l] + j] = dx;
      }
      __syncthreads();
      {  // dX = dZ W_l: the gradient w.r.t. the output of the previous block
        int Nn, K;
        const double* src = pass_src(d, params, wt, 2 * NL - 1 - l, Nn, K);
        const int KP = gemv_f64(d, params, wt, s, src, dz_nxt, Nn, K, red_s);
        for (int o = threadIdx.x; o < RT * K; o += NT_FB) {
          const int r = o / K, j = o - r * K;
          dz_cur[j * RT + r] = red_sum(red_s, KP, K, r, j);
        }
        __syncthreads();
      }
    }
    // ---------------- backward: encoder (dz_cur = gradient w.r.t. the output of encoder layer l)
    for (int l = 3; l >= 0; --l) {
      const int N = d.dims[l + 1];
      const double* a_out = act_s + d.a_off[l + 1] * RT;
      for (int o = threadIdx.x; o < RT * N; o += NT_FB) {
        const int r = o / N, j = o - r * N;
        double g = 0.0;
        if (r < rows) {
          g = dz_cur[j * RT + r];
          if (!(a_out[j * RT + r] > 0.0)) g = __dmul_rn(g, 0.01);
          g = __dmul_rn(g, dbn_keep(a, l, row0 + r, j, N) ? a.keep_scale[l] : 0.0);
          a.dz_g[(size_t)(row0 + r) * d.z_stride + d.z_off[l] + j] = g;
        }
        dz_nxt[j * RT + r] = g;
      }
      __syncthreads();
      if (l >= 1) {
        int Nn, K;
        const double* src = pass_src(d, params, wt, 2 * NL - 1 - l, Nn, K);
        const int KP = gemv_f64(d, params, wt, s, src, dz_nxt, Nn, K, red_s);
        for (int o = threadIdx.x; o < RT * K; o += NT_FB) {
          const int r = o / K, j = o - r * K;
          dz_cur[j * RT + r] = red_sum(red_s, KP, K, r, j);
        }
        __syncthreads();
      }
    }
  }
  cp_async_wait_all();
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) loss_local = __dadd_rn(loss_local, __shfl_xor_sync(0xffffffffu, loss_local, off));
  if ((threadIdx.x & 31) == 0) warp_loss[threadIdx.x >> 5] = loss_local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int w = 0; w < NT_FB / 32; ++w) v = __dadd_rn(v, warp_loss[w]);
    a.loss_part[blockIdx.x] = v;
  }
}

// partial[split][w_off[l] + n * K + k] = sum_{r in split} dZ_l[r][n] * A_l[r][k]  (+ the second chain), b likewise
__global__ void __launch_bounds__(NT)
train_dw_f64_kernel(const __grid_constant__ F64TrainLayout d, const Tile* __restrict__ tiles, const double* __restrict__ act_g,
                    const double* __restrict__ dz_g, const size_t chain_act_stride, const size_t chain_dz_stride,
                    const int n_chains, const int batch_rows, double* __restrict__ partial) {
  __shared__ __align__(16) double dz_s[DW_R][DW_LD];
  __shared__ __align__(16) double a_s[DW_R][DW_LD];
  pdl_launch_dependents();
  pdl_wait();  // activations and dZ come from the forward / backward kernel
  const Tile tile = tiles[blockIdx.x];
  const int l = tile.l, N = d.dims[l + 1], K = d.dims[l];
  const int tn = threadIdx.x >> 4, tk = threadIdx.x & 15;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  double bsum = 0.0;
  for (int c = 0; c < n_chains; ++c) {
    const double* dz = dz_g + c * chain_dz_stride + d.z_off[l];
    const double* a = act_g + c * chain_act_stride + d.a_off[l];
    for (int h = 0; h < DW_T; h += DW_R) {
      const int r0 = blockIdx.y * DW_T + h;
      const int rows = min(DW_R, batch_rows - r0);
      __syncthreads();  // the previous half is no longer read
      for (int e = threadIdx.x; e < DW_R * DW_T; e += NT) {
        const int rr = e >> 6, cc = e & 63;
        const bool rv = rr < rows;
        dz_s[rr][cc] = (rv && tile.n0 + cc < N) ? __ldg(dz + (size_t)(r0 + rr) * d.z_stride + tile.n0 + cc) : 0.0;
        a_s[rr][cc] = (rv && tile.k0 + cc < K) ? __ldg(a + (size_t)(r0 + rr) * d.a_stride + tile.k0 + cc) : 0.0;
      }
      __syncthreads();
      for (int rr = 0; rr < DW_R; ++rr) {
        const double2 d0 = *reinterpret_cast<const double2*>(&dz_s[rr][tn * 4]);
        const double2 d1 = *reinterpret_cast<const double2*>(&dz_s[rr][tn * 4 + 2]);
        const double2 a0 = *reinterpret_cast<const double2*>(&a_s[rr][tk * 4]);
        const double2 a1 = *reinterpret_cast<const double2*>(&a_s[rr][tk * 4 + 2]);
        const double dd[4] = {d0.x, d0.y, d1.x, d1.y}, aa[4] = {a0.x, a0.y, a1.x, a1.y};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fma(dd[i], aa[j], acc[i][j]);
      }
      if (tile.k0 == 0 && threadIdx.x < DW_T)
        for (int rr = 0; rr < DW_R; ++rr) bsum = __dadd_rn(bsum, dz_s[rr][threadIdx.x]);
    }
  }
  double* out = partial + (size_t)blockIdx.y * d.n_params;
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

struct AdamArgs {
  double step_size;  // lr / (1 - beta1^t)
  double sqrt_bc2;   // sqrt(1 - beta2^t)
  double beta2, one_m_beta1, one_m_beta2, eps;
};

// mode 0: grads = sum of partials, then Adam.  mode 1: grads = sum of partials only (+ loss slot).
// mode 2: Adam from grads (after the caller's all-reduce).  torch.optim.Adam, single-tensor, in its operation order:
//   m.lerp_(g, 1 - b1); v.mul_(b2).addcmul_(g, g, 1 - b2); denom = v.sqrt() / sqrt(bc2) + eps; p.addcdiv_(m, denom, -lr / bc1)
__global__ void __launch_bounds__(NT)
train_adam_f64_kernel(const int n_params, const int mode, const double* __restrict__ partial, const int n_splits,
                      double* __restrict__ grads, double* __restrict__ params, double* __restrict__ wt,
                      const int* __restrict__ wt_index, double* __restrict__ m, double* __restrict__ v, const AdamArgs a,
                      const double* __restrict__ loss_part, const int n_loss_parts, double* __restrict__ loss_accum) {
  pdl_launch_dependents();
  pdl_wait();  // gradient partials come from the dW kernel
  const int p = blockIdx.x * NT + threadIdx.x;
  if (p < n_params) {
    double g;
    if (mode == 2) {
      g = grads[p];
    } else {
      g = 0.0;
      for (int s = 0; s < n_splits; ++s) g = __dadd_rn(g, __ldg(partial + (size_t)s * n_params + p));
      grads[p] = g;
    }
    if (mode != 1) {
      const double mm = __dadd_rn(m[p], __dmul_rn(__dsub_rn(g, m[p]), a.one_m_beta1));
      const double vv = __dadd_rn(__dmul_rn(v[p], a.beta2), __dmul_rn(__dmul_rn(a.one_m_beta2, g), g));
      m[p] = mm;
      v[p] = vv;
      const double denom = __dadd_rn(__ddiv_rn(__dsqrt_rn(vv), a.sqrt_bc2), a.eps);
      const double np = __dsub_rn(params[p], __ddiv_rn(__dmul_rn(a.step_size, mm), denom));
      params[p] = np;
      const int wi = wt_index[p];
      if (wi >= 0) wt[wi] = np;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (mode != 2) {
      double s = 0.0;
      for (int i = 0; i < n_loss_parts; ++i) s = __dadd_rn(s, loss_part[i]);
      grads[n_params] = s;  // the loss rides in the last slot so one all-reduce covers it
    }
    if (mode != 1 && loss_accum) *loss_accum = __dadd_rn(*loss_accum, grads[n_params]);
  }
}

}  // namespace

struct F64Trainer {
  F64TrainLayout d;
  int max_batch = 0, n_tiles = 0, last_rows = 0;
  size_t smem_bytes = 0;
  double *params = nullptr, *wt = nullptr, *grads = nullptr, *m = nullptr, *v = nullptr;
  double *act_g = nullptr, *dz_g = nullptr, *partial = nullptr, *loss_part = nullptr;
  int* wt_index = nullptr;
  Tile* tiles = nullptr;
  // AE_Dropout_BN
  double *bn_part = nullptr, *rm = nullptr, *rv = nullptr;
  long long* nbt = nullptr;
  size_t dbn_smem = 0;
  int dbn_max_ctas = 0;
  const unsigned char* mask_dev[4] = {nullptr, nullptr, nullptr, nullptr};
  unsigned long long seed = 0;
  // torch's stream: the twister state (624 words + position) and two mask slots [rows][sum N_l] filled on a side stream
  bool mt_armed = false;
  uint32_t* mt_state = nullptr;
  unsigned char* mt_slot[2] = {nullptr, nullptr};
  cudaStream_t mt_stream = nullptr;
  cudaEvent_t mt_ready[2] = {nullptr, nullptr}, mt_free[2] = {nullptr, nullptr};
  long long mt_draws = 0;
};

void bb_f64_train_destroy(F64Trainer* f) {
  if (!f) return;
  if (f->mt_stream) cudaStreamSynchronize(f->mt_stream);
  void* ptrs[] = {f->params, f->wt, f->grads, f->m, f->v, f->act_g, f->dz_g, f->partial, f->loss_part, f->wt_index, f->tiles,
                  f->bn_part, f->rm, f->rv, f->nbt, f->mt_state, f->mt_slot[0], f->mt_slot[1]};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  for (int i = 0; i < 2; ++i) {
    if (f->mt_ready[i]) cudaEventDestroy(f->mt_ready[i]);
    if (f->mt_free[i]) cudaEventDestroy(f->mt_free[i]);
  }
  if (f->mt_stream) cudaStreamDestroy(f->mt_stream);
  delete f;
}

int bb_f64_train_create(bb_ctx* ctx, const F64TrainLayout& d, const double* params_host, const double* bn_stats_host,
                        const long long* nbt_host, int max_batch, F64Trainer** out) {
  if (!ctx || !params_host || !out || max_batch < 1) return BB_ERR_INVALID;
  if (d.kind == 1 && (!bn_stats_host || !nbt_host)) return BB_ERR_INVALID;
  if (d.max_dim > NT_FB) return BB_ERR_UNSUPPORTED;
  const size_t stage = (size_t)((KC * d.max_dim + 2 + 1) & ~1);
  const size_t smem = ((size_t)(d.a_stride + 2 * d.max_dim + (d.max_dim > NT_FB ? d.max_dim : NT_FB)) * RT + 2 * stage) * sizeof(double);
  if (smem > ctx->smem_optin) return BB_ERR_UNSUPPORTED;
  F64Trainer* f = new (std::nothrow) F64Trainer();
  if (!f) return BB_ERR_NOMEM;
  f->d = d;
  f->max_batch = max_batch;
  f->smem_bytes = smem;
  const int p = d.n_params;
  std::vector<double> hwt(p, 0.0);
  std::vector<int> hidx(p, -1);
  std::vector<Tile> tiles;
  int wtn = 0;
  for (int l = 0; l < NL; ++l) {
    const int K = d.dims[l], N = d.dims[l + 1];
    for (int n = 0; n < N; ++n)
      for (int k = 0; k < K; ++k) {
        hwt[d.wt_off[l] + k * N + n] = params_host[d.w_off[l] + n * K + k];
        hidx[d.w_off[l] + n * K + k] = d.wt_off[l] + k * N + n;
      }
    wtn += K * N;
    for (int n0 = 0; n0 < N; n0 += DW_T)
      for (int k0 = 0; k0 < K; k0 += DW_T) tiles.push_back({l, n0, k0});
  }
  f->n_tiles = (int)tiles.size();
  const int max_splits = (max_batch + DW_T - 1) / DW_T;
  const int max_ctas = (max_batch + RT - 1) / RT;
  int rc = BB_OK;
  auto alloc = [&](void** ptr, size_t bytes) { if (rc == BB_OK) rc = (int)cudaMalloc(ptr, bytes); };
  // (+ 8 doubles: a chunk copy aligned down to 16 bytes may read one double past its matrix)
  alloc((void**)&f->params, sizeof(double) * (p + 8));
  alloc((void**)&f->wt, sizeof(double) * (wtn + 8));
  alloc((void**)&f->grads, sizeof(double) * (p + 1));
  alloc((void**)&f->m, sizeof(double) * p);
  alloc((void**)&f->v, sizeof(double) * p);
  alloc((void**)&f->act_g, sizeof(double) * 2 * (size_t)max_batch * d.a_stride);
  alloc((void**)&f->dz_g, sizeof(double) * 2 * (size_t)max_batch * d.z_stride);
  alloc((void**)&f->partial, sizeof(double) * (size_t)max_splits * p);
  alloc((void**)&f->loss_part, sizeof(double) * max_ctas);
  alloc((void**)&f->wt_index, sizeof(int) * p);
  alloc((void**)&f->tiles, sizeof(Tile) * tiles.size());
  if (rc == BB_OK) rc = (int)cudaMemset(f->params, 0, sizeof(double) * (p + 8));
  if (rc == BB_OK) rc = (int)cudaMemset(f->wt, 0, sizeof(double) * (wtn + 8));
  if (rc == BB_OK) rc = (int)cudaMemcpy(f->params, params_host, sizeof(double) * p, cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemcpy(f->wt, hwt.data(), sizeof(double) * wtn, cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemcpy(f->wt_index, hidx.data(), sizeof(int) * p, cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemcpy(f->tiles, tiles.data(), sizeof(Tile) * tiles.size(), cudaMemcpyHostToDevice);
  if (rc == BB_OK) rc = (int)cudaMemset(f->m, 0, sizeof(double) * p);
  if (rc == BB_OK) rc = (int)cudaMemset(f->v, 0, sizeof(double) * p);
  if (rc == BB_OK) rc = (int)cudaMemset(f->grads, 0, sizeof(double) * (p + 1));
  // the BatchNorm entries of splits > 0 stay zero: the dW kernel writes Linear entries only
  if (rc == BB_OK) rc = (int)cudaMemset(f->partial, 0, sizeof(double) * (size_t)max_splits * p);
  if (rc == BB_OK)
    rc = (int)cudaFuncSetAttribute(train_fwd_bwd_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (rc == BB_OK && d.kind == 1) {
    const int nb = d.bn_f_total;
    alloc((void**)&f->bn_part, sizeof(double) * 12 * (size_t)max_ctas * 2 * d.max_dim);
    alloc((void**)&f->rm, sizeof(double) * nb);
    alloc((void**)&f->rv, sizeof(double) * nb);
    alloc((void**)&f->nbt, sizeof(long long) * 4);
    if (rc == BB_OK) rc = (int)cudaMemcpy(f->rm, bn_stats_host, sizeof(double) * nb, cudaMemcpyHostToDevice);
    if (rc == BB_OK) rc = (int)cudaMemcpy(f->rv, bn_stats_host + nb, sizeof(double) * nb, cudaMemcpyHostToDevice);
    if (rc == BB_OK) rc = (int)cudaMemcpy(f->nbt, nbt_host, sizeof(long long) * 4, cudaMemcpyHostToDevice);
    f->dbn_smem = smem + ((size_t)2 * nb * RT + ((nb + 1) & ~1) + 2 * d.max_dim) * sizeof(double);
    if (rc == BB_OK && f->dbn_smem > ctx->smem_optin) rc = BB_ERR_UNSUPPORTED;
    if (rc == BB_OK)
      rc = (int)cudaFuncSetAttribute(train_dbn_f64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)f->dbn_smem);
    int per_sm = 0;
    if (rc == BB_OK) rc = (int)cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, train_dbn_f64_kernel, NT_FB, f->dbn_smem);
    f->dbn_max_ctas = per_sm * ctx->sm_count;
  }
  if (rc == BB_OK) rc = (int)cudaDeviceSynchronize();
  if (rc != BB_OK) { bb_f64_train_destroy(f); return rc; }
  *out = f;
  return BB_OK;
}

namespace {
int launch_fwd(F64Trainer* f, const void* x, int x_is_f64, int rows, int backward, const bb_train_hyper* h, cudaStream_t s) {
  const int world = h && h->world_size > 0 ? h->world_size : 1;
  const double reg_inv_rows = h ? h->reg_param / ((double)rows * world) : 0.0;
  f->last_rows = rows;
  return (int)pdl_launch(train_fwd_bwd_f64_kernel, dim3((rows + RT - 1) / RT), dim3(NT_FB), f->smem_bytes, s, f->d, f->params,
                         f->wt, x, x_is_f64, rows, f->act_g, f->dz_g, (size_t)f->max_batch * f->d.a_stride,
                         (size_t)f->max_batch * f->d.z_stride, backward, h ? h->l1 : 0, reg_inv_rows, f->loss_part);
}

// the keep-masks of this batch from torch's stream: drawn on the side stream into the slot the step before last read
int draw_mt(F64Trainer* f, int rows, const unsigned char** masks, cudaStream_t s) {
  const int k = (int)(f->mt_draws & 1);
  int widths[4], tot = 0;
  unsigned char* out[4];
  for (int l = 0; l < 4; ++l) {
    widths[l] = f->d.dims[l + 1];
    out[l] = f->mt_slot[k] + (size_t)rows * tot;
    masks[l] = out[l];
    tot += widths[l];
  }
  const double keep[4] = {1.0 - 0.5, 1.0 - 0.4, 1.0 - 0.3, 1.0 - 0.2};  // models.py:263-275
  BB_CUDA(cudaStreamWaitEvent(f->mt_stream, f->mt_free[k], 0));
  int rc = bb_mt_dropout_launch(f->mt_state, rows, widths, keep, out, f->mt_stream);
  if (rc != BB_OK) return rc;
  BB_CUDA(cudaEventRecord(f->mt_ready[k], f->mt_stream));
  BB_CUDA(cudaStreamWaitEvent(s, f->mt_ready[k], 0));
  ++f->mt_draws;
  return BB_OK;
}

int launch_dbn(F64Trainer* f, const void* x, int x_is_f64, int rows, int mode, long long step, cudaStream_t s) {
  const int grid = (rows + RT - 1) / RT;
  if (grid > f->dbn_max_ctas) return BB_ERR_UNSUPPORTED;  // cooperative launch: every CTA must be resident
  f->last_rows = rows;
  F64DbnArgs a;
  a.x = x; a.x_is_f64 = x_is_f64; a.batch_rows = rows; a.mode = mode;
  a.act_g = f->act_g; a.dz_g = f->dz_g; a.loss_part = f->loss_part; a.bn_part = f->bn_part;
  a.rm = f->rm; a.rv = f->rv; a.nbt = f->nbt; a.bn_grad = f->partial;
  for (int i = 0; i < 4; ++i) a.mask[i] = f->mask_dev[i];
  a.seed = f->seed; a.step = (unsigned long long)step;
  const double p[4] = {0.5, 0.4, 0.3, 0.2};
  for (int i = 0; i < 4; ++i) a.keep_scale[i] = 1.0 / (1.0 - p[i]);
  const bool mt = mode == 0 && f->mt_armed;
  if (mt) {
    const int rc = draw_mt(f, rows, a.mask, s);
    if (rc != BB_OK) return rc;
  }
  void* args[] = {(void*)&f->d, (void*)&f->params, (void*)&f->wt, (void*)&a};
  BB_CUDA(cudaLaunchCooperativeKernel((const void*)train_dbn_f64_kernel, dim3(grid), dim3(NT_FB), args, f->dbn_smem, s));
  if (mt) BB_CUDA(cudaEventRecord(f->mt_free[(f->mt_draws - 1) & 1], s));
  return BB_OK;
}
}  // namespace

int bb_f64_train_step(F64Trainer* f, const void* x_dev, int x_is_f64, int rows, const bb_train_hyper* h, int phase,
                      long long step, double* loss_accum_dev, cudaStream_t s) {
  if (!f || !h || !x_dev || rows < 1 || rows > f->max_batch || phase < 0 || phase > 2) return BB_ERR_INVALID;
  const int p = f->d.n_params;
  const int n_splits = (rows + DW_T - 1) / DW_T;
  if (phase != 2) {
    int rc;
    if (f->d.kind == 1) {
      // AE_Dropout_BN: MSE only; the Philox counter takes the step the kernel's update will be (bb_train.cu's t->step)
      if (h->l1) return BB_ERR_UNSUPPORTED;
      rc = launch_dbn(f, x_dev, x_is_f64, rows, 0, phase == 0 ? step - 1 : step, s);
    } else {
      rc = launch_fwd(f, x_dev, x_is_f64, rows, 1, h, s);
    }
    if (rc != BB_OK) return rc;
    BB_CUDA(pdl_launch(train_dw_f64_kernel, dim3(f->n_tiles, n_splits), dim3(NT), 0, s, f->d, f->tiles, f->act_g, f->dz_g,
                       (size_t)f->max_batch * f->d.a_stride, (size_t)f->max_batch * f->d.z_stride, h->l1 ? 2 : 1, rows,
                       f->partial));
  }
  AdamArgs a = {};
  if (phase != 1) {
    // Python floats: bias_correction1 = 1 - beta1 ** step, step_size = lr / bc1, sqrt(1 - beta2 ** step)
    a.step_size = h->lr / (1.0 - std::pow(h->beta1, (double)step));
    a.sqrt_bc2 = std::sqrt(1.0 - std::pow(h->beta2, (double)step));
    a.beta2 = h->beta2;
    a.one_m_beta1 = 1.0 - h->beta1;
    a.one_m_beta2 = 1.0 - h->beta2;
    a.eps = h->eps;
  }
  return (int)pdl_launch(train_adam_f64_kernel, dim3((p + NT - 1) / NT), dim3(NT), 0, s, p, phase, (const double*)f->partial,
                         n_splits, f->grads, f->params, f->wt, (const int*)f->wt_index, f->m, f->v, a,
                         (const double*)f->loss_part, (rows + RT - 1) / RT, loss_accum_dev);
}

int bb_f64_train_eval(F64Trainer* f, const void* x_dev, int x_is_f64, int rows, double* loss_accum_dev, cudaStream_t s) {
  if (!f || !x_dev || rows < 1 || rows > f->max_batch) return BB_ERR_INVALID;
  int rc = f->d.kind == 1 ? launch_dbn(f, x_dev, x_is_f64, rows, 1, 0, s) : launch_fwd(f, x_dev, x_is_f64, rows, 0, nullptr, s);
  if (rc != BB_OK) return rc;
  const AdamArgs a = {};
  // mode 1 with zero parameters only folds the loss partials into the gradient's loss slot ...
  train_adam_f64_kernel<<<1, NT, 0, s>>>(0, 1, nullptr, 0, f->grads + f->d.n_params, nullptr, nullptr, nullptr, nullptr,
                                         nullptr, a, f->loss_part, (rows + RT - 1) / RT, nullptr);
  // ... and mode 2 with zero parameters adds that slot to the accumulator
  train_adam_f64_kernel<<<1, NT, 0, s>>>(0, 2, nullptr, 0, f->grads + f->d.n_params, nullptr, nullptr, nullptr, nullptr,
                                         nullptr, a, nullptr, 0, loss_accum_dev);
  return (int)cudaGetLastError();
}

int bb_f64_train_activation_means(F64Trainer* f, double* out) {
  if (!f || !out) return BB_ERR_INVALID;
  const int rows = f->last_rows, stride = f->d.a_stride;
  std::vector<double> h((size_t)rows * stride);
  if (rows) BB_CUDA(cudaMemcpy(h.data(), f->act_g, h.size() * sizeof(double), cudaMemcpyDeviceToHost));
  const int layers[6] = {1, 2, 3, 5, 6, 7};  // A_l = LeakyReLU(output of Linear l - 1)
  for (int i = 0; i < 6; ++i) {
    const int l = layers[i], n = f->d.dims[l];
    for (int j = 0; j < 200; ++j) {
      double s = NAN;
      if (j < n && rows) {
        s = 0.0;
        for (int r = 0; r < rows; ++r) s += h[(size_t)r * stride + f->d.a_off[l] + j];
        s /= rows;
      }
      out[i * 200 + j] = s;
    }
  }
  return BB_OK;
}

int bb_f64_train_get_params(F64Trainer* f, double* params_host) {
  if (!f || !params_host) return BB_ERR_INVALID;
  BB_CUDA(cudaMemcpy(params_host, f->params, sizeof(double) * f->d.n_params, cudaMemcpyDeviceToHost));
  return BB_OK;
}

double* bb_f64_train_params(F64Trainer* f) { return f ? f->params : nullptr; }
double* bb_f64_train_grads(F64Trainer* f) { return f ? f->grads : nullptr; }

int bb_f64_train_set_dropout(F64Trainer* f, unsigned long long seed, const unsigned char* const* masks_dev) {
  if (!f || f->d.kind != 1) return BB_ERR_INVALID;
  f->seed = seed;
  for (int i = 0; i < 4; ++i) f->mask_dev[i] = masks_dev ? masks_dev[i] : nullptr;
  f->mt_armed = false;
  return BB_OK;
}

int bb_f64_train_set_mt19937(F64Trainer* f, const uint32_t* key_624, int pos) {
  if (!f || f->d.kind != 1 || !key_624 || pos < 0 || pos > 624) return BB_ERR_INVALID;
  int rc = BB_OK;
  if (!f->mt_stream) {
    rc = (int)cudaStreamCreateWithFlags(&f->mt_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && rc == BB_OK; ++i) {
      rc = (int)cudaEventCreateWithFlags(&f->mt_ready[i], cudaEventDisableTiming);
      if (rc == BB_OK) rc = (int)cudaEventCreateWithFlags(&f->mt_free[i], cudaEventDisableTiming);
    }
    size_t per_row = 0;
    for (int l = 0; l < 4; ++l) per_row += f->d.dims[l + 1];
    if (rc == BB_OK) rc = (int)cudaMalloc((void**)&f->mt_state, sizeof(uint32_t) * 625);
    for (int i = 0; i < 2 && rc == BB_OK; ++i) rc = (int)cudaMalloc((void**)&f->mt_slot[i], per_row * f->max_batch);
    if (rc != BB_OK) return rc;
  }
  uint32_t h[625];
  memcpy(h, key_624, sizeof(uint32_t) * 624);
  h[624] = (uint32_t)pos;
  BB_CUDA(cudaMemcpyAsync(f->mt_state, h, sizeof(h), cudaMemcpyHostToDevice, f->mt_stream));
  BB_CUDA(cudaStreamSynchronize(f->mt_stream));
  for (int i = 0; i < 4; ++i) f->mask_dev[i] = nullptr;
  f->mt_armed = true;
  return BB_OK;
}

int bb_f64_train_get_mt19937(F64Trainer* f, uint32_t* key_624, int* pos) {
  if (!f || !key_624 || !pos) return BB_ERR_INVALID;
  if (!f->mt_armed) return BB_ERR_INVALID;
  uint32_t h[625];
  BB_CUDA(cudaMemcpyAsync(h, f->mt_state, sizeof(h), cudaMemcpyDeviceToHost, f->mt_stream));
  BB_CUDA(cudaStreamSynchronize(f->mt_stream));
  memcpy(key_624, h, sizeof(uint32_t) * 624);
  *pos = (int)h[624];
  return BB_OK;
}

int bb_f64_train_bn_running(F64Trainer* f, double** rm_dev, double** rv_dev) {
  if (!f || f->d.kind != 1 || !rm_dev || !rv_dev) return BB_ERR_INVALID;
  *rm_dev = f->rm; *rv_dev = f->rv;
  return BB_OK;
}

int bb_f64_train_get_bn_stats(F64Trainer* f, double* rm_host, double* rv_host, long long* nbt_host) {
  if (!f || f->d.kind != 1 || !rm_host || !rv_host || !nbt_host) return BB_ERR_INVALID;
  BB_CUDA(cudaMemcpy(rm_host, f->rm, sizeof(double) * f->d.bn_f_total, cudaMemcpyDeviceToHost));
  BB_CUDA(cudaMemcpy(rv_host, f->rv, sizeof(double) * f->d.bn_f_total, cudaMemcpyDeviceToHost));
  BB_CUDA(cudaMemcpy(nbt_host, f->nbt, sizeof(long long) * 4, cudaMemcpyDeviceToHost));
  return BB_OK;
}

int bb_f64_train_dbn_max_ctas(F64Trainer* f) { return f ? f->dbn_max_ctas : 0; }
