// Internal definitions shared by the baler_b200 CUDA translation units (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <functional>
#include <vector>

#include "../../include/baler_b200.h"

#define BB_CUDA(expr)                          \
  do {                                         \
    cudaError_t _e = (expr);                   \
    if (_e != cudaSuccess) return (int)_e;     \
  } while (0)

constexpr int BB_MAX_LAYERS = 8;
constexpr float BB_LEAKY = 0.01f;

struct bb_ctx {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;  // max dynamic shared memory per block
  float* minmax_scratch = nullptr;  // [2][blocks][cols] partials of the column min/max pass
  size_t minmax_scratch_bytes = 0;
  unsigned int* minmax_counter = nullptr;
};

// One dense layer of a fused chain as the fp32 kernel sees it.
struct ChainLayer {
  int K, N, Npad;  // in features, out features, out features padded to the thread tile
  int act;         // BB_ACT_*
  int tn;          // columns per thread tile: 8, 4, 2 or 1
  int w_off;       // float offset of Wt[K][Npad] (k-major) in the weight blob
  int b_off;       // float offset of bias[Npad]
};

struct ChainDesc {
  int n_layers;
  int in_dim, out_dim;
  int blob_floats;     // size of the fp32 weight blob
  int buf_rows[2];     // rows ([feature] index) of the two ping-pong activation buffers
  ChainLayer layer[BB_MAX_LAYERS];
};

// One layer / one direction of the float64 chain (bb_chain_f64.cu); filled lazily by bb_chain_f64_prepare.
struct F64Layer {
  int K, Kpad, N, Npad;  // in features (padded to whole weight chunks), out features (padded to the thread tile)
  int act, tn;           // BB_ACT_*, columns per thread
  int w_off, b_off;      // double offsets of Wt[Kpad][Npad] (k-major, zero padded) and bias[Npad] in the blob
};
struct F64Desc {
  int n_layers, in_dim, out_dim;
  int tr;              // rows per tile (64 or 32)
  int max_npad;        // widest padded layer: row length of the weight ring
  int buf_rows[2];     // rows ([feature] index) of the two ping-pong activation buffers
  F64Layer layer[BB_MAX_LAYERS];
};

// Launch plan of the statically shaped tcgen05 kernel (bb_chain_tc4.cu); filled by bb_tc_prepare.
struct Tc4Plan {
  bool ok = false;
  int enc = 0, ka = 0, nl = 0;  // direction, padded K of the first layer, padded N of the last layer
  float c1[4] = {0, 0, 0, 0}, c2[4] = {0, 0, 0, 0};  // y = c1 * acc + c2 * |acc| per layer
};

// Kernel that ran a direction's last launch (Chain::last_route; read back by the test hook bb_debug_last_route).
enum BbRoute {
  BB_ROUTE_NONE = 0,
  BB_ROUTE_F32 = 1,          // chain_f32_kernel (bb_chain_f32.cu)
  BB_ROUTE_TC4 = 2,          // chain_tc4_kernel (bb_chain_tc4.cu)
  BB_ROUTE_TC = 3,           // chain_tc_kernel, table-driven (bb_chain_tc.cu)
  BB_ROUTE_LAYERED_F32 = 4,  // dense_layer_kernel per layer (bb_chain_layered.cu)
  BB_ROUTE_LAYERED_MMA = 5,  // dense_layer_tc_kernel per layer, mma.sync (bb_chain_layered.cu)
  BB_ROUTE_LAYERED_TC5 = 6,  // gemm_tc5_kernel per layer, tcgen05 (bb_gemm_tc5.cu)
  BB_ROUTE_F64 = 7,          // chain_f64_kernel (bb_chain_f64.cu)
};

// Host + device state of one direction (encoder or decoder).
struct Chain {
  ChainDesc desc;
  float* blob_dev = nullptr;   // fp32 packed weights (FFMA kernel)
  size_t smem_bytes = 0;       // dynamic smem the fp32 kernel needs
  int f32_tr = 0;              // rows per tile of the fp32 kernel (80, 64 or 32)
  // tcgen05 path (filled by bb_tc_prepare when the shape is supported)
  bool tc_ok = false;
  void* tc_blob_dev = nullptr;
  size_t tc_blob_bytes = 0;
  void* tc_host = nullptr;     // TcHost: step program + launch geometry of the tcgen05 kernel
  Tc4Plan tc4;                 // statically shaped kernel, when the chain is the reference AE family
  // layered GEMM path (any shape)
  bool f32_ok = false;         // the fused fp32 kernel fits shared memory
  bool lay_ok = false;
  float* lay_blob_dev = nullptr;
  size_t lay_w_off[BB_MAX_LAYERS] = {0}, lay_b_off[BB_MAX_LAYERS] = {0};
  // ping-pong activation scratch of the layered path: per chain (not per context: two models, or an encode on the caller's
  // stream next to a host pipeline on the model's own stream, must not share it); grown on demand, kept
  mutable float* lay_scratch = nullptr;
  mutable size_t lay_scratch_bytes = 0;
  bool lay_tc_ok = false;      // ... and its tensor-core form: fp16 hi / lo weight images per layer
  void* lay_tc_blob_dev = nullptr;
  size_t lay_tc_off[BB_MAX_LAYERS] = {0};
  // ... and its tcgen05 form (bb_gemm_tc5.cu): weights packed per column tile in the UMMA core-matrix layout
  bool g5_ok = false;
  void* g5_blob_dev = nullptr;
  float* g5_bias_dev = nullptr;
  size_t g5_w_off[BB_MAX_LAYERS] = {0}, g5_b_off[BB_MAX_LAYERS] = {0};
  float g5_unscale[BB_MAX_LAYERS] = {0};
  int lay_max_ld = 0;
  // float64 path (bb_chain_f64.cu): packed on the first BB_PREC_FP64 call, released by bb_model_trim
  mutable F64Desc f64 = {};
  mutable double* f64_blob_dev = nullptr;
  mutable size_t f64_smem = 0;
  std::vector<double> w_host[BB_MAX_LAYERS];  // kept for re-packing
  std::vector<double> b_host[BB_MAX_LAYERS];
  // what the last launch of this direction ran, set by the host-side launchers: a BbRoute and the rows of its tile (fused
  // fp32 / fp64 chains), rows per chunk (layered GEMMs) or rows in flight per CTA (tcgen05 kernels: 128 per pipeline)
  mutable int last_route = BB_ROUTE_NONE;
  mutable int last_tile_rows = 0;
};

struct bb_model {
  bb_ctx* ctx = nullptr;
  Chain enc, dec;
  int* flag_dev = nullptr;  // overflow flag of the split16 path
  // host pipeline resources (lazily created)
  cudaStream_t s_copy_in = nullptr, s_compute = nullptr, s_copy_out = nullptr;
  void* stage_dev[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [in/out][slot]
  size_t stage_bytes[2] = {0, 0};
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
  float* feat_dev = nullptr;  // [min | range | max] x n_features
  double* feat64_dev = nullptr;  // the same for float64 tables (bb_compress_host_f64 / bb_decompress_host_f64), lazily
  // kept between calls (a 9.6 GB cudaMalloc + cudaFree costs ~0.12 s, a 240 MB cudaMallocHost ~0.05 s): the table that
  // stays resident between the min/max pass and the encode pass of bb_compress_host, and the pinned float32 bounce
  // buffers of the float64 host paths; released by bb_model_destroy / bb_model_trim
  float* resident_dev = nullptr;
  size_t resident_bytes = 0;
  float* pinned_f32[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [in/out][slot] (float64 chunks of the fp64 path too)
  size_t pinned_bytes[2] = {0, 0};
};

// --- launches implemented in the kernel translation units
int bb_chain_f32_prepare(bb_ctx* ctx, Chain* c);
int bb_chain_f32_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows,
                        const float* pre_min, const float* pre_range, const float* post_min,
                        const float* post_range, void* out, int out_dtype, cudaStream_t stream);
int bb_chain_layered_prepare(bb_ctx* ctx, Chain* c);
int bb_chain_layered_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows,
                            const float* pre_min, const float* pre_range, const float* post_min,
                            const float* post_range, void* out, int out_dtype, int tensor_cores, int* flag_dev,
                            cudaStream_t stream);
int bb_gemm_tc5_prepare(bb_ctx* ctx, Chain* c);
size_t bb_gemm_tc5_buf_bytes(const Chain* c, int64_t rows);
int bb_gemm_tc5_chunk(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t rows, const float* pre_min,
                      const float* pre_range, void* buf0, void* buf1, int* flag_dev, int* out_buf, int* ld_out,
                      cudaStream_t stream);
// x / min / max of element type dtype (BB_F32 or BB_F64)
int bb_colminmax_launch(bb_ctx* ctx, const void* x, int dtype, int64_t n_rows, int n_cols, void* min_dev,
                        void* max_dev, int reset, cudaStream_t stream);
int bb_chain_f64_prepare(bb_ctx* ctx, const Chain* c);
void bb_chain_f64_release(const Chain* c);
// features (pre_* on the way in, post_* on the way out) are of type feat_dtype (BB_F32 or BB_F64)
int bb_chain_f64_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows, const void* pre_min,
                        const void* pre_range, const void* post_min, const void* post_range, int feat_dtype, void* out,
                        int out_dtype, cudaStream_t stream);
// quantised latent of `bits` (2..8) bits per code (bb_latent_q8.cu): blocks of BB_Q8_BLOCK_ROWS rows start at row 0 of the
// arrays passed; codes are n_rows x ceil(Z * bits / 8) bytes
int bb_latent_quantize_launch(bb_ctx* ctx, const float* z, int64_t n_rows, int Z, int bits, uint8_t* codes, float* lo,
                              float* step, cudaStream_t stream);
int bb_latent_dequantize_launch(bb_ctx* ctx, int bits, const uint8_t* codes, const float* lo, const float* step,
                                int64_t n_rows, int Z, float* z, cudaStream_t stream);
int bb_tc_prepare(bb_ctx* ctx, Chain* c);
void bb_tc_release(Chain* c);
int bb_tc_launch_dbg(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows, const float* pre_min,
                     const float* pre_range, const float* post_min, const float* post_range, void* out, int out_dtype,
                     int fast, int* flag_dev, int dbg_step, float* dbg_out, int force_groups, cudaStream_t stream);
int bb_tc4_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows, const float* pre_min,
                  const float* pre_range, const float* post_min, const float* post_range, void* out, int out_dtype, int fast,
                  int* flag_dev, uint32_t* trace, cudaStream_t stream);
int bb_tc_launch(bb_ctx* ctx, const Chain* c, const void* in, int in_dtype, int64_t n_rows,
                 const float* pre_min, const float* pre_range, const float* post_min,
                 const float* post_range, void* out, int out_dtype, int fast, int* flag_dev,
                 cudaStream_t stream);

// --- host tables streamed through the device (bb_api.cu): the training entry points *_epoch_host / *_validate_host
// Two device slots of window_rows rows, filled on an internal copy stream while `body` runs on `s` on the other one; events
// order the reuse of each slot.  A pageable table goes through two pinned staging buffers (copied on the worker pool), a
// pinned one is copied directly.  `body(x_dev, rows)` enqueues the work of one window on `s`; windows are cut every
// window_rows rows, so a caller that passes a multiple of its batch sees whole batches.  The slots and streams are kept in
// *win between calls (created on first use, released by bb_host_window_free).
struct HostWindow;
int bb_host_window_run(HostWindow** win, const void* x_host, size_t row_bytes, int64_t n_rows, int64_t window_rows,
                       cudaStream_t s, const std::function<int(const void*, int64_t)>& body);
void bb_host_window_free(HostWindow* win);
