/*
 * baler_b200 - C ABI of the B200-native autoencoder train / compress / decompress path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / C++ types.  The reference
 * (baler v1.4.0, pure Python) has no FFI of its own; its operator boundary for this path is the
 * model protocol (`model.encode / model.decode / model.forward`), the numpy normalisation helpers
 * and `training.fit`.  Each entry point below names the reference interface it replaces
 * (file:line relative to the reference repository).  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 (BB_OK) or a negative BB_ERR_* / a positive cudaError_t value;
 *     `bb_strerror` describes either.  No exceptions, no global state besides the CUDA context.
 *   - `*_dev` pointers are device pointers owned by the caller, `*_host` are host pointers.
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream).  Calls taking a
 *     stream are asynchronous with respect to the host.
 *   - handles are not thread-safe; use one per host thread / stream.
 *   - there is NO CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef BALER_B200_H
#define BALER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BB_VERSION 100 /* 0.1.0 */

/* error codes (negative; positive values are cudaError_t) */
#define BB_OK 0
#define BB_ERR_INVALID -1     /* bad argument */
#define BB_ERR_UNSUPPORTED -2 /* shape / mode not supported by the kernels */
#define BB_ERR_NOMEM -3
#define BB_ERR_NODEVICE -4
#define BB_ERR_OVERFLOW -5 /* fp16 split range guard tripped: rerun with BB_PREC_FP32 */

/* element types of caller buffers */
#define BB_F32 0
#define BB_F16 1
#define BB_F64 2

/* activation after a dense layer */
#define BB_ACT_NONE 0
#define BB_ACT_LEAKY 1 /* F.leaky_relu, slope 0.01 (models.py:142) */
#define BB_ACT_RELU 2

/* arithmetic of the fused dense chain */
#define BB_PREC_AUTO 0    /* SPLIT16 when the shape is supported by the tcgen05 kernel, else FP32 */
#define BB_PREC_FP32 1    /* fp32 FFMA on CUDA cores; reference tolerance 1e-5 met with margin */
#define BB_PREC_SPLIT16 2 /* tcgen05 tensor cores, fp16 hi/lo 3-product split, fp32 accumulate in TMEM */
#define BB_PREC_FAST16 3  /* tcgen05 single fp16 product: OUTSIDE the 1e-5 tolerance (~3e-4), opt-in */
#define BB_PREC_FP64 4    /* float64 DFMA chain, the reference's own arithmetic (its AE models are float64, helper.py:565):
                             matches the reference's files to ~1e-15, opt-in.  Dense chains of <= 8 layers whose widths
                             are all <= 256 (AE, CFD_dense_AE and AE_Dropout_BN up to 256 columns); other shapes return
                             BB_ERR_UNSUPPORTED.  The float64 weight image is packed on the first call. */

typedef struct bb_ctx bb_ctx;         /* one per device */
typedef struct bb_model bb_model;     /* packed encoder + decoder weights of one autoencoder */
typedef struct bb_trainer bb_trainer; /* parameters + Adam state + scratch of one training run */
typedef void* bb_stream_t;            /* cudaStream_t */

int bb_version(void);
const char* bb_strerror(int code);

/* replaces helper.get_device (helper.py:425-439): binds a context to CUDA device `device` */
int bb_ctx_create(int device, bb_ctx** out);
int bb_ctx_destroy(bb_ctx* ctx);
int bb_ctx_sm_count(const bb_ctx* ctx);

/*
 * Pack a dense autoencoder for inference.  Replaces data_processing.load_model
 * (data_processing.py:89-110) + model.eval(): the caller reads model.pt (a state_dict) and hands
 * over the Linear tensors as the reference stores them, `weights[l]` = (dims[l+1], dims[l])
 * row-major float64, `biases[l]` = (dims[l+1]).  Eval-mode BatchNorm is folded into the
 * neighbouring Linear by the caller (exact affine algebra, done in float64 on the host).
 *   AE / CFD_dense_AE (models.py:116-157,186-226):
 *        enc dims {F,200,100,50,z} acts {LEAKY,LEAKY,LEAKY,NONE}; dec mirrored.
 *   AE_Dropout_BN (models.py:256-313): enc acts all LEAKY; dec acts {LEAKY,LEAKY,LEAKY,RELU}.
 */
int bb_model_create_dense(bb_ctx* ctx,
                          int n_enc_layers, const int* enc_dims, const int* enc_acts,
                          const double* const* enc_weights_host, const double* const* enc_biases_host,
                          int n_dec_layers, const int* dec_dims, const int* dec_acts,
                          const double* const* dec_weights_host, const double* const* dec_biases_host,
                          bb_model** out);
int bb_model_destroy(bb_model* m);
/* The host pipelines keep their device / pinned scratch between calls (the resident copy of the table between the two
 * passes of bb_compress_host can be as large as the table), and the layered GEMM path of wide models (Conv_AE,
 * CFD_dense_AE) keeps its activation scratch (up to 2 x 1.24 GB per direction).  This releases both; the next call allocates again.  The
 * reference has no counterpart: helper.compress (helper.py:473-616) holds the whole table in host memory instead. */
int bb_model_trim(bb_model* m);
int bb_model_n_features(const bb_model* m);
int bb_model_z_dim(const bb_model* m);
/* which arithmetic BB_PREC_AUTO resolves to for this model (BB_PREC_FP32 or BB_PREC_SPLIT16) */
int bb_model_auto_precision(const bb_model* m);
/* Per direction: which arithmetic BB_PREC_AUTO resolves to for the encoder (direction 0) / the decoder (1) alone -
 * BB_PREC_SPLIT16 when that chain has a tensor-core form, else BB_PREC_FP32 (bb_model_auto_precision: both have one). */
int bb_model_chain_precision(const bb_model* m, int direction);
/*
 * Range guard of BB_PREC_SPLIT16 / FAST16: activations are carried as fp16 hi + lo, so a value beyond
 * +-65504 anywhere in the chain poisons that row (inf/NaN).  The kernels raise a sticky device flag when
 * an output is not finite.  This call synchronises the device, returns the flag in *out (0 / 1) and
 * clears it when `reset` != 0; on 1 the caller re-runs the rows with BB_PREC_FP32.  The host pipelines
 * (bb_compress_host / bb_decompress_host) do this check and fall back internally.
 */
int bb_model_range_flag(bb_model* m, int reset, int* out);

/*
 * Per-column min and max of a row-major n x c float32 table.
 * Replaces data_processing.find_minmax (data_processing.py:113-130); range = max - min is left to
 * the caller so that shards can be combined (min of mins, max of maxes) before subtracting.
 * NaNs propagate like numpy's min/max.
 */
int bb_colminmax_f32(bb_ctx* ctx, const float* x_dev, int64_t n_rows, int n_cols,
                     float* min_dev, float* max_dev, bb_stream_t stream);
/* The same for a float64 table: data_processing.find_minmax (data_processing.py:113-130) on the float64 arrays the
 * reference loads, exact (-0 < +0, NaN propagates per column). */
int bb_colminmax_f64(bb_ctx* ctx, const double* x_dev, int64_t n_rows, int n_cols,
                     double* min_dev, double* max_dev, bb_stream_t stream);

/*
 * Stand-alone column normalisation and its inverse on device tables (row-major n x c float32):
 *   out = (x - min) / range      helper.normalize (helper.py:261-274, data_processing.py:133-153)
 *   out = y * range + min        helper.renormalize (helper.py:322-333, data_processing.py:188-203)
 * `out_dev` may alias the input.  The compress / decompress kernels below fuse these instead.
 */
int bb_normalize_f32(bb_ctx* ctx, const float* x_dev, int64_t n_rows, int n_cols, const float* min_dev,
                     const float* range_dev, float* out_dev, bb_stream_t stream);
int bb_renormalize_f32(bb_ctx* ctx, const float* y_dev, int64_t n_rows, int n_cols, const float* min_dev,
                       const float* range_dev, float* out_dev, bb_stream_t stream);
/* out = (x - min) / range on a row-major n x c float64 table: the reference's float64 numpy normalisation of a float64
 * file (data_processing.py:133-153), one IEEE subtract and one IEEE divide per element, bit-equal to numpy (0 / 0 gives
 * NaN as there).  `out_dev` may alias the input. */
int bb_normalize_f64(bb_ctx* ctx, const double* x_dev, int64_t n_rows, int n_cols, const double* min_dev,
                     const double* range_dev, double* out_dev, bb_stream_t stream);

/*
 * z = encode((x - min) / range)  for n_rows rows of the row-major table x (n_rows x n_features).
 * Replaces helper.normalize (helper.py:261-274, data_processing.py:133-153) fused with the
 * `model.encode` loop of helper.compress (helper.py:583-611).  The fused form computes
 * (x - min) * rcp(range) (one multiply by the correctly rounded reciprocal: <= 1 ulp from the
 * reference's IEEE divide, inside the 1e-5 bar); the stand-alone bb_normalize_f32 above is the
 * bit-equal subtract + divide.  min_dev/range_dev may both be NULL (apply_normalization = False).
 * z_dtype: BB_F32 or BB_F16 (row-major n_rows x z_dim).
 * precision BB_PREC_FP64: the table is normalised in float32 (bit-equal to numpy's float32 arithmetic, the
 * reference converts to a float64 tensor after normalising, data_processing.py:133-153), widened and run through
 * the float64 chain; z_dtype may then also be BB_F64.
 */
int bb_encode_f32(bb_model* m, const float* x_dev, int64_t n_rows,
                  const float* min_dev, const float* range_dev,
                  void* z_dev, int z_dtype, int precision, bb_stream_t stream);

/*
 * y = decode(z) * range + min.  Replaces the `model.decode` loop of helper.decompress
 * (helper.py:701-723) fused with helper.renormalize (helper.py:322-333,
 * data_processing.py:188-203).  min_dev/range_dev may both be NULL.
 */
int bb_decode_f32(bb_model* m, const void* z_dev, int z_dtype, int64_t n_rows,
                  const float* min_dev, const float* range_dev,
                  float* y_dev, int precision, bb_stream_t stream);
/* (bb_decode_f32 with BB_PREC_FP64: z_dtype BB_F32 / BB_F16 / BB_F64, chain and un-normalisation in float64, float32 out.) */

/*
 * Float64 tables (BB_PREC_FP64 arithmetic throughout): helper.compress / helper.decompress on the float64 files the
 * reference reads and writes (helper.py:473-616, 619-733).
 *   bb_encode_f64: z = encode((x - min) / range), normalised in float64 (data_processing.py:133-153) and fused with the
 *                  `model.encode` loop (helper.py:583-611).
 *   bb_decode_f64: y = decode(z) * range + min in float64 (helper.py:701-723 fused with data_processing.py:188-203).
 * min_dev / range_dev may both be NULL.  BB_ERR_UNSUPPORTED for shapes outside BB_PREC_FP64's.
 */
int bb_encode_f64(bb_model* m, const double* x_dev, int64_t n_rows, const double* min_dev,
                  const double* range_dev, double* z_dev, bb_stream_t stream);
int bb_decode_f64(bb_model* m, const double* z_dev, int64_t n_rows, const double* min_dev,
                  const double* range_dev, double* y_dev, bb_stream_t stream);

/*
 * The host-side steps of the two pipelines below, callable on their own (no device needed):
 *   bb_host_convert        float32 -> float64 (exact) or float64 -> float32 (round to nearest even) of n values on the
 *                          library's worker threads with non-temporal stores - the astype() of helper.py:565 / 653 that
 *                          turns the latent / reconstruction into the dtypes the reference writes;
 *   bb_host_colminmax_f32  per-column min and max of a row-major float32 table (data_processing.py:113-130), the scan
 *                          bb_compress_host overlaps with the upload; a column holding a nan gives nan, as numpy does.
 */
int bb_host_convert(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n);
int bb_host_colminmax_f32(const float* x_host, int64_t n_rows, int n_cols, float* min_out, float* max_out);

/*
 * Whole-table compress / decompress with HOST buffers: chunked, double-buffered H2D copy ->
 * kernels -> D2H copy on internal streams; returns when the output is complete in host memory.
 * These are what the reference-facing `helper.compress` / `helper.decompress` drop-ins call and
 * what `bench.py` times as `e2e`.
 *   bb_compress_host: if `features_host_inout` has `recompute_minmax` != 0 the column min / range
 *     are computed from THIS table first (as helper.compress does, helper.py:500-502) and written
 *     to features_host (2 x n_features float32: [min; range]); otherwise they are read from it.
 *     features_host == NULL: no normalisation.
 *   z_dtype / y_dtype: BB_F32, BB_F64 (what the reference writes for AE, helper.py:565) or, for z,
 *     BB_F16.  Pinned (page-locked) host buffers make the copies asynchronous; pageable works too.
 *   precision BB_PREC_FP64: the float64 chain (see bb_encode_f32 / bb_decode_f32); BB_F64 latents and reconstructions
 *     then cross PCIe as float64, with no float32 step on the host.
 */
int bb_compress_host(bb_model* m, const float* x_host, int64_t n_rows,
                     float* features_host, int recompute_minmax,
                     void* z_host, int z_dtype, int precision);
int bb_decompress_host(bb_model* m, const void* z_host, int z_dtype, int64_t n_rows,
                       const float* features_host, void* y_host, int y_dtype, int precision);
/* The same pipelines for float64 tables, in float64 throughout (BB_PREC_FP64): helper.compress / helper.decompress
 * (helper.py:473-616, 619-733) on a float64 file.  features_host is 2 x n_features float64 [min; range] (computed from
 * THIS table when recompute_minmax != 0, exact float64 column min / max; helper.py:500-502), or NULL. */
int bb_compress_host_f64(bb_model* m, const double* x_host, int64_t n_rows, double* features_host,
                         int recompute_minmax, double* z_host);
int bb_decompress_host_f64(bb_model* m, const double* z_host, int64_t n_rows, const double* features_host,
                           double* y_host);

/* ------------------------------------------------------------------ 8-bit latent (latent_dtype "q8") */
/*
 * The latent [n_rows, z_dim] as uint8 codes plus a float32 pair (lo, step) per latent column and block of
 * BB_Q8_BLOCK_ROWS consecutive rows, counted from row 0 of the arrays passed (the last block may be short):
 *   lo / hi   min / max of the block column's finite values (-0 < +0; 0 when it has none)
 *   step      float32((float64(hi) - float64(lo)) / 254)
 *   code      255 for a non-finite value (it decodes to NaN); 0 when step == 0;
 *             else clamp(rint((float64(v) - lo) * (1.0 / float64(step))), 0, 254), each float64 operation IEEE
 *   decoded   float32(float64(lo) + float64(code) * float64(step)): |decoded - v| <= step / 2 plus float32 rounding
 * lo_dev / step_dev hold ceil(n_rows / BB_Q8_BLOCK_ROWS) x z_dim floats.  The reference has no counterpart: it writes the
 * latent as float64 (helper.py:565).
 */
#define BB_Q8_BLOCK_ROWS 128
int bb_latent_quantize_q8(bb_ctx* ctx, const float* z_dev, int64_t n_rows, int z_dim, uint8_t* codes_dev, float* lo_dev,
                          float* step_dev, bb_stream_t stream);
int bb_latent_dequantize_q8(bb_ctx* ctx, const uint8_t* codes_dev, const float* lo_dev, const float* step_dev,
                            int64_t n_rows, int z_dim, float* z_dev, bb_stream_t stream);
/* bb_compress_host / bb_decompress_host with the 8-bit latent: encode a chunk -> quantise on the device -> copy codes and
 * parameters out (and back: copy in -> dequantise -> decode with the fused un-normalisation).  Same chunking, streams and
 * features as the float pipelines; chunks start on block boundaries, so the result does not depend on the chunking.
 * codes_host is n_rows x z_dim bytes, lo_host / step_host ceil(n_rows / 128) x z_dim floats.  y_dtype BB_F32 or BB_F64.
 * BB_PREC_FP64 returns BB_ERR_UNSUPPORTED: an 8-bit latent discards far more than float64 arithmetic gains. */
int bb_compress_host_q8(bb_model* m, const float* x_host, int64_t n_rows, float* features_host, int recompute_minmax,
                        uint8_t* codes_host, float* lo_host, float* step_host, int precision);
int bb_decompress_host_q8(bb_model* m, const uint8_t* codes_host, const float* lo_host, const float* step_host, int64_t n_rows,
                          const float* features_host, void* y_host, int y_dtype, int precision);

/* ------------------------------------------------------------------ b-bit latent (latent_dtype "q2" ... "q8") */
/*
 * The 8-bit latent above at `bits` bits per code, BB_LATENT_MIN_BITS <= bits <= BB_LATENT_MAX_BITS.  With L = 2^bits - 2:
 *   step      float32((float64(hi) - float64(lo)) / L)
 *   code      2^bits - 1 for a non-finite value; 0 when step == 0; else clamp(rint(...), 0, L) as above
 * Row r of the codes is row_bytes = ceil(z_dim * bits / 8) bytes: column j's code is bits [j * bits, (j + 1) * bits) of the
 * row, bit k being bit k % 8 of byte k / 8; the unused high bits of the last byte are 0.  codes are n_rows x row_bytes bytes,
 * lo / step ceil(n_rows / BB_Q8_BLOCK_ROWS) x z_dim floats.  bits = 8 is the 8-bit latent, byte for byte: the four _q8
 * entry points are these with bits = 8.  bits outside the range returns BB_ERR_INVALID; BB_PREC_FP64 BB_ERR_UNSUPPORTED.
 * The quantise kernel stages a block's codes in shared memory: 128 x (row_bytes + z_dim) bytes (128 x z_dim for bits = 8)
 * must fit a block's shared memory (z_dim up to about 1,700 at 8 bits on a B200), else BB_ERR_UNSUPPORTED.
 */
#define BB_LATENT_MIN_BITS 2
#define BB_LATENT_MAX_BITS 8
int bb_latent_quantize_packed(bb_ctx* ctx, const float* z_dev, int64_t n_rows, int z_dim, int bits, uint8_t* codes_dev,
                              float* lo_dev, float* step_dev, bb_stream_t stream);
int bb_latent_dequantize_packed(bb_ctx* ctx, int bits, const uint8_t* codes_dev, const float* lo_dev, const float* step_dev,
                                int64_t n_rows, int z_dim, float* z_dev, bb_stream_t stream);
int bb_compress_host_packed(bb_model* m, const float* x_host, int64_t n_rows, float* features_host, int recompute_minmax,
                            int bits, uint8_t* codes_host, float* lo_host, float* step_host, int precision);
int bb_decompress_host_packed(bb_model* m, int bits, const uint8_t* codes_host, const float* lo_host, const float* step_host,
                              int64_t n_rows, const float* features_host, void* y_host, int y_dtype, int precision);

/* ------------------------------------------------------------------ training (dense AE) */

typedef struct bb_train_hyper {
  double lr;        /* config.lr; Adam defaults below match training.py:266 */
  double beta1;     /* 0.9 */
  double beta2;     /* 0.999 */
  double eps;       /* 1e-8 */
  double reg_param; /* config.reg_param, used only when l1 != 0 */
  int l1;           /* 0: mse_sum_loss_l1(validate=True) as training.fit ships (training.py:83-89);
                       1: + reg_param * L1 chain (utils.py:201-209) */
  int world_size;   /* data-parallel ranks; gradients are SUM-reduced (loss is a sum, utils.py:195) */
} bb_train_hyper;

/*
 * Replaces `model = AE(n_features, z_dim)` + torch.optim.Adam(model.parameters()) (training.py:266).
 * `weights/biases` as for bb_model_create_dense, 8 layers F-200-100-50-z-50-100-200-F, float64 host.
 */
int bb_trainer_create(bb_ctx* ctx, int n_features, int z_dim,
                      const double* const* weights_host, const double* const* biases_host,
                      int max_batch, bb_trainer** out);
/*
 * AE_Dropout_BN (models.py:256-313) in train mode: the 8 Linear tensors as above plus, for the 4 decoder
 * BatchNorm1d layers (dec_nn.2, .5, .8, .10), weight / bias / running_mean / running_var (float64 host) and
 * num_batches_tracked.  Dropout p = .5/.4/.3/.2 after the encoder Linears, BatchNorm with whole-batch statistics
 * (biased variance, eps 1e-5, momentum 0.1).  Runs on the tensor-core step (BB_PREC_SPLIT16, the default): batches of
 * up to 16 rows x resident CTAs per GPU (2368 on B200: the tiles of a batch meet at the 8 BatchNorm reduction points
 * of a step); data parallel through bb_trainer_dp_connect with the statistics of the GLOBAL batch (the per-rank sums
 * of every reduction point are exchanged over NVLink peer memory inside the kernel) and a dropout stream keyed by
 * the global batch row, i.e. the replicas compute what one GPU computes at batch_size = global batch.  The fp32
 * kernels (BB_PREC_FP32) remain as the reference-accuracy path: one GPU's statistics, batch <= 592 rows.
 * MSE loss only: what training.fit evaluates (it calls the loss with validate=True, so the L1 term never trains).
 */
int bb_trainer_create_dbn(bb_ctx* ctx, int n_features, int z_dim,
                          const double* const* weights_host, const double* const* biases_host,
                          const double* const* bn_weight_host, const double* const* bn_bias_host,
                          const double* const* bn_mean_host, const double* const* bn_var_host,
                          const long long* bn_batches_tracked, int max_batch, bb_trainer** out);
/* dropout: in-kernel Philox4x32-10 keyed by (seed, step, layer, row, column); `masks_dev` (4 device pointers to
 * [batch x width] uint8 keep-masks, or NULL) injects torch-generated masks for parity tests.  Disarms the torch stream. */
int bb_trainer_set_dropout(bb_trainer* t, unsigned long long seed, const unsigned char* const* masks_dev);
/* dropout from torch's CPU generator (BB_PREC_FP64 only; other precisions: BB_ERR_UNSUPPORTED).  The reference draws
 * every mask with bernoulli_(1 - p) on torch's default generator, an MT19937: per batch, layer 0..3, [rows x width]
 * row-major, two words per element (first word high), keep = (random64 & (2^53 - 1)) * 2^-53 < 1 - p.
 * set_dropout_mt19937 arms that stream for the following steps from the generator's state: its 624-word key and the
 * position 0..624 of the next word (numpy's count; 624 - (left - 1) of torch.Generator.get_state()).  Each training
 * step then draws its batch's masks on the device, on a side stream one step ahead, without a host synchronisation.
 * get_dropout_mt19937 returns the state after the last drawn word (synchronises the side stream); writing it back into
 * the generator leaves it where the reference's would be.  BB_ERR_INVALID before the stream is armed. */
int bb_trainer_set_dropout_mt19937(bb_trainer* t, const uint32_t* key_624, int pos);
int bb_trainer_get_dropout_mt19937(bb_trainer* t, uint32_t* key_out_624, int* pos_out);
/* device views of the concatenated BatchNorm running statistics (4 layers, 50 + 100 + 200 + n_features values each).
 * Data parallel inside the library keeps them identical on every rank; host-loop data parallel (per-rank statistics)
 * averages them over ranks (torch DDP broadcasts rank 0's buffers instead; models.py:275-296) */
int bb_trainer_bn_running_dev(bb_trainer* t, float** running_mean_dev, float** running_var_dev, int* n);
/* BB_PREC_FP64: the float64 running statistics the float64 step updates (BB_ERR_UNSUPPORTED for other precisions) */
int bb_trainer_bn_running_dev_f64(bb_trainer* t, double** running_mean_dev, double** running_var_dev, int* n);
/* gamma / beta, running statistics and num_batches_tracked as float64 (BB_PREC_FP64: the float64 master as it is) */
int bb_trainer_get_bn(bb_trainer* t, double* const* bn_weight_host, double* const* bn_bias_host,
                      double* const* bn_mean_host, double* const* bn_var_host, long long* bn_batches_tracked);
int bb_trainer_destroy(bb_trainer* t);
/*
 * Arithmetic of the training step (the reference trains in float64 on torch, training.py:64-97; both choices here meet
 * the 1e-5 per-step bar on loss, gradients and the Adam update):
 *   BB_PREC_SPLIT16  tensor cores (mma.sync m16n8k16, fp16 hi / lo 3-product split, fp32 accumulate), one persistent
 *                    kernel per epoch; the default (BB_PREC_AUTO) for `AE` / `CFD_dense_AE` / `AE_Dropout_BN` with the
 *                    MSE loss.
 *   BB_PREC_FP32     fp32 FFMA kernels; always used for the opt-in L1 chain.
 *   BB_PREC_FP64     float64 DFMA kernels with float64 master parameters and Adam state: the reference's float64
 *                    training to rounding (~1e-14), MSE and L1 chain.  Only before the first step or epoch (later:
 *                    BB_ERR_INVALID).  It uploads the float64 weights (and for bb_trainer_create_dbn the BatchNorm
 *                    gamma / beta, running statistics and num_batches_tracked) that create received, exactly.  The
 *                    float32 table entry points widen x exactly; the *_f64 ones below take float64 tables.  The in-kernel
 *                    exchange (bb_trainer_dp_export / _connect) is not available: data parallel runs phase 1, an
 *                    all-reduce of the float64 gradient (bb_trainer_grads_dev_f64) and phase 2.
 *                    AE_Dropout_BN: one cooperative kernel with whole-batch float64 BatchNorm statistics, MSE loss only,
 *                    batches up to 4 rows x resident CTAs (592 on B200; beyond: BB_ERR_UNSUPPORTED), one GPU's
 *                    statistics; dropout from Philox (the same masks as BB_PREC_FP32), injected masks or torch's
 *                    stream (bb_trainer_set_dropout_mt19937).
 * bb_trainer_precision returns what the next MSE step will run on.  Values beyond +-65504 (un-normalised tables) leave
 * the fp16 range on the SPLIT16 path: the batch loss turns non-finite, a sticky flag is raised and
 * bb_trainer_range_flag reports it (synchronises the device); the caller restarts with BB_PREC_FP32.
 */
int bb_trainer_set_precision(bb_trainer* t, int precision);
int bb_trainer_precision(const bb_trainer* t);
int bb_trainer_range_flag(bb_trainer* t, int reset, int* out);
/* Diagnostics of the SPLIT16 step (tests): what the last step left in its scratch for `layer` (0..7), as float32
 * [features][rows] in out_host: which = 0 the layer's input (in_features + 1 rows of features, the last one the bias
 * column of ones), which = 1 the gradient of the loss with respect to its pre-activation output (out_features).
 * Returns the number of features (> 0) or an error (< 0). */
int bb_trainer_debug_layer(bb_trainer* t, int which, int layer, int rows, float* out_host, int capacity_floats);
/* Diagnostics of the SPLIT16 step: arm SM-clock stamps of CTA 0 for step `step` of the following launches (step < 0:
 * off) and read the stamps of the last armed launch into out_host_128 (nullable): [0] step start, [1] forward /
 * backward done, [2] grid barrier passed, [3] weight gradients + Adam done, [4] second barrier passed, [8 + p] / [32 + p] /
 * [48 + p] start / end of the MMAs / end of the epilogue of layer pass p (0-7 forward, 8-14 backward).  Returns the
 * number of weight chunks per step. */
int bb_trainer_profile(bb_trainer* t, int step, long long* out_host_128);
/* flat float32 views (device) of parameters / gradients, layout: for l in 0..7: W_l (out,in) then b_l */
int bb_trainer_param_count(const bb_trainer* t);
float* bb_trainer_params_dev(bb_trainer* t);
float* bb_trainer_grads_dev(bb_trainer* t);
/* BB_PREC_FP64: the float64 master parameters and the float64 gradient (n_params entries, then the batch loss), same
 * layout; NULL for the other precisions (the float32 views above keep their meaning and are not updated by fp64 steps) */
double* bb_trainer_params_dev_f64(bb_trainer* t);
double* bb_trainer_grads_dev_f64(bb_trainer* t);
/* copy parameters back as the reference's float64 state_dict tensors (BB_PREC_FP64: the float64 master as it is) */
int bb_trainer_get_params(bb_trainer* t, double* const* weights_host, double* const* biases_host);

/*
 * One optimisation step on `batch_rows` rows (x_dev row-major float32, already normalised):
 * zero_grad -> forward -> loss -> backward [-> caller all-reduces grads] -> Adam.
 * Replaces the body of the batch loop of training.fit (training.py:64-97).
 *   phase 0: everything (single GPU);  phase 1: forward + backward only (grads and loss left in
 *   device memory for an all-reduce);  phase 2: Adam only.
 * The batch loss is ADDED to *loss_accum_dev (double) so an epoch needs no host sync.
 */
int bb_trainer_step(bb_trainer* t, const float* x_dev, int batch_rows, const bb_train_hyper* h,
                    int phase, double* loss_accum_dev, bb_stream_t stream);
/*
 * Data parallel training inside the library (one process per GPU, NVLink peer memory; the reference is single-process:
 * this is the run with batch_size = global batch, training.py:253-263, spread over the GPUs).  Every rank
 *   1. bb_trainer_dp_export: allocates its exchange block and writes its 64-byte CUDA IPC handle,
 *   2. (host side: all-gather of the handles, e.g. torch.distributed.all_gather_object),
 *   3. bb_trainer_dp_connect: maps the peers' blocks (`handles` = world_size x 64 bytes in rank order).
 * Afterwards bb_trainer_epoch with h->world_size == world_size takes the FULL table and the GLOBAL batch: each rank
 * processes its contiguous share of every global batch; inside the weight-gradient phase of the step kernel each rank
 * pushes every 32 x 32 gradient tile into all ranks' buffers over NVLink as 8-byte {value, step tag} packets and sums the
 * world's tiles in rank order as they land, before Adam - a fused SUM all-reduce (the loss is a sum: utils.py:195),
 * bit-identical replicas, no collective call on the host inside an epoch.  The epoch loss each rank gets back is ITS share
 * (sum of its rows' terms / number of batches): the caller adds the ranks' values.  SPLIT16 step only (MSE loss).
 * AE_Dropout_BN additionally exchanges, at each of its 8 BatchNorm reduction points, the per-rank column sums as 16-byte
 * {a, tag, b, tag} packets and combines them in rank order: BatchNorm over the global batch, identical on every rank.
 */
int bb_trainer_dp_export(bb_trainer* t, int world_size, unsigned char* handle_out_64);
int bb_trainer_dp_connect(bb_trainer* t, int rank, int world_size, const unsigned char* handles);
/*
 * One epoch over n_rows rows in sequential batches of `batch` (last one ragged, drop_last=False,
 * shuffle=False: training.py:253-263).  h->world_size > 1: see bb_trainer_dp_connect.  Writes the epoch loss
 * (mean of batch losses, training.py:99) to *epoch_loss_host after synchronising `stream`.
 */
int bb_trainer_epoch(bb_trainer* t, const float* x_dev, int64_t n_rows, int batch,
                     const bb_train_hyper* h, double* epoch_loss_host, bb_stream_t stream);
/* forward only in eval mode, sum-MSE / n_cols per batch averaged over batches: training.validate
 * (training.py:104-137) */
int bb_trainer_validate(bb_trainer* t, const float* x_dev, int64_t n_rows, int batch,
                        double* epoch_loss_host, bb_stream_t stream);
/* bb_trainer_step / _epoch / _validate on a float64 table (the reference's float64 training tensor, training.py:230):
 * BB_PREC_FP64 trainers only (BB_ERR_INVALID otherwise) */
int bb_trainer_step_f64(bb_trainer* t, const double* x_dev, int batch_rows, const bb_train_hyper* h,
                        int phase, double* loss_accum_dev, bb_stream_t stream);
int bb_trainer_epoch_f64(bb_trainer* t, const double* x_dev, int64_t n_rows, int batch,
                         const bb_train_hyper* h, double* epoch_loss_host, bb_stream_t stream);
int bb_trainer_validate_f64(bb_trainer* t, const double* x_dev, int64_t n_rows, int batch,
                            double* epoch_loss_host, bb_stream_t stream);
/*
 * bb_trainer_epoch / _validate (and their _f64 forms) on a HOST table, for tables larger than device memory: the reference
 * trains on the CPU (training.py:253-263), so it takes whatever fits in host memory.  x_host is row-major n_rows x
 * n_features of x_dtype: BB_F32, or BB_F64 for BB_PREC_FP64 trainers (others: BB_ERR_INVALID).  The library keeps two
 * device slots of `window_rows` rows (a positive multiple of `batch`, else BB_ERR_INVALID; allocated on first use, kept
 * until bb_trainer_destroy).  An internal copy stream fills one slot while the epoch's kernels run on `stream` over the
 * other; events order the reuse of each slot.  A pageable table is staged through two 64 MiB pinned buffers on the
 * library's worker threads (the table itself is never pinned); a pinned one is copied directly.
 * Windows are cut at batch boundaries and the step counter runs on across them (Philox dropout keys, Adam's bias
 * correction, data-parallel packet tags), the torch-stream masks are drawn per batch in order, batch losses go into the
 * same device accumulator in batch order, and BatchNorm statistics advance per batch: the results are bit-identical to
 * the resident calls on the same table, for every trainer and precision (h->world_size > 1 included: every rank passes the
 * full table and the global batch).  Returns after synchronising `stream`.
 */
int bb_trainer_epoch_host(bb_trainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch, const bb_train_hyper* h,
                          int64_t window_rows, double* epoch_loss_host, bb_stream_t stream);
int bb_trainer_validate_host(bb_trainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch, int64_t window_rows,
                             double* epoch_loss_host, bb_stream_t stream);

/*
 * Per-node mean activation of the six hidden layers (en1,en2,en3,de1,de2,de3) over the rows of the LAST
 * forward pass, as a 6 x 200 float64 matrix padded with NaN: what model.get_activations() +
 * diagnostics.dict_to_square_matrix write to activations.npy (models.py:160-179, diagnostics.py:10-47).
 */
int bb_trainer_activation_means(bb_trainer* t, double* out_host_6x200);

/*
 * Layer-by-layer trainer for dense autoencoders whose weights do not fit the fused training kernels: CFD_dense_AE on
 * 2500-feature snapshots (models.py:186-226) or any chain of up to 8 Linears with dims[0] == dims[n_layers].  Same
 * contract as bb_trainer_* (training.fit training.py:31-101, Adam training.py:266, sum-MSE / n_columns
 * utils.py:195-199), one fp32 GEMM launch per matrix product.  `weights[l]` = (dims[l+1], dims[l]) row-major float64,
 * `acts[l]` = BB_ACT_*.  MSE only (h->l1 must be 0); phase as in bb_trainer_step.
 */
typedef struct bb_ltrainer bb_ltrainer;
int bb_ltrainer_create(bb_ctx* ctx, int n_layers, const int* dims, const int* acts, const double* const* weights_host,
                       const double* const* biases_host, int max_batch, bb_ltrainer** out);
/*
 * The same trainer for Conv_AE (models.py:316-407, float32) on a fixed block shape.  A (transposed) convolution is a
 * layer with n_shared_w[l] > 0: its dense (dims[l+1], dims[l]) matrix is w_maps[l][i] -> index of the kernel weight entry
 * i repeats (-1: structural zero), its bias is one value per channel (n_bias[l] channels of dims[l+1] / n_bias[l]
 * consecutive outputs); `weights_host[l]` / `biases_host[l]` then hold the n_shared_w[l] kernel weights / n_bias[l]
 * channel biases, and only those are trained.  bn_channels[l] > 0 puts nn.BatchNorm2d(bn_channels[l]) between the
 * affine map and the activation (training steps: batch statistics, eps 1e-5, running statistics with momentum 0.1;
 * bb_ltrainer_validate: running statistics); `bn_host[l]` = gamma | beta | running_mean | running_var, 4 x channels.
 * loss_columns: the divisor of the summed squared error (utils.py:197 `true_data.shape[1]`: 1 for (B, 1, H, W)
 * batches); 0 = dims[n_layers].  Any of n_shared_w, w_maps, n_bias, bn_channels, bn_host may be NULL (plain Linears).
 * Up to 16 layers.  The flat vector behind params_dev / grads_dev holds, layer after layer, weights | biases | gamma |
 * beta of the TRAINABLE parameters.
 */
int bb_ltrainer_create_ex(bb_ctx* ctx, int n_layers, const int* dims, const int* acts, const int* n_shared_w,
                          const int32_t* const* w_maps, const int* n_bias, const int* bn_channels,
                          const double* const* weights_host, const double* const* biases_host, const double* const* bn_host,
                          int loss_columns, int max_batch, bb_ltrainer** out);
int bb_ltrainer_get_bn(bb_ltrainer* t, double* const* bn_host); /* per BatchNorm layer: gamma | beta | running_mean | running_var */
float* bb_ltrainer_bn_running_dev(bb_ltrainer* t, int* n_floats); /* running (mean | var) of every BatchNorm layer, layer after layer */
int bb_ltrainer_destroy(bb_ltrainer* t);
int bb_ltrainer_param_count(const bb_ltrainer* t);
float* bb_ltrainer_params_dev(bb_ltrainer* t);
float* bb_ltrainer_grads_dev(bb_ltrainer* t);  /* n_params gradient entries, then the batch loss */
int bb_ltrainer_get_params(bb_ltrainer* t, double* const* weights_host, double* const* biases_host);
int bb_ltrainer_step(bb_ltrainer* t, const float* x_dev, int batch_rows, const bb_train_hyper* h, int phase,
                     double* loss_accum_dev, bb_stream_t stream);
/*
 * One training step with config.custom_loss_function = "loss_function_swae" (training.py:70-78, utils.py:27-91):
 * loss = sum-MSE / n_columns + reg_weight / (B (B - 1)) * mean over projections s and ranks i of
 * (sort(z P)[s][i] - sort(prior P)[s][i])^2, z the latent batch (output of layer `latent_layer`).  The two random
 * inputs of utils.compute_swd are the caller's: `prior_dev` [batch_rows][z_dim] (torch.randn_like(z)) and `proj_dev`
 * [n_projections][z_dim] unit rows (utils.get_random_projections), so a caller that draws them from torch's generator
 * in the reference's order reproduces the reference's stream.  Upstream encodes twice per step (model(inputs), then
 * model.encode(inputs)) with the same batch and weights: the same values and batch statistics, and the gradient of
 * the two backward passes is this step's single one.  BatchNorm layers at or before `latent_layer` update their running
 * statistics twice per step and count 2 batches (bb_ltrainer_bn_batches_tracked), later ones once.  Layers with dropout
 * (the second encode would draw other masks): BB_ERR_UNSUPPORTED.  2 <= batch_rows <= max_batch: up to 2048 rows each
 * projection is sorted in shared memory, above that by a stable radix sort in global memory (ties in row order), whose
 * scratch (4 x max_batch x n_projections x 4 bytes) is allocated by the first step of a trainer with max_batch > 2048.
 * phase as in bb_ltrainer_step.
 */
int bb_ltrainer_step_swae(bb_ltrainer* t, const float* x_dev, int batch_rows, const bb_train_hyper* h, int phase,
                          const float* prior_dev, const float* proj_dev, int n_projections, int latent_layer, float reg_weight,
                          double* loss_accum_dev, bb_stream_t stream);
int bb_ltrainer_epoch(bb_ltrainer* t, const float* x_dev, int64_t n_rows, int batch, const bb_train_hyper* h,
                      double* epoch_loss_host, bb_stream_t stream);
int bb_ltrainer_validate(bb_ltrainer* t, const float* x_dev, int64_t n_rows, int batch, double* epoch_loss_host,
                         bb_stream_t stream);
/* bb_ltrainer_epoch / _validate on a host table, streamed as bb_trainer_epoch_host does (x_dtype BB_F32 only) */
int bb_ltrainer_epoch_host(bb_ltrainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch,
                           const bb_train_hyper* h, int64_t window_rows, double* epoch_loss_host, bb_stream_t stream);
int bb_ltrainer_validate_host(bb_ltrainer* t, const void* x_host, int x_dtype, int64_t n_rows, int batch,
                              int64_t window_rows, double* epoch_loss_host, bb_stream_t stream);
/*
 * AE_Dropout_BN (models.py:256-313) on the layer-by-layer trainer, at any batch size that fits in memory (the fused
 * bb_trainer_create_dbn step needs every tile of a batch resident: 16 rows x SMs on the tensor-core step).  Same
 * arguments as bb_trainer_create_dbn.  The chain: encoder 4 x (Linear -> Dropout p = .5/.4/.3/.2 -> LeakyReLU), the latent
 * included; decoder 3 x (Linear -> LeakyReLU -> BatchNorm1d), then Linear -> BatchNorm1d -> ReLU.  Training steps draw
 * their keep-masks as the fused dbn steps do (bb_trainer_set_dropout: Philox keyed by the seed and the number of earlier
 * Adam updates, or injected masks) and use batch statistics (biased variance, eps 1e-5, running statistics with momentum
 * 0.1 and the unbiased variance); bb_ltrainer_validate uses no dropout and the running statistics.  MSE only
 * (h->l1: BB_ERR_UNSUPPORTED), one process (bb_ltrainer_epoch).  The flat parameters hold, layer after layer,
 * weights | biases | gamma | beta; bb_ltrainer_get_params / bb_ltrainer_get_bn (layers 4-7) read them back.
 */
int bb_ltrainer_create_dbn(bb_ctx* ctx, int n_features, int z_dim, const double* const* weights_host,
                           const double* const* biases_host, const double* const* bn_weight_host,
                           const double* const* bn_bias_host, const double* const* bn_mean_host,
                           const double* const* bn_var_host, const long long* bn_batches_tracked, int max_batch,
                           bb_ltrainer** out);
/* AE_Dropout_BN trainers: dropout source of the following steps, as bb_trainer_set_dropout (seed, or 4 device uint8
 * keep-masks [batch][width_l], kept while they are in use; NULL: Philox) */
int bb_ltrainer_set_dropout(bb_ltrainer* t, unsigned long long seed, const unsigned char* const* masks_dev);
/* num_batches_tracked of every layer (n_layers entries; 0 for layers without BatchNorm) */
int bb_ltrainer_bn_batches_tracked(bb_ltrainer* t, long long* out_n_layers);
/* bb_trainer_activation_means of the 8-Linear autoencoders (AE, CFD_dense_AE, AE_Dropout_BN): column means of the outputs
 * of layers 0, 1, 2, 4, 5, 6 over the rows of the last forward pass (training step or validate), NaN beyond a layer's
 * width; synchronises the device.  Other chains or layers wider than 200: BB_ERR_UNSUPPORTED. */
int bb_ltrainer_activation_means(bb_ltrainer* t, double* out_host_6x200);

/*
 * Error-bounded deltas: helper.save_error_bounded_requirement (helper.py:442-470) for n_rows rows at once.  `x_dev` raw
 * rows (normalised here with [min; range] when given, exactly as helper.normalize does), `y_dev` their decoded, still
 * normalised reconstruction.  An element is a hit when |(y - x) / x * 100| > bound_percent (x == 0 never is); for every
 * hit the global row (row0 + r), the column and float16(y) - float16(x) are appended in arbitrary order; *count_dev
 * receives the number of hits (it may exceed `capacity`: entries beyond it are dropped, call again with more room).
 */
int bb_error_bounded_deltas_f32(bb_ctx* ctx, const float* x_dev, const float* y_dev, int64_t n_rows, int n_cols,
                                const float* min_dev, const float* range_dev, double bound_percent, int64_t row0,
                                int64_t capacity, unsigned long long* count_dev, long long* rows_out_dev,
                                int* cols_out_dev, void* deltas_f16_out_dev, bb_stream_t stream);

/* sum((a - b)^2) over n float32 elements, ADDED to *out_dev (double): nn.MSELoss(reduction="sum") of
 * utils.mse_sum_loss_l1 (utils.py:195-196) on loose tensors. */
int bb_mse_sum_f32(bb_ctx* ctx, const float* a_dev, const float* b_dev, int64_t n, double* out_dev, bb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BALER_B200_H */
