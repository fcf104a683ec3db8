// Float64 training step of the dense autoencoders (bb_train_f64.cu), driven by the bb_trainer of bb_train.cu when its
// precision is BB_PREC_FP64.  The trainer owns one F64Trainer: float64 master parameters, Adam state and scratch.
#pragma once

#include <curand_philox4x32_x.h>

#include "bb_common.cuh"

struct F64Trainer;

// Layout of the 8-layer chain F-200-100-50-z-50-100-200-F (the same offsets bb_train.cu uses, in doubles).
struct F64TrainLayout {
  int dims[9];
  int act[8];
  int w_off[8], b_off[8], wt_off[8];  // W_l (out, in) and b_l in the flat parameters; W_l^T [in][out] in the copy `wt`
  int a_off[9], a_stride;             // layer inputs A_0..A_8 in the per-row activation scratch
  int z_off[8], z_stride;             // dZ_0..dZ_7 in the per-row gradient scratch
  int n_params, max_dim;
  // AE_Dropout_BN (kind 1): gamma / beta of the 4 decoder BatchNorms follow the Linear layers in the flat parameters;
  // bn_f_off[i] is BatchNorm i's offset in the per-feature arrays (running statistics), bn_f_total their length
  int kind;
  int bn_g_off[4], bn_b_off[4], bn_f_off[4], bn_f_total;
};

// AE_Dropout_BN dropout keep-bit of the Philox stream: Philox4x32-10 keyed by (seed, step), counter (column / 4, row,
// layer).  Stateless, so any launch geometry draws the same masks; shared by the fp32 and the float64 kernels.
__device__ __forceinline__ bool bb_philox_keep(unsigned long long seed, unsigned long long step, int l, int grow, int j) {
  const uint4 r = curand_Philox4x32_10(make_uint4((unsigned)(j >> 2), (unsigned)grow, (unsigned)l, (unsigned)step),
                                       make_uint2((unsigned)seed, (unsigned)(seed >> 32) ^ (unsigned)(step >> 32)));
  const unsigned v = (j & 3) == 0 ? r.x : (j & 3) == 1 ? r.y : (j & 3) == 2 ? r.z : r.w;
  const float keep_p[4] = {0.5f, 0.6f, 0.7f, 0.8f};  // 1 - p of models.py:263-275
  return v < (unsigned)(keep_p[l] * 4294967296.0);
}

// params_host: n_params doubles in the flat layout, uploaded as they are.  AE_Dropout_BN also takes its running
// statistics (bn_stats_host: running_mean then running_var, bn_f_total doubles each) and num_batches_tracked[4].
// BB_ERR_UNSUPPORTED when the step's shared memory does not fit or a layer is wider than 512.
int bb_f64_train_create(bb_ctx* ctx, const F64TrainLayout& d, const double* params_host, const double* bn_stats_host,
                        const long long* nbt_host, int max_batch, F64Trainer** out);
void bb_f64_train_destroy(F64Trainer* f);
// phase as bb_trainer_step; `step` = Adam's step count t (1-based) of the update this call applies (phases 0 and 2).
// AE_Dropout_BN: BB_ERR_UNSUPPORTED for the L1 chain and for batches whose CTAs cannot all be resident.
int bb_f64_train_step(F64Trainer* f, const void* x_dev, int x_is_f64, int rows, const bb_train_hyper* h, int phase,
                      long long step, double* loss_accum_dev, cudaStream_t s);
// eval-mode forward of one batch; adds its sum-MSE / n_cols to *loss_accum_dev
int bb_f64_train_eval(F64Trainer* f, const void* x_dev, int x_is_f64, int rows, double* loss_accum_dev, cudaStream_t s);
int bb_f64_train_activation_means(F64Trainer* f, double* out_6x200);
int bb_f64_train_get_params(F64Trainer* f, double* params_host);
double* bb_f64_train_params(F64Trainer* f);
double* bb_f64_train_grads(F64Trainer* f);
// AE_Dropout_BN: dropout source of the following steps.  set_dropout: Philox seed, or 4 device keep-masks [batch][N_l]
// (uint8).  set_mt19937: torch's CPU Mersenne Twister (624-word key, position 0..624 as numpy counts it); every step then
// draws its masks on the device, as torch's bernoulli_ does, and get_mt19937 returns the state after the last drawn word.
int bb_f64_train_set_dropout(F64Trainer* f, unsigned long long seed, const unsigned char* const* masks_dev);
int bb_f64_train_set_mt19937(F64Trainer* f, const uint32_t* key_624, int pos);
int bb_f64_train_get_mt19937(F64Trainer* f, uint32_t* key_624, int* pos);
// AE_Dropout_BN: running statistics (float64, bn_f_total each) and num_batches_tracked[4]
int bb_f64_train_bn_running(F64Trainer* f, double** rm_dev, double** rv_dev);
int bb_f64_train_get_bn_stats(F64Trainer* f, double* rm_host, double* rv_host, long long* nbt_host);
// Resident CTAs of the AE_Dropout_BN step (4 rows each): its batch limit is 4 x this.
int bb_f64_train_dbn_max_ctas(F64Trainer* f);

// bb_dropout_mt.cu: the keep-masks of one AE_Dropout_BN batch from torch's CPU Mersenne Twister, in the order the
// reference draws them (layer 0..3, each [rows][widths[l]] row-major, 2 words per element, keep = uniform53 < keep[l]).
// state_dev: 624 key words then the position (numpy's count, 0..624); read at the start, advanced state written back.
// One CTA on `s`.
int bb_mt_dropout_launch(uint32_t* state_dev, int rows, const int* widths_4, const double* keep_4,
                         unsigned char* const* out_4, cudaStream_t s);
