// Float64 training step of the dense autoencoder (bb_train_f64.cu), driven by the bb_trainer of bb_train.cu when its
// precision is BB_PREC_FP64.  The trainer owns one F64Trainer: float64 master parameters, Adam state and scratch.
#pragma once

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
};

// params_host: n_params doubles in the flat layout, uploaded as they are.  BB_ERR_UNSUPPORTED when the step's shared
// memory does not fit or a layer is wider than 512.
int bb_f64_train_create(bb_ctx* ctx, const F64TrainLayout& d, const double* params_host, int max_batch, F64Trainer** out);
void bb_f64_train_destroy(F64Trainer* f);
// phase as bb_trainer_step; `step` = Adam's step count t (1-based) of the update this call applies (phases 0 and 2)
int bb_f64_train_step(F64Trainer* f, const void* x_dev, int x_is_f64, int rows, const bb_train_hyper* h, int phase,
                      long long step, double* loss_accum_dev, cudaStream_t s);
// eval-mode forward of one batch; adds its sum-MSE / n_cols to *loss_accum_dev
int bb_f64_train_eval(F64Trainer* f, const void* x_dev, int x_is_f64, int rows, double* loss_accum_dev, cudaStream_t s);
int bb_f64_train_activation_means(F64Trainer* f, double* out_6x200);
int bb_f64_train_get_params(F64Trainer* f, double* params_host);
double* bb_f64_train_params(F64Trainer* f);
double* bb_f64_train_grads(F64Trainer* f);
