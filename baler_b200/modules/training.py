"""Training loop of the hot path (reference baler/modules/training.py): same `fit / validate / train`
entry points; the batch loop runs on the GPU (bb_trainer_epoch) without a host sync per batch."""
import os
import time

import numpy as np
import torch

from .. import engine, sharded
from . import utils


dist_env = sharded.dist_env
FUSED_TRAINER_MAX_FEATURES = 100  # bb_trainer stages whole weight matrices in shared memory (widest: 200 x 100)
FP64_TRAINING_MODELS = ("AE", "CFD_dense_AE")  # what precision "fp64" trains: the fused trainer's models without BatchNorm
DROPOUT_STREAMS = ("torch",)
# AE_Dropout_BN's float64 step is one cooperative kernel of 4-row CTAs, one CTA per SM: every CTA of a batch must be
# resident (148 SMs on a B200: 592 rows)
FP64_DBN_ROWS_PER_CTA = 4
B200_SM_COUNT = 148
# AE_Dropout_BN's fused step (tensor cores) keeps every 16-row tile of a batch resident, one CTA per SM (2368 rows on a
# B200); larger batches train on the layer-by-layer trainer
DBN_FUSED_ROWS_PER_CTA = 16


def is_fp64(precision):
    return engine.PRECISIONS.get(precision or "auto") == engine.BB_PREC_FP64


def _sm_count():
    """SMs of the current GPU (a B200's without one)"""
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count \
        if torch.cuda.is_available() else B200_SM_COUNT


def fp64_dbn_max_batch():
    """largest AE_Dropout_BN batch of the float64 step: 4 rows x the SMs of the current GPU (a B200's without one)"""
    return FP64_DBN_ROWS_PER_CTA * _sm_count()


def dbn_fused_max_batch():
    """largest AE_Dropout_BN batch of the fused step: 16 rows x the SMs of the current GPU (a B200's without one); larger
    batches of one process train on the layer-by-layer trainer"""
    return DBN_FUSED_ROWS_PER_CTA * _sm_count()


def refuse_dbn_rank_share(model_name, batch_size, world):
    """NotImplementedError for AE_Dropout_BN under torchrun when a rank's share of the global batch exceeds the fused step's
    batch: the layer-by-layer trainer normalises over one process's batch only"""
    if model_name != "AE_Dropout_BN" or world <= 1 or batch_size is None:
        return
    share = (batch_size + world - 1) // world
    if share > dbn_fused_max_batch():
        raise NotImplementedError("AE_Dropout_BN with %d ranks trains per-rank shares of at most %d rows (the fused step); "
                                  "batch_size %d gives %d per rank.  BatchNorm over the global batch of larger shares is "
                                  "not implemented: lower batch_size or train in one process"
                                  % (world, dbn_fused_max_batch(), batch_size, share))


def refuse_dropout_stream(model_name, precision, dropout_stream):
    """config.dropout_stream outside precision "fp64": ValueError for an unknown value, NotImplementedError for
    AE_Dropout_BN (only the float64 step draws from torch's stream)"""
    if dropout_stream is None:
        return
    if dropout_stream not in DROPOUT_STREAMS:
        raise ValueError("dropout_stream must be one of %s, not %r" % (DROPOUT_STREAMS, dropout_stream))
    if model_name == "AE_Dropout_BN" and not is_fp64(precision):
        raise NotImplementedError("dropout_stream = %r is drawn by the float64 step of AE_Dropout_BN only; set "
                                  "precision = 'fp64' (precision is %r)" % (dropout_stream, precision))


def refuse_fp64_training(model_name, n_features, swae=False, dropout_stream=None, batch_size=None, world=1):
    """NotImplementedError naming what the float64 trainer (precision "fp64") does not take: models other than AE /
    CFD_dense_AE and AE_Dropout_BN with dropout_stream = "torch" (Conv_AE), loss_function_swae, rows wider than the
    fused trainer's; for AE_Dropout_BN also several processes and batches beyond the resident limit"""
    refuse_dropout_stream(model_name, "fp64", dropout_stream)
    if model_name == "AE_Dropout_BN":
        if dropout_stream != "torch":
            raise NotImplementedError(
                "precision='fp64' trains AE_Dropout_BN only with dropout_stream = 'torch' (the reference's own dropout "
                "masks, drawn on the device from torch's generator); with other masks a float64 run is no closer to "
                "the reference than the default precision")
        if world > 1:
            raise NotImplementedError("precision='fp64' trains AE_Dropout_BN in one process (BatchNorm over the global "
                                      "batch of %d ranks is not implemented for float64)" % world)
        if batch_size is not None and batch_size > fp64_dbn_max_batch():
            raise NotImplementedError("precision='fp64' trains AE_Dropout_BN with batch_size <= %d (every CTA of a "
                                      "batch resident); batch_size is %d" % (fp64_dbn_max_batch(), batch_size))
    elif model_name not in FP64_TRAINING_MODELS:
        raise NotImplementedError("precision='fp64' trains %s only; %s is not trained in float64 (use another precision)"
                                  % (" and ".join(FP64_TRAINING_MODELS), model_name))
    if swae:
        raise NotImplementedError("precision='fp64' trains with the MSE loss (and l1_in_training) only, not "
                                  "custom_loss_function = 'loss_function_swae'")
    if n_features > FUSED_TRAINER_MAX_FEATURES:
        raise NotImplementedError("precision='fp64' trains models of at most %d columns (the fused trainer); %s has %d"
                                  % (FUSED_TRAINER_MAX_FEATURES, model_name, n_features))


def broadcast_initial_state(model):
    """data-parallel runs start every replica from rank 0's freshly initialised model (what DistributedDataParallel does
    at construction): each process draws its own random initial weights otherwise"""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"  # gloo: the CPU tests of the host logic
    sd = model.state_dict()
    for k in sd:
        t = sd[k].to(dev)
        dist.broadcast(t, src=0)
        sd[k] = t.cpu()
    model.load_state_dict(sd)


def consume_loader_seed(n_rows, batch_size):
    """draw from torch's default generator what iter() of the reference's DataLoader(shuffle=False) over n_rows rows
    draws (its base seed), by making that iterator over a placeholder of the same length"""
    iter(torch.utils.data.DataLoader(range(n_rows), batch_size=batch_size, shuffle=False))


# Device memory kept free of training tables (torch's allocator, the library's per-call scratch, other work on the GPU)
DEVICE_TABLE_RESERVE = 1 << 30
# Largest device window of a streamed table, per slot.  The upload of the first window is not overlapped with training, so
# windows are kept well below what the budget would allow: 256 MiB is ~10 ms of PCIe and millions of rows per window.
STREAM_WINDOW_MAX_BYTES = 1 << 28


def device_table_budget():
    """bytes of device memory the training tables may take: what cudaMemGetInfo reports free (once the trainer and its
    scratch exist) less DEVICE_TABLE_RESERVE"""
    free, _ = torch.cuda.mem_get_info()
    return max(0, free - DEVICE_TABLE_RESERVE)


def stream_window_rows(row_bytes, batch_size, budget):
    """rows of each of the two device windows a streamed table of `row_bytes` rows gets from `budget` bytes: the largest
    multiple of the batch that fits twice, up to STREAM_WINDOW_MAX_BYTES per window.  MemoryError below one batch."""
    rows = min(budget // 2, STREAM_WINDOW_MAX_BYTES) // row_bytes // batch_size * batch_size
    if rows < batch_size:
        raise MemoryError("device memory left for the training table (%d bytes) does not hold two batches of %d rows of %d "
                          "bytes" % (budget, batch_size, row_bytes))
    return int(rows)


class DeviceBatches:
    """Stands in for the reference's DataLoader(shuffle=False, drop_last=False) (training.py:253-263): the (normalised)
    table plus the batch size.  The table is a CUDA tensor resident in HBM (window_rows None), or a C-contiguous numpy
    array in host memory that every pass streams through two device windows of window_rows rows."""

    def __init__(self, data, batch_size, window_rows=None):
        self.data, self.batch_size, self.window_rows = data, int(batch_size), window_rows

    def __len__(self):
        return (self.data.shape[0] + self.batch_size - 1) // self.batch_size


class DeviceAdam:
    """Stands in for torch.optim.Adam(model.parameters(), lr) (training.py:266): Adam state lives in
    the bb_trainer; `lr` is what LRScheduler adjusts.  precision "fp64": the float64 step of the fused trainer (AE /
    CFD_dense_AE up to FUSED_TRAINER_MAX_FEATURES columns; refuse_fp64_training names what it does not take)."""

    def __init__(self, model, lr, max_batch, l1=False, reg_param=0.0, dropout_seed=0, block_hw=None, swae=False,
                 precision=None, dropout_stream=None):
        """dropout_stream = "torch" (AE_Dropout_BN under precision "fp64"): every epoch draws its dropout masks on the
        device from torch's default CPU generator, as the reference's fit does, and writes the state back.
        AE_Dropout_BN batches beyond dbn_fused_max_batch() train on the layer-by-layer trainer (one process)."""
        if is_fp64(precision):
            refuse_fp64_training(type(model).__name__, getattr(model, "n_features", 0), swae, dropout_stream, max_batch,
                                 dist_env()[1])
        else:
            refuse_dropout_stream(type(model).__name__, precision, dropout_stream)
            refuse_dbn_rank_share(type(model).__name__, max_batch, int(os.environ.get("WORLD_SIZE", "1")))
        self.torch_stream = is_fp64(precision) and dropout_stream == "torch" and hasattr(model, "bn_tensors")
        self.rank, self.world = dist_env()
        broadcast_initial_state(model)
        self.model = model
        self.has_bn = hasattr(model, "bn_tensors")
        self.conv = hasattr(model, "training_spec")
        self.trainer, self.steps = None, 0
        self.lr, self.l1, self.reg_param, self.swae = lr, l1, reg_param, swae
        if swae and (self.conv or self.has_bn or self.world > 1):
            # upstream encodes twice per step with this loss (training.py:66-72): BatchNorm / dropout state would move twice
            raise NotImplementedError("loss_function_swae: dense models without BatchNorm / dropout, one process")
        if self.conv:
            # Conv_AE: (transposed) convolutions as weight-sharing dense layers, BatchNorm2d on batch statistics; the loss
            # divisor is true_data.shape[1] = 1 channel (utils.py:197)
            sp = model.training_spec(*block_hw)
            self.trainer = engine.LayeredTrainer(sp["weights"], sp["biases"], sp["acts"], max_batch, dims=sp["dims"],
                                                 w_maps=sp["w_maps"], bn=sp["bn"], loss_columns=1)
            self.dp = sharded.DataParallelTrainer(self.trainer) if self.world > 1 else None
            return
        w, b = model.linear_tensors()
        if is_fp64(precision):
            # no layered fallback: the float64 step is the fused trainer's; data parallel all-reduces its float64 gradient
            self.trainer = engine.Trainer(w, b, model.n_features, model.z_dim, max_batch,
                                          bn=model.bn_tensors() if self.has_bn else None)
            self.trainer.set_precision("fp64")
            self.dp = sharded.DataParallelTrainer(self.trainer, fused=False) if self.world > 1 else None
            return
        if self.has_bn and self.world == 1 and max_batch > dbn_fused_max_batch():
            # batches the fused AE_Dropout_BN step cannot hold resident: the layer-by-layer trainer, same dropout stream
            self.trainer = engine.LayeredTrainer.dbn(w, b, model.n_features, model.z_dim, max_batch, model.bn_tensors())
        elif not swae and (self.has_bn or model.n_features <= FUSED_TRAINER_MAX_FEATURES):
            try:
                self.trainer = engine.Trainer(w, b, model.n_features, model.z_dim, max_batch,
                                              bn=model.bn_tensors() if self.has_bn else None)
            except Exception:
                if self.has_bn:
                    raise
        if self.trainer is None:
            # wide rows (CFD_dense_AE on flattened 2-D snapshots): the layer-by-layer GEMM trainer
            self.trainer = engine.LayeredTrainer(w, b, ["leaky", "leaky", "leaky", "none"] * 2, max_batch)
        self.dp = sharded.DataParallelTrainer(self.trainer, fused=not l1) if self.world > 1 else None
        if self.has_bn:
            # fused data parallel: one dropout stream keyed by the global batch row, the same on every rank; otherwise every
            # rank draws its own
            fused = self.dp is not None and self.dp.fused
            self.trainer.set_dropout(seed=dropout_seed + (0 if fused else self.rank))

    def hyper(self, world_size=None):
        return engine.make_hyper(lr=self.lr, reg_param=self.reg_param, l1=self.l1,
                                 world_size=self.world if world_size is None else world_size)

    def epoch(self, data, batch_size, window_rows=None):
        """one pass over `data` in the reference's batch order; data-parallel when launched with several ranks.  A numpy
        `data` streams from host memory in windows of `window_rows` rows (DeviceBatches)"""
        self.steps += (data.shape[0] + batch_size - 1) // batch_size
        if self.torch_stream:
            # the reference's fit iterates a fresh iter(train_dl) (one draw for its base seed), then draws every mask
            consume_loader_seed(data.shape[0], batch_size)
            self.trainer.set_dropout_torch()
            loss = self.trainer.epoch(data, batch_size, self.hyper(), window_rows)
            self.trainer.write_back_dropout_torch()
            return loss
        if self.dp is None:
            return self.trainer.epoch(data, batch_size, self.hyper(), window_rows)
        return self.dp.epoch_table(data, batch_size, self.hyper(), self.rank, self.world, window_rows)

    SWAE_PROJECTIONS, SWAE_REG_WEIGHT = 2000, 100.0  # defaults of utils.loss_function_swae (utils.py:27-36)

    def epoch_swae(self, data, batch_size, latent_dim):
        """one pass with config.custom_loss_function = "loss_function_swae" (training.py:70-78).  The two random inputs of
        utils.compute_swd are drawn here from torch's global CPU generator in the reference's order - randn_like(z), then
        randn(num_projections, latent_dim) normalised per row (utils.py:57-90) - in float32 (upstream cannot run this loss on
        the float64 AE: its float32 projections meet a double latent), and handed to the device step."""
        tr = self.trainer
        tr.loss_accum.zero_()
        n_batches = 0
        for r0 in range(0, data.shape[0], batch_size):
            xb = data[r0:r0 + batch_size]
            if isinstance(xb, np.ndarray):  # a table in host memory: one batch on the device at a time
                xb = torch.from_numpy(np.ascontiguousarray(xb)).to(tr.loss_accum.device)
            prior = torch.randn((xb.shape[0], latent_dim), dtype=torch.float32)
            proj = torch.randn(self.SWAE_PROJECTIONS, latent_dim)
            proj = proj / proj.norm(dim=1).view(-1, 1)
            tr.step_swae(xb, self.hyper(), prior.cuda(), proj.cuda(), latent_layer=3, reg_weight=self.SWAE_REG_WEIGHT)
            n_batches += 1
        self.steps += n_batches
        return tr.loss_accum.item() / n_batches

    def sync_model(self):
        if self.conv:
            w, b = self.trainer.get_params()
            self.model.load_trained(w, b, self.trainer.get_bn(), self.steps)
            self.steps = 0
            return
        w, b = self.trainer.get_params()
        self.model.set_linear_tensors(w, b)
        if self.has_bn:
            self.model.set_bn_tensors(self.trainer.get_bn())


def fit(config, model, train_dl, model_children, regular_param, optimizer, latent_dim, RHO, l1, n_dimensions):
    """One epoch (reference training.py:31-101).  Returns (epoch_loss, mse_loss, l1_loss, model); the
    reference always evaluates the loss with validate=True, i.e. without the L1 term (SURVEY F2) -
    the L1 branch is opt-in through `config.l1_in_training`."""
    print("### Beginning Training")
    model.train()
    if hasattr(config, "custom_loss_function") and config.custom_loss_function == "loss_function_swae":
        epoch_loss = optimizer.epoch_swae(train_dl.data, train_dl.batch_size, latent_dim)
    else:
        epoch_loss = optimizer.epoch(train_dl.data, train_dl.batch_size, train_dl.window_rows)
    print(f"# Finished. Training Loss: {epoch_loss:.6f}")
    return epoch_loss, epoch_loss, 0, model


def validate(model, test_dl, model_children, reg_param, optimizer=None):
    """reference training.py:104-137: eval-mode forward + sum-MSE / n_columns, mean over batches"""
    print("### Beginning Validating")
    model.eval()
    if getattr(optimizer, "torch_stream", False):
        consume_loader_seed(test_dl.data.shape[0], test_dl.batch_size)  # the reference's iter(test_dl)
    epoch_loss = optimizer.trainer.validate(test_dl.data, test_dl.batch_size, test_dl.window_rows)
    print(f"# Finished. Validation Loss: {epoch_loss:.6f}")
    return epoch_loss


def _refuse_table_model(config):
    if config.data_dimension == 2 and config.model_type == "convolutional" and config.model_name != "Conv_AE":
        raise NotImplementedError("convolutional models other than Conv_AE: see DESIGN.md (out of scope)")


def _training_table(data, config):
    """the (normalised) table as the trainers read it, in host memory: C-contiguous rows of float32, or float64 as it is
    under precision "fp64" (the float64 step widens a float32 table exactly, as the reference's torch.tensor(...,
    float64) does, training.py:230)"""
    arr = np.asarray(data)
    dtype = np.float64 if is_fp64(getattr(config, "precision", None)) and arr.dtype == np.float64 else np.float32
    if config.data_dimension == 2:
        _refuse_table_model(config)
        # dense: (N, H * W) rows (training.py:195-204); Conv_AE: (N, 1, H, W) batches (:222-228), the same memory
        arr = arr.reshape(arr.shape[0], arr.shape[1] * arr.shape[2])
    return np.ascontiguousarray(arr, dtype=dtype)


def _to_device_table(data, config):
    """the (normalised) table resident on the device (_training_table's rows)"""
    return torch.from_numpy(_training_table(data, config)).cuda()


def _place_table(data, config, batch_size, budget, window_rows=None):
    """(table, window_rows, device bytes it holds): the table resident on the device when it fits `budget` bytes, else
    the host table streamed in windows - `window_rows` when given (the windows another streamed table already holds),
    else the largest the budget allows (stream_window_rows).  Both run the same steps and give the same bits."""
    arr = _training_table(data, config)
    if arr.nbytes <= budget:
        return _to_device_table(data, config), None, arr.nbytes
    row_bytes = max(1, arr.strides[0])
    window_rows = window_rows or stream_window_rows(row_bytes, batch_size, budget)
    return arr, window_rows, 2 * window_rows * row_bytes


def train(model, variables, train_data, test_data, project_path, config):
    """reference training.py:150-348.  Same side effects: `loss_data.npy` ([train; val] per epoch),
    optional `model_{epoch}.pt`, `activations.npy`; returns the trained model."""
    from . import helper

    dist_env()  # under torchrun: pick this rank's GPU before anything is allocated on a device
    if config.deterministic_algorithm:
        import random

        random.seed(0)
        torch.manual_seed(0)
        np.random.seed(0)
    bs = config.batch_size
    _refuse_table_model(config)  # before the trainer is built
    model_children = list(model.children())
    conv = config.data_dimension == 2 and config.model_type == "convolutional"
    optimizer = DeviceAdam(model, config.lr, max_batch=bs, l1=bool(getattr(config, "l1_in_training", False)),
                           reg_param=config.reg_param, dropout_seed=int(torch.initial_seed()) & 0x7FFFFFFFFFFFFFFF,
                           block_hw=tuple(np.asarray(train_data).shape[1:3]) if conv else None,
                           swae=getattr(config, "custom_loss_function", None) == "loss_function_swae",
                           precision=getattr(config, "precision", None),
                           dropout_stream=getattr(config, "dropout_stream", None))
    # tables that fit the device memory the trainer left are resident; larger ones stream from host memory
    budget = device_table_budget()
    train_ds, train_win, used = _place_table(train_data, config, bs, budget)
    if test_data is train_data:
        valid_ds, valid_win = train_ds, train_win
    else:
        valid_ds, valid_win, _ = _place_table(test_data, config, bs, budget - used, train_win)
    train_dl, valid_dl = DeviceBatches(train_ds, bs, train_win), DeviceBatches(valid_ds, bs, valid_win)
    early_stopping = utils.EarlyStopping(config.early_stopping_patience, config.min_delta) if config.early_stopping else None
    lr_scheduler = utils.LRScheduler(optimizer, config.lr_scheduler_patience) if config.lr_scheduler else None
    train_loss, val_loss = [], []
    start = time.time()
    for epoch in range(config.epochs):
        print(f"Epoch {epoch + 1} of {config.epochs}")
        train_epoch_loss, _, _, _ = fit(config, model, train_dl, model_children, config.reg_param, optimizer,
                                        getattr(config, "latent_space_size", None), config.RHO, config.l1,
                                        config.data_dimension)
        train_loss.append(train_epoch_loss)
        if config.test_size:
            val_epoch_loss = validate(model, valid_dl, model_children, config.reg_param, optimizer)
        else:
            val_epoch_loss = train_epoch_loss
        val_loss.append(val_epoch_loss)
        if lr_scheduler:
            lr_scheduler(val_epoch_loss)
        if early_stopping:
            early_stopping(val_epoch_loss)
            if early_stopping.early_stop:
                break
        if config.intermittent_model_saving and epoch % config.intermittent_saving_patience == 0:
            optimizer.sync_model()
            if optimizer.rank == 0:
                helper.model_saver(model, os.path.join(project_path, f"model_{epoch}.pt"))
    end = time.time()
    optimizer.sync_model()
    if optimizer.rank == 0:  # replicas are identical: one writer
        if getattr(config, "activation_extraction", False):
            np.save(os.path.join(project_path, "activations.npy"), optimizer.trainer.activation_means())
        np.save(os.path.join(project_path, "loss_data.npy"), np.array([train_loss, val_loss]))
        if conv:
            # reference training.py:344-346: the conv-stack output shape of the LAST forward, which is validate()'s last
            # batch when test_size > 0, else the last training batch; decompress reads its batch size back (helper.py:650-688)
            last = valid_dl if config.test_size else train_dl
            rows = last.data.shape[0] - (last.data.shape[0] - 1) // bs * bs
            model.set_final_layer_dims(torch.Size((rows,) + tuple(model._conv_out)))
            np.save(os.path.join(project_path, "final_layer.npy"), np.array(model.get_final_layer_dims()))
    print(f"{(end - start) / 60:.3} minutes")
    return model
