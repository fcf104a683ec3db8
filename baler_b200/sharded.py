"""Multi-GPU host logic: one process per GPU (torch.distributed), rows sharded contiguously.

compress / decompress: no collective on the data path; the only exchange is the 2 x n_features
column min / max (all-reduce MIN and MAX) when normalisation features are recomputed from the input
(reference helper.py:500-502 computes them over the whole file).
training: data-parallel; every global batch (reference order, shuffle=False) is cut into `world`
contiguous sub-batches; the flat gradient (+ batch loss in its last slot) is all-reduced with SUM -
not mean - because the reference loss is a sum over rows (utils.py:195-199), then every rank applies
the identical Adam step.
"""
import numpy as np
import torch
import torch.distributed as dist


def dist_env():
    """(rank, world).  Launched under torchrun (`python -m torch.distributed.run --nproc-per-node N -m baler_b200 ...`)
    the CLI modes run one process per GPU over NCCL; otherwise (one process) rank 0 of 1.  Picks this rank's GPU before
    anything is allocated on a device."""
    import os
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and not dist.is_initialized():
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def row_range(n_rows, rank, world, align=1):
    """contiguous shard [lo, hi) of n_rows rows for `rank` (first n_rows % world ranks get one extra row).  With `align` > 1
    the shards are cut from whole groups of `align` rows (the 128-row blocks of a q8 latent) the same way, so every shard
    starts on a group boundary; only the last group may be short."""
    if align > 1:
        lo, hi = row_range((n_rows + align - 1) // align, rank, world)
        return min(n_rows, lo * align), min(n_rows, hi * align)
    base, extra = divmod(n_rows, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def dp_batch_slices(n_rows, global_batch, rank, world):
    """[(lo, hi)] global row ranges this rank processes, one per global batch (drop_last=False: the last
    batch is ragged and a rank's slice of it may be empty)"""
    out = []
    for b0 in range(0, n_rows, global_batch):
        rows = min(global_batch, n_rows - b0)
        lo, hi = row_range(rows, rank, world)
        out.append((b0 + lo, b0 + hi))
    return out


def combine_minmax_(mn, mx, group=None):
    """in-place global column min / max over all ranks: ONE MIN all-reduce of [min | -max] (2 x C values; negation is
    exact, so max = -min(-max) bit for bit)"""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        c = mn.numel()
        both = torch.cat([mn.reshape(-1), -mx.reshape(-1)])
        dist.all_reduce(both, op=dist.ReduceOp.MIN, group=group)
        mn.copy_(both[:c].reshape(mn.shape))
        mx.copy_((-both[c:]).reshape(mx.shape))
    return mn, mx


def allreduce_sum_(flat, group=None):
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    return flat


class DataParallelTrainer:
    """engine.Trainer on every rank + SUM all-reduce of the flat gradient between backward and Adam."""

    def __init__(self, trainer, group=None, fused=True):
        self.trainer, self.group = trainer, group
        self.grads = trainer.grads_view()  # n_params + 1 floats: gradient, then the batch loss
        # the tensor-core step exchanges its gradient tiles itself (NVLink peer memory, fused with the weight-gradient
        # phase): no collective and no host loop per step.  AE_Dropout_BN on that path also exchanges the BatchNorm sums
        # at its 8 reduction points, i.e. it normalises with the statistics of the GLOBAL batch and keys the dropout
        # stream by global row: the replicas compute exactly what one GPU computes at batch_size = global batch
        # (models.py:256-313 under training.py:253-263).  Everything else (fp32 step, the layered trainer, the CPU
        # stand-in of the gloo tests) all-reduces the flat gradient between the two phases.
        self.fused = False
        if (fused and hasattr(trainer, "dp_connect") and dist.is_initialized()
                and dist.get_backend(group) == "nccl" and dist.get_world_size(group) > 1
                and getattr(trainer, "precision", None) == "split16"):
            trainer.dp_connect(group)
            self.fused = True
        # AE_Dropout_BN without the fused exchange (fused=False, the labelled local-statistics mode): every rank normalises
        # ITS slice of the batch (per-rank BatchNorm statistics, as torch DistributedDataParallel runs the reference model)
        # and draws its own dropout stream; the running statistics are averaged over ranks at the end of an epoch so that
        # the replicas save the same model.pt
        self.bn_running = trainer.bn_running_views() if getattr(trainer, "_bn", None) is not None and not self.fused else None

    def sync_running_stats(self):
        if self.bn_running is None or not (dist.is_available() and dist.is_initialized()):
            return
        world = dist.get_world_size(self.group)
        if world > 1:
            for t in self.bn_running:
                dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
                t.div_(world)

    def step(self, x_local, hyper):
        """x_local: this rank's contiguous slice of the global batch (may have 0 rows)"""
        if x_local.shape[0] > 0:
            self.trainer.step(x_local, hyper, phase=1)
        else:
            self.grads.zero_()
        allreduce_sum_(self.grads, self.group)
        self.trainer.step(x_local if x_local.shape[0] > 0 else self._dummy(x_local), hyper, phase=2)

    def _dummy(self, x_local):
        return torch.zeros((1, x_local.shape[1]), dtype=x_local.dtype, device=x_local.device)

    def epoch_table(self, data, batch_size, hyper, rank, world, window_rows=None):
        """one pass over the full (replicated) table in global batches of `batch_size`; returns the epoch loss.  `data` is
        a CUDA table, or a numpy table in host memory (streamed in windows of `window_rows` rows by the fused step, one
        slice at a time otherwise)"""
        if self.fused:
            # the library returns this rank's share of every batch loss; one reduction per epoch completes the sum
            loss = torch.tensor([self.trainer.epoch(data, batch_size, hyper, window_rows)], dtype=torch.float64,
                                device=self.grads.device)
            dist.all_reduce(loss, op=dist.ReduceOp.SUM, group=self.group)
            return loss.item()
        slices = dp_batch_slices(data.shape[0], batch_size, rank, world)
        return self.epoch((data[lo:hi] for lo, hi in slices), hyper)

    def epoch(self, x_local_batches, hyper):
        """x_local_batches: this rank's slices, one per global batch (CUDA tensors, or numpy arrays uploaded one at a
        time); returns the epoch loss"""
        self.trainer.loss_accum.zero_()
        n = 0
        for xb in x_local_batches:
            if not isinstance(xb, torch.Tensor):
                xb = torch.from_numpy(np.ascontiguousarray(xb)).to(self.grads.device)
            self.step(xb, hyper)
            n += 1
        self.sync_running_stats()
        return self.trainer.loss_accum.item() / max(n, 1)


def global_minmax(shard, group=None):
    """per-column [min; max - min] of the WHOLE table from this rank's row shard (numpy, any float dtype): local min / max,
    then the 2 x C exchange.  Same arithmetic as data_processing.find_minmax (data_processing.py:113-130) on the full
    table: min and max are exact, the range is one subtraction in the table's dtype."""
    import numpy as np
    c = shard.shape[1]
    dev = "cuda" if dist.is_initialized() and dist.get_backend(group) == "nccl" else "cpu"
    if len(shard):
        mn, mx = torch.from_numpy(shard.min(axis=0)).to(dev), torch.from_numpy(shard.max(axis=0)).to(dev)
    else:  # more ranks than rows
        mn = torch.full((c,), float("inf"), dtype=torch.from_numpy(shard[:0]).dtype, device=dev)
        mx = -mn
    combine_minmax_(mn, mx, group)
    mn, mx = mn.cpu().numpy(), mx.cpu().numpy()
    return np.stack([mn, mx - mn])


def gather_rows_to_rank0(shard, n_rows, group=None, chunk_rows=1 << 22, align=1):
    """contiguous row shards (numpy [rows_r, C], rank order = row order, cut by row_range(n_rows, rank, world, align)) ->
    the full [n_rows, C] array on rank 0, None on the other ranks.  Point to point in chunks through a device staging
    buffer, so no rank ever holds more than its own shard plus one chunk on the GPU."""
    import numpy as np
    rank, world = (dist.get_rank(group), dist.get_world_size(group)) if dist.is_initialized() else (0, 1)
    if world == 1:
        return shard
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    c = shard.shape[1]
    if rank == 0:
        out = np.empty((n_rows, c), dtype=shard.dtype)
        out[:len(shard)] = shard
        for src in range(1, world):
            lo, hi = row_range(n_rows, src, world, align)
            for r0 in range(lo, hi, chunk_rows):
                r1 = min(hi, r0 + chunk_rows)
                buf = torch.empty((r1 - r0, c), dtype=torch.from_numpy(shard[:0]).dtype, device=dev)
                dist.recv(buf, src=src, group=group)
                out[r0:r1] = buf.cpu().numpy()
        return out
    for r0 in range(0, len(shard), chunk_rows):
        dist.send(torch.from_numpy(np.ascontiguousarray(shard[r0:r0 + chunk_rows])).to(dev), dst=0, group=group)
    return None


def gather_objects_to_rank0(obj, group=None):
    """[obj of rank 0, obj of rank 1, ...] on rank 0, None on the other ranks (variable-length host data: the
    error-bounded-delta hit lists)"""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return [obj]
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    out = [None] * world if rank == 0 else None
    dist.gather_object(obj, out, dst=0, group=group)
    return out
