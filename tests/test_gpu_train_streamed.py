"""Training epochs streamed from host memory (bb_trainer_epoch_host / bb_ltrainer_epoch_host and their validate forms):
bit for bit the resident epochs on the same table, for every trainer; row-chunked preprocessing bit for bit the
whole-table passes; the CLI with a small device budget writes the resident run's files; device memory stays bounded."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

from baler_b200 import engine, synth
from baler_b200.modules import data_processing, models, training

pytestmark = pytest.mark.gpu
BATCHES_PER_WINDOW = 3


def _bytes(obj):
    """the bits of nested lists / dicts / arrays / numbers (NaN-exact)"""
    if isinstance(obj, dict):
        return b"".join(k.encode() + _bytes(obj[k]) for k in sorted(obj))
    if isinstance(obj, (list, tuple)):
        return b"".join(_bytes(o) for o in obj)
    if isinstance(obj, torch.Tensor):
        return obj.detach().cpu().numpy().tobytes()
    return np.asarray(obj).tobytes()


def _state(tr):
    """parameters, the last step's gradient and batch loss, BatchNorm parameters / running statistics /
    num_batches_tracked, activation means"""
    out = [tr.params_view(), tr.grads_view(), tr.get_params()]
    if getattr(tr, "_bn", None) is not None:
        out.append(tr.get_bn())
    try:
        out.append(tr.activation_means())
    except NotImplementedError:  # (Conv_AE: not an 8-Linear autoencoder)
        pass
    return _bytes(out)


def _epoch(tr, x, batch, hyper, **kw):
    return tr.epoch(x, batch, hyper, **kw)


def _run_pair(make, table, batch, hyper, epoch=_epoch, epochs=2):
    """the same trainer built twice: resident epochs + validate on one, streamed ones (windows of 3 batches, a ragged last
    batch) on the other; then one more resident epoch on both, so that equal parameters afterwards pin Adam's m and v"""
    assert table.shape[0] % batch and table.shape[0] > 2 * BATCHES_PER_WINDOW * batch
    runs = []
    for streamed in (False, True):
        tr = make()
        x = table if streamed else torch.from_numpy(table).cuda()
        kw = {"window_rows": BATCHES_PER_WINDOW * batch} if streamed else {}
        losses = [epoch(tr, x, batch, hyper, **kw) for _ in range(epochs)]
        losses.append(tr.validate(x, batch, **kw))
        state = _state(tr)
        losses.append(epoch(tr, torch.from_numpy(table[:2 * batch]).cuda(), batch, hyper))
        runs.append((losses, state, _state(tr)))
    assert np.isfinite(runs[0][0]).all()
    assert runs[0][0] == runs[1][0], (runs[0][0], runs[1][0])
    assert runs[0][1] == runs[1][1]
    assert runs[0][2] == runs[1][2]
    return runs[0][0]


def _table(n, dtype=np.float32, seed=3):
    x = synth.cms_table(n, seed=seed).astype(np.float64)
    x = (x - x.min(0)) / (x.max(0) - x.min(0))
    return np.ascontiguousarray(x, dtype=dtype)


def _ae(precision=None, max_batch=512):
    torch.manual_seed(0)
    w, b = models.AE(24, 15).linear_tensors()

    def make():
        tr = engine.Trainer(w, b, 24, 15, max_batch)
        if precision:
            tr.set_precision(precision)
        return tr
    return make


def _dbn_model():
    torch.manual_seed(1)
    m = models.AE_Dropout_BN(24, 15)
    return m.linear_tensors(), m.bn_tensors()


@pytest.mark.parametrize("precision,l1,dtype", [(None, False, np.float32), ("fp32", False, np.float32),
                                                ("fp32", True, np.float32), ("fp64", False, np.float32),
                                                ("fp64", False, np.float64), ("fp64", True, np.float64)])
def test_ae_streamed_equals_resident(precision, l1, dtype):
    tr = _ae(precision)()
    assert tr.precision == (precision or "split16")
    hyper = engine.make_hyper(lr=1e-3, l1=l1, reg_param=1e-3)
    _run_pair(_ae(precision), _table(10 * 512 + 37, dtype), 512, hyper)


def test_dbn_fused_philox_streamed_equals_resident():
    (w, b), bn = _dbn_model()

    def make():
        tr = engine.Trainer(w, b, 24, 15, 512, bn=bn)
        assert tr.precision == "split16"
        tr.set_dropout(seed=11)
        return tr
    _run_pair(make, _table(10 * 512 + 101), 512, engine.make_hyper(lr=1e-3))


def test_dbn_fp64_torch_stream_streamed_equals_resident():
    (w, b), bn = _dbn_model()
    gens = []

    def make():
        tr = engine.Trainer(w, b, 24, 15, 256, bn=bn)
        tr.set_precision("fp64")
        gens.append(torch.Generator().manual_seed(5))
        return tr

    def epoch(tr, x, batch, hyper, **kw):
        tr.set_dropout_torch(gens[-1])
        loss = tr.epoch(x, batch, hyper, **kw)
        tr.write_back_dropout_torch()
        return loss
    _run_pair(make, _table(10 * 256 + 19, np.float64), 256, engine.make_hyper(lr=1e-3), epoch=epoch)
    assert gens[0].get_state().numpy().tobytes() == gens[1].get_state().numpy().tobytes()


def test_dbn_layered_streamed_equals_resident():
    (w, b), bn = _dbn_model()

    def make():
        tr = engine.LayeredTrainer.dbn(w, b, 24, 15, 4096, bn)
        tr.set_dropout(seed=13)
        return tr
    _run_pair(make, _table(7 * 4096 + 1001), 4096, engine.make_hyper(lr=1e-3))


def test_cfd_dense_wide_streamed_equals_resident():
    torch.manual_seed(2)
    w, b = models.CFD_dense_AE(2500, 100).linear_tensors()
    x = synth.cfd_snapshots(7 * 64 + 9, seed=4).reshape(-1, 2500)
    x = np.ascontiguousarray((x - x.min()) / (x.max() - x.min()), dtype=np.float32)
    _run_pair(lambda: engine.LayeredTrainer(w, b, ["leaky", "leaky", "leaky", "none"] * 2, 64), x, 64,
              engine.make_hyper(lr=1e-3))


def test_conv_ae_streamed_equals_resident():
    torch.manual_seed(0)
    sp = models.Conv_AE(5, 250).training_spec(5, 5)
    x = synth.cfd_snapshots(8, seed=6).reshape(-1, 25)  # 5 x 5 blocks, 800 rows
    x = np.ascontiguousarray((x - x.min()) / (x.max() - x.min()), dtype=np.float32)

    def make():
        return engine.LayeredTrainer(sp["weights"], sp["biases"], sp["acts"], 64, dims=sp["dims"], w_maps=sp["w_maps"],
                                     bn=sp["bn"], loss_columns=1)
    _run_pair(make, x, 64, engine.make_hyper(lr=1e-3))


def test_swae_host_table_equals_resident():
    """loss_function_swae uploads one batch at a time from a host table: the same draws, steps and bits"""
    x = _table(7 * 128 + 5)
    out = []
    for table in (torch.from_numpy(x).cuda(), x):
        torch.manual_seed(0)
        m = models.AE(24, 15)
        opt = training.DeviceAdam(m, 1e-3, max_batch=128, swae=True)
        losses = [opt.epoch_swae(table, 128, 15) for _ in range(2)]
        out.append((losses, _state(opt.trainer), _bytes(torch.get_rng_state())))
    assert out[0] == out[1]


def test_window_must_hold_whole_batches():
    tr = _ae()()
    x = _table(1000)
    for bad in (0, 100, 512 + 1, 3 * 512 - 1):
        with pytest.raises(ValueError):
            tr.epoch(x, 512, engine.make_hyper(), window_rows=bad)
    from baler_b200 import _lib
    out, hyper = ctypes.c_double(), engine.make_hyper()
    rc = _lib.lib().bb_trainer_epoch_host(tr.handle, x.ctypes.data, engine.BB_F32, 1000, 512, ctypes.byref(hyper), 700,
                                          ctypes.byref(out), None)
    assert rc == -1  # BB_ERR_INVALID
    # a float64 table is for float64 trainers only
    with pytest.raises(_lib.BalerB200Error):
        tr.epoch(x.astype(np.float64), 512, hyper, window_rows=512)


def test_streamed_epoch_device_memory_is_bounded():
    """device memory in use grows by the two windows (kept for the next epoch) and a margin, not by the table"""
    batch, win = 512, 64 * 512
    x = _table(2_000_000 + 37)
    row = x.strides[0]
    tr = _ae()()
    tr.epoch(torch.from_numpy(x[:4096]).cuda(), batch, engine.make_hyper())  # the trainer's scratch exists
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    tr.epoch(x, batch, engine.make_hyper(), window_rows=win)
    grown = free0 - torch.cuda.mem_get_info()[0]
    margin = 16 << 20  # allocation granularity and the per-step hyper-parameter buffer of a window
    print("device memory grown by %d bytes for a %d-byte table (windows 2 x %d)" % (grown, x.nbytes, win * row))
    assert grown <= 2 * win * row + margin and grown < x.nbytes // 4


# ---------------------------------------------------------------- row-chunked preprocessing


def _pre_cases():
    f32 = synth.cms_table(30_011, seed=9)
    nan = f32.copy()
    nan[777, 4] = np.nan
    ill = f32.astype(np.float64)
    ill[:, 5] = 1.0e9 + np.arange(len(ill)) % 977  # offset >> spread: the exact float64 host path
    snaps = synth.cfd_snapshots(12, seed=2)
    return {"float32": f32, "float64": f32.astype(np.float64) * 1.5, "nan_column": nan, "ill_conditioned": ill,
            "dense_2d": snaps, "conv_blocks": data_processing.convert_to_blocks_util([1, 5, 5], snaps)}


@pytest.mark.parametrize("case", sorted(_pre_cases()))
def test_chunked_preprocessing_equals_whole_table(case, monkeypatch):
    data = _pre_cases()[case]

    def results():
        feats = data_processing.find_minmax(data)
        normed = data_processing.normalize(data, False)
        flat = np.asarray(normed).reshape(len(normed), -1)
        f2 = np.asarray(feats).reshape(2, -1)
        out = [feats, normed, data_processing.renormalize_func(flat, f2[0], f2[1])]
        if data.dtype == np.float64:
            out.append(data_processing.minmax_normalize_f64(data))
        return _bytes(out)
    whole = results()
    monkeypatch.setattr(data_processing, "PREPROCESS_CHUNK_BYTES", 4096 + 8)  # many chunks, a ragged last one
    assert results() == whole


# ---------------------------------------------------------------- the CLI with a small device budget


def _cli_files(out, conv):
    names = ["training/loss_data.npy", "training/normalization_features.npy"]
    names += ["training/final_layer.npy"] if conv else ["training/activations.npy"]
    files = {n: open(os.path.join(out, n), "rb").read() for n in names}
    sd = torch.load(os.path.join(out, "compressed_output", "model.pt"))
    files.update({k: _bytes(v) for k, v in sd.items()})
    return files


def _cli_run(tmp_path, monkeypatch, sub, table, budget, conv=False, **cfg_extra):
    from baler_b200 import baler
    from baler_b200.modules import helper
    from test_gpu_train_fp64 import _cfg, _project
    d = tmp_path / sub
    d.mkdir()
    out, path = _project(d, monkeypatch, table)
    cfg = _cfg(helper, path, **cfg_extra)
    if conv:
        cfg.data_dimension, cfg.model_type, cfg.convert_to_blocks, cfg.compression_ratio = 2, "convolutional", [1, 5, 5], 10
    seen = []
    monkeypatch.setattr(training, "device_table_budget", lambda: budget)
    real = training.DeviceBatches.__init__

    def spy(self, data, batch_size, window_rows=None):
        seen.append(window_rows)
        real(self, data, batch_size, window_rows)
    monkeypatch.setattr(training.DeviceBatches, "__init__", spy)
    if budget < 1 << 30:
        monkeypatch.setattr(data_processing, "PREPROCESS_CHUNK_BYTES", 64 << 10)
    torch.manual_seed(0)
    baler.perform_training(out, cfg, False)
    files = _cli_files(out, conv)
    monkeypatch.undo()
    return files, seen


CLI_CASES = {
    "cms_ae_test_size": (lambda: synth.cms_table(20_000, seed=21), False,
                         dict(precision="auto", test_size=0.2, l1=False, epochs=2), 1 << 20),
    "fp64_dbn_torch_stream": (lambda: synth.cms_table(6_000, seed=22).astype(np.float64), False,
                              dict(model_name="AE_Dropout_BN", precision="fp64", dropout_stream="torch", batch_size=256,
                                   test_size=0.2, l1=False, epochs=2, early_stopping=False, lr_scheduler=False), 1 << 19),
    "conv_ae_blocks": (lambda: synth.cfd_snapshots(6).astype(np.float32), True,
                       dict(model_name="Conv_AE", precision="auto", batch_size=200, test_size=0, l1=False, epochs=3,
                            apply_normalization=True, custom_norm=False, activation_extraction=False,
                            early_stopping=False, lr_scheduler=False, deterministic_algorithm=True), 48_000),
}


@pytest.mark.parametrize("case", sorted(CLI_CASES))
def test_cli_streamed_writes_the_resident_files(case, tmp_path, monkeypatch):
    make, conv, extra, budget = CLI_CASES[case]
    table = make()
    resident, seen_r = _cli_run(tmp_path, monkeypatch, "resident", table, 1 << 40, conv, **extra)
    streamed, seen_s = _cli_run(tmp_path, monkeypatch, "streamed", table, budget, conv, **extra)
    assert all(w is None for w in seen_r) and seen_s and all(w is not None for w in seen_s), (seen_r, seen_s)
    assert all(w % extra.get("batch_size", 512) == 0 for w in seen_s)
    assert sorted(resident) == sorted(streamed)
    for k in resident:
        assert resident[k] == streamed[k], k


# ---------------------------------------------------------------- two ranks


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        x = _table(12 * 1024 + 77)
        torch.manual_seed(0)
        w, b = models.AE(24, 15).linear_tensors()
        res = []
        for streamed in (False, True):
            tr = engine.Trainer(w, b, 24, 15, 512)
            tr.dp_connect()
            hyper = engine.make_hyper(lr=1e-3, world_size=world)
            table = x if streamed else torch.from_numpy(x).cuda()
            kw = {"window_rows": 3 * 1024} if streamed else {}
            losses = [tr.epoch(table, 1024, hyper, **kw) for _ in range(2)]
            res.append(np.concatenate([losses, tr.params_view().cpu().numpy().astype(np.float64)]))
        np.save(os.path.join(out_dir, "dp_%d.npy" % rank), np.stack(res))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_streamed_equals_resident(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_dp_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "dp_0.npy"), np.load(tmp_path / "dp_1.npy")
    assert r0[0].tobytes() == r0[1].tobytes() and r1[0].tobytes() == r1[1].tobytes()
    assert r0[1, 2:].tobytes() == r1[1, 2:].tobytes()  # replicas
