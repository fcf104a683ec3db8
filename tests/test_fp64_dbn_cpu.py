"""Float64 AE_Dropout_BN training without a device: the new entry points are declared, bound and exported; the numpy
restatement of torch's dropout stream and the torch twin reproduce the reference's fixture; the generator-state parse
and write-back round trip; dropout_stream is refused where it cannot be honoured, before anything is written; no CPU
fallback."""
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import rel_max, sub_sd
from dbn_reference import DROPOUT_P, bernoulli_masks, mt19937_from, twin_from_state, loss_fn
from oracle import baler_oracle as orc
from baler_b200 import _lib, build, engine, synth
from baler_b200.modules import models, training
from test_fp64_train_cpu import _workspace, _written

SYMBOLS = ("bb_trainer_set_dropout_mt19937", "bb_trainer_get_dropout_mt19937", "bb_trainer_bn_running_dev_f64")
WIDTHS = (200, 100, 50, 15)


def test_dbn_fp64_symbols_declared_bound_and_exported():
    build.build()
    hdr = open(os.path.join(os.path.dirname(_lib.HERE), "include", "baler_b200.h")).read()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in SYMBOLS:
        assert name + "(" in hdr and name in _lib.exported_symbols() and (" T " + name) in out, name


@pytest.mark.parametrize("shape", [(512, 200), (7, 13), (1, 1), (33, 15), (3, 1001)])
@pytest.mark.parametrize("p", DROPOUT_P)
def test_numpy_stream_equals_bernoulli(shape, p):
    torch.manual_seed(11)
    torch.rand(37)  # start mid-block
    mt = mt19937_from()
    for _ in range(3):
        ref = torch.empty(shape, dtype=torch.float64).bernoulli_(1 - p).numpy().astype(bool)
        (got,) = bernoulli_masks(mt, shape[0], (shape[1],), (p,))
        assert np.array_equal(got, ref)


def test_numpy_stream_across_batches_with_a_ragged_one():
    torch.manual_seed(3)
    mt = mt19937_from()
    for rows in (512, 512, 512, 89):
        ref = [torch.empty(rows, w, dtype=torch.float64).bernoulli_(1 - p).numpy().astype(bool) for w, p in zip(WIDTHS, DROPOUT_P)]
        got = bernoulli_masks(mt, rows, WIDTHS)
        assert all(np.array_equal(a, b) for a, b in zip(got, ref))
    key, pos = engine.mt19937_from_torch_state(torch.get_rng_state())
    st = mt.state["state"]
    assert pos == st["pos"] and np.array_equal(key, st["key"])


def test_numpy_stream_equals_fixture_masks(golden):
    g = golden("ae_dbn.npz")
    torch.manual_seed(5)
    got = bernoulli_masks(mt19937_from(), 512, WIDTHS)
    for i in range(4):
        assert np.array_equal(got[i], g["mask%d" % i]), i


def test_state_write_back_round_trip_and_loader_draw():
    torch.manual_seed(17)
    torch.rand(1001)
    blob = torch.get_rng_state()
    key, pos = engine.mt19937_from_torch_state(blob)
    ref = torch.rand(8)
    torch.set_rng_state(engine.mt19937_to_torch_state(blob, key, pos))
    assert torch.equal(torch.rand(8), ref)
    # draw a batch's masks from numpy's copy of the stream and write its state back: torch continues where its own
    # bernoulli_ calls would have left it
    torch.set_rng_state(blob)
    mt = mt19937_from()
    bernoulli_masks(mt, 77, WIDTHS)
    st = mt.state["state"]
    torch.set_rng_state(engine.mt19937_to_torch_state(torch.get_rng_state(), st["key"], st["pos"]))
    got = torch.rand(8)
    torch.set_rng_state(blob)
    for w, p in zip(WIDTHS, DROPOUT_P):
        torch.empty(77, w, dtype=torch.float64).bernoulli_(1 - p)
    assert torch.equal(got, torch.rand(8))
    # the placeholder iter() draws what iter() of a DataLoader over a real table draws
    x = torch.from_numpy(synth.cms_table(1000, seed=1).astype(np.float64))
    torch.manual_seed(2)
    iter(torch.utils.data.DataLoader(x, batch_size=512, shuffle=False, drop_last=False))
    a = torch.rand(4)
    torch.manual_seed(2)
    training.consume_loader_seed(1000, 512)
    assert torch.equal(torch.rand(4), a)
    torch.manual_seed(2)
    assert not torch.equal(torch.rand(4), a)  # it does draw


def test_torch_twin_reproduces_fixture_step(golden):
    """the twin's first step after manual_seed(5) is the reference's (its masks are the fixture's)"""
    g = golden("ae_dbn.npz")
    sd0, sd1, gref = sub_sd(g, "sd0"), sub_sd(g, "sd1"), sub_sd(g, "g")
    m = twin_from_state(sd0)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    x = torch.from_numpy(g["x_norm"][:512].astype(np.float64))
    torch.manual_seed(5)
    m.train()
    opt.zero_grad()
    recon = m(x)
    loss = loss_fn(recon, x)
    loss.backward()
    assert abs(loss.item() - float(g["loss_train"])) <= 1e-12 * float(g["loss_train"])
    assert rel_max(recon.detach().numpy(), g["recon_train"]) <= 1e-11
    named = dict(m.named_parameters())
    gscale = max(np.abs(v).max() for v in gref.values())
    for k, v in gref.items():
        assert np.abs(named[k].grad.numpy() - v).max() <= 1e-11 * gscale, k
    opt.step()
    sd = m.state_dict()
    for b in models.AE_Dropout_BN.bn_names:
        for s in ("running_mean", "running_var"):
            assert rel_max(sd[b + "." + s].numpy(), sd1[b + "." + s]) <= 1e-12, (b, s)
        assert int(sd[b + ".num_batches_tracked"]) == int(sd1[b + ".num_batches_tracked"])
    # Adam as test_dbn_train_step_golden bounds the oracle's step
    _, _, grads, _ = orc.dbn_train_step(sd0, g["x_norm"][:512], [g["mask%d" % i].astype(np.float64) for i in range(4)])
    ref = np.concatenate([gref[k].ravel() for k in gref])
    live = np.abs(ref) > 1e-6 * np.abs(ref).max()
    got = np.concatenate([sd[k].numpy().ravel() for k in gref])
    want = np.concatenate([sd1[k].ravel() for k in gref])
    assert np.abs(got - want)[live].max() <= 1e-9 and np.abs(got - want).max() <= 1.001e-3


def _dbn_workspace(tmp_path, monkeypatch, **extra):
    cfg_extra = dict(model_name="AE_Dropout_BN", l1=False)
    cfg_extra.update(extra)
    return _workspace(tmp_path, monkeypatch, synth.cms_table(64, seed=1), **cfg_extra)


@pytest.mark.parametrize("case", ["fp32", "split16", "world2", "batch600", "unknown"])
def test_dropout_stream_refusals_before_anything_is_written(tmp_path, monkeypatch, case):
    from baler_b200 import baler
    from baler_b200.modules import helper

    def no_device(*a, **k):
        raise AssertionError("the device was touched before the refusal")
    monkeypatch.setattr(helper, "process", no_device)
    extra = {"dropout_stream": "torch"}
    err, match = NotImplementedError, "dropout_stream"
    if case in ("fp32", "split16"):
        extra["precision"] = case
    elif case == "world2":
        monkeypatch.setenv("WORLD_SIZE", "2")
        match = "one process"
    elif case == "batch600":
        extra["batch_size"] = 600
        match = "batch_size <= 592"
        monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    else:
        extra["dropout_stream"] = "philox"
        err = ValueError
    out, cfg = _dbn_workspace(tmp_path, monkeypatch, **extra)
    with pytest.raises(err, match=match):
        baler.perform_training(out, cfg, False)
    assert _written(out) == []


def test_dropout_stream_refusals_of_device_adam(monkeypatch):
    model = models.AE_Dropout_BN(24, 15)
    with pytest.raises(NotImplementedError, match="dropout_stream"):
        training.DeviceAdam(model, 1e-3, 64, precision="fp64")  # fp64 without the key: names the key
    with pytest.raises(NotImplementedError, match="precision = 'fp64'"):
        training.DeviceAdam(model, 1e-3, 64, dropout_stream="torch")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(NotImplementedError, match="592"):
        training.DeviceAdam(model, 1e-3, 593, precision="fp64", dropout_stream="torch")
    assert training.fp64_dbn_max_batch() == 592


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fp64_dbn_training_has_no_cpu_fallback(tmp_path, monkeypatch):
    from baler_b200 import baler
    out, cfg = _dbn_workspace(tmp_path, monkeypatch, dropout_stream="torch")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        baler.perform_training(out, cfg, False)
    assert _written(out) == []
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        training.DeviceAdam(models.AE_Dropout_BN(24, 15), 1e-3, 64, precision="fp64", dropout_stream="torch")
