"""precision "fp64" training without a device: the float64 training entry points are declared, bound and exported; models,
losses and widths the float64 trainer does not take are refused before anything is read from a device or written; with
no device fp64 training fails like every other compute path (no CPU fallback)."""
import os

import numpy as np
import pytest
import torch

from baler_b200 import _lib, build, synth
from baler_b200.modules import helper, models, training

FP64_TRAIN_SYMBOLS = ("bb_trainer_step_f64", "bb_trainer_epoch_f64", "bb_trainer_validate_f64", "bb_trainer_params_dev_f64",
                      "bb_trainer_grads_dev_f64", "bb_normalize_f64")


def test_fp64_train_symbols_declared_bound_and_exported():
    import subprocess
    build.build()
    hdr = open(os.path.join(os.path.dirname(_lib.HERE), "include", "baler_b200.h")).read()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in FP64_TRAIN_SYMBOLS:
        assert name + "(" in hdr and name in _lib.exported_symbols() and (" T " + name) in out, name
    assert "BB_PREC_FP64" in hdr[hdr.index("bb_trainer_set_precision") - 2000:hdr.index("bb_trainer_set_precision")]


def _workspace(tmp_path, monkeypatch, table, **extra):
    os.makedirs(tmp_path, exist_ok=True)
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("WS", "P")
    path = os.path.join("workspaces", "WS", "data", "P_data.npz")
    np.savez(path, data=table, names=["c%d" % i for i in range(table.shape[-1])])
    out = os.path.join("workspaces", "WS", "P", "output")

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name = 1, 1.6, True, "AE"
        epochs, lr, batch_size, early_stopping, lr_scheduler = 2, 0.001, 512, True, True
        early_stopping_patience, min_delta, lr_scheduler_patience, custom_norm = 100, 0, 50, False
        reg_param, RHO, test_size, extra_compression = 0.001, 0.05, 0, False
        intermittent_model_saving, intermittent_saving_patience = False, 100
        l1, activation_extraction, deterministic_algorithm = True, True, False
        convert_to_blocks, separate_model_saving, save_error_bounded_deltas = False, False, False
        precision = "fp64"
    for k, v in extra.items():
        setattr(cfg, k, v)
    return out, cfg


def _written(out):
    return sorted(f for d in ("training", "compressed_output") for f in os.listdir(os.path.join(out, d)))


@pytest.mark.parametrize("case", ["dropout_bn", "conv", "swae", "wide"])
def test_fp64_training_refusals_before_anything_is_written(tmp_path, monkeypatch, case):
    from baler_b200 import baler

    def no_device(*a, **k):
        raise AssertionError("the device was touched before the refusal")
    monkeypatch.setattr(helper, "process", no_device)
    table = synth.cms_table(64, seed=1)
    if case == "dropout_bn":
        out, cfg = _workspace(tmp_path, monkeypatch, table, model_name="AE_Dropout_BN")
        match = "AE_Dropout_BN"
    elif case == "conv":
        snaps = np.random.default_rng(1).random((4, 5, 5)).astype(np.float32)
        out, cfg = _workspace(tmp_path, monkeypatch, snaps, data_dimension=2, model_type="convolutional",
                              model_name="Conv_AE", compression_ratio=2.0)
        match = "Conv_AE"
    elif case == "swae":
        out, cfg = _workspace(tmp_path, monkeypatch, table, model_name="CFD_dense_AE",
                              custom_loss_function="loss_function_swae")
        match = "loss_function_swae"
    else:  # 2-D dense snapshots of 11 x 11 = 121 columns: wider than the fused trainer's 100
        snaps = np.random.default_rng(2).random((8, 11, 11)).astype(np.float32)
        out, cfg = _workspace(tmp_path, monkeypatch, snaps, data_dimension=2, model_type="dense",
                              model_name="CFD_dense_AE")
        match = "121"
    with pytest.raises(NotImplementedError, match=match):
        baler.perform_training(out, cfg, False)
    assert _written(out) == []


def test_fp64_device_adam_refuses_before_the_device():
    with pytest.raises(NotImplementedError, match="AE_Dropout_BN"):
        training.DeviceAdam(models.AE_Dropout_BN(24, 15), 1e-3, 64, precision="fp64")
    with pytest.raises(NotImplementedError, match="loss_function_swae"):
        training.DeviceAdam(models.AE(24, 15), 1e-3, 64, swae=True, precision="fp64")
    with pytest.raises(NotImplementedError, match="at most 100 columns"):
        training.DeviceAdam(models.CFD_dense_AE(400, 20), 1e-3, 64, precision="fp64")
    assert training.is_fp64("fp64") and not training.is_fp64(None) and not training.is_fp64("fp32")


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_fp64_training_has_no_cpu_fallback(tmp_path, monkeypatch, dtype):
    from baler_b200 import baler
    out, cfg = _workspace(tmp_path, monkeypatch, synth.cms_table(64, seed=2).astype(dtype))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        baler.perform_training(out, cfg, False)
    assert _written(out) == []
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        training.DeviceAdam(models.AE(24, 15), 1e-3, 64, precision="fp64")
