"""precision "fp64" without a device: the float64 entry points are declared, bound and exported; shapes and options the
float64 chain does not take are refused before anything is read from a device or written; with no device it fails like
every other compute path (no CPU fallback)."""
import os

import numpy as np
import pytest
import torch

from conftest import sub_sd
from baler_b200 import _lib, build, engine, synth
from baler_b200.modules import helper, models

FP64_SYMBOLS = ("bb_colminmax_f64", "bb_encode_f64", "bb_decode_f64", "bb_compress_host_f64", "bb_decompress_host_f64")


def test_fp64_symbols_declared_bound_and_exported():
    import subprocess
    build.build()
    hdr = open(os.path.join(os.path.dirname(_lib.HERE), "include", "baler_b200.h")).read()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in FP64_SYMBOLS:
        assert name + "(" in hdr and name in _lib.exported_symbols() and (" T " + name) in out, name
    assert "#define BB_PREC_FP64 4" in hdr and _lib.PRECISIONS["fp64"] == _lib.BB_PREC_FP64 == 4


def test_fp64_refusal_names_the_shape():
    assert engine.fp64_refusal({"encoder": [24, 200, 100, 50, 15], "decoder": [15, 50, 100, 200, 24]}) is None
    assert engine.fp64_refusal({"encoder": [256, 200, 100, 50, 160]}) is None
    msg = engine.fp64_refusal({"encoder": [2500, 200, 100, 50, 1563]})
    assert "2500-200-100-50-1563" in msg and "256" in msg
    assert "4-4-4-4-4-4-4-4-4-4" in engine.fp64_refusal({"encoder": [4] * 10})  # 9 layers


def _workspace(tmp_path, monkeypatch, model, table, **extra):
    os.makedirs(tmp_path, exist_ok=True)
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CMS_workspace", "CMS_project_v1")
    path = os.path.join("workspaces", "CMS_workspace", "data", "example_CMS_data.npz")
    names = ["c%d" % i for i in range(table.shape[1])]
    np.savez(path, data=table, names=names)
    out = os.path.join("workspaces", "CMS_workspace", "CMS_project_v1", "output")
    torch.save(model.state_dict(), os.path.join(out, "compressed_output", "model.pt"))
    flat = table.reshape(len(table), -1)
    np.save(os.path.join(out, "training", "normalization_features.npy"), np.stack([flat.min(0), np.ptp(flat, 0)]))

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name = 1, 1.6, True, type(model).__name__
        batch_size, custom_norm, extra_compression, separate_model_saving = 512, False, False, False
        save_error_bounded_deltas, convert_to_blocks, precision = False, False, "fp64"
    for k, v in extra.items():
        setattr(cfg, k, v)
    return out, cfg


def test_fp64_refusals_before_anything_is_written(tmp_path, monkeypatch):
    from baler_b200 import baler
    table = synth.cms_table(64, seed=1)
    # error-bounded deltas
    out, cfg = _workspace(tmp_path / "a", monkeypatch, models.AE(24, 15), table, save_error_bounded_deltas=True,
                          error_bounded_requirement=1.0)
    with pytest.raises(NotImplementedError, match="save_error_bounded_deltas"):
        baler.perform_compression(out, cfg, False)
    assert "compressed.npz" not in os.listdir(os.path.join(out, "compressed_output"))
    # CFD_dense_AE on 2500-feature (50 x 50) snapshots: widths beyond the kernel's 256
    wide = np.random.default_rng(0).random((8, 2500)).astype(np.float32)
    out, cfg = _workspace(tmp_path / "b", monkeypatch, models.CFD_dense_AE(2500, 1563), wide, compression_ratio=1.6)
    with pytest.raises(NotImplementedError, match="2500-200-100-50-1563"):
        baler.perform_compression(out, cfg, False)
    assert "compressed.npz" not in os.listdir(os.path.join(out, "compressed_output"))
    # Conv_AE (5 x 5 blocks of a 2-D file)
    snaps = np.random.default_rng(1).random((4, 5, 5)).astype(np.float32)
    out, cfg = _workspace(tmp_path / "c", monkeypatch, models.Conv_AE(5, 13), snaps, data_dimension=2,
                          model_type="convolutional", compression_ratio=2.0)
    with pytest.raises(NotImplementedError, match="Conv_AE"):
        baler.perform_compression(out, cfg, False)
    assert "compressed.npz" not in os.listdir(os.path.join(out, "compressed_output"))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fp64_has_no_cpu_fallback(tmp_path, monkeypatch, golden):
    m = models.AE(24, 15)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sub_sd(golden("ae_cms.npz"), "sd").items()})
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.eval().codec()  # DenseCodec: the float64 chain, like every other, needs the device
    out, cfg = _workspace(tmp_path, monkeypatch, m, synth.cms_table(64, seed=2).astype(np.float64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        helper.compress(os.path.join(out, "compressed_output", "model.pt"), cfg)
