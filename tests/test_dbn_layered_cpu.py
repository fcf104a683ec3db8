"""AE_Dropout_BN on the layer-by-layer trainer without a device: the new entry points are declared, bound and exported;
the numpy restatement of the Philox keep-bits matches curand_Philox4x32_10; the fused step's batch limit is 16 rows x SMs;
under torchrun a per-rank share beyond it is refused before anything is read or written."""
import os
import subprocess

import pytest
import torch

from dbn_philox import philox_masks
from baler_b200 import _lib, build, synth
from baler_b200.modules import helper, models, training
from test_fp64_train_cpu import _workspace, _written

SYMBOLS = ("bb_ltrainer_create_dbn", "bb_ltrainer_set_dropout", "bb_ltrainer_bn_batches_tracked",
           "bb_ltrainer_activation_means")


def test_layered_dbn_symbols_declared_bound_and_exported():
    build.build()
    hdr = open(os.path.join(os.path.dirname(_lib.HERE), "include", "baler_b200.h")).read()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in SYMBOLS:
        assert name + "(" in hdr and name in _lib.exported_symbols() and (" T " + name) in out, name


# FNV-1a hash and count of the keep-bits of 37 rows, from bb_philox_keep compiled for the host with curand's own
# curand_Philox4x32_10: (seed, step, layer) -> (hash, kept)
PHILOX_PINS = {(4321, 0, 0): (10094349353173728462, 3717), (4321, 0, 3): (5633031345690349143, 442),
               (4321, 2, 1): (12289546290885616643, 2176), (0x123456789ABCDEF, 1, 2): (14142533150917886839, 1296),
               (0x123456789ABCDEF, 2, 3): (10457897181053330483, 446)}


@pytest.mark.parametrize("case", sorted(PHILOX_PINS))
def test_numpy_philox_restates_curand(case):
    seed, step, layer = case
    m = philox_masks(seed, step, 37)[layer]
    h = 1469598103934665603
    for k in m.ravel():
        h = ((h ^ int(k)) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    assert (h, int(m.sum())) == PHILOX_PINS[case]


def test_fused_dbn_limit_is_16_rows_per_sm(monkeypatch):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    assert training.dbn_fused_max_batch() == 16 * 148 == 2368
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)

    class Props:
        multi_processor_count = 132
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda d: Props)
    assert training.dbn_fused_max_batch() == 16 * 132
    assert training.fp64_dbn_max_batch() == 4 * 132


@pytest.mark.parametrize("batch,world,refused", [(4738, 2, True), (4736, 2, False), (9000, 1, False), (2369, 1, False)])
def test_rank_share_refusal(monkeypatch, batch, world, refused):
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    if refused:
        with pytest.raises(NotImplementedError, match="per-rank shares of at most 2368"):
            training.refuse_dbn_rank_share("AE_Dropout_BN", batch, world)
    else:
        training.refuse_dbn_rank_share("AE_Dropout_BN", batch, world)
    training.refuse_dbn_rank_share("AE", batch, world)  # other models: untouched


def test_rank_share_refused_before_anything_is_written(tmp_path, monkeypatch):
    from baler_b200 import baler

    def no_device(*a, **k):
        raise AssertionError("the device was touched before the refusal")
    monkeypatch.setattr(helper, "process", no_device)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    monkeypatch.setenv("WORLD_SIZE", "2")
    out, cfg = _workspace(tmp_path, monkeypatch, synth.cms_table(64, seed=1), model_name="AE_Dropout_BN", l1=False,
                          precision="auto", batch_size=5000)
    with pytest.raises(NotImplementedError, match="2368"):
        baler.perform_training(out, cfg, False)
    assert _written(out) == []
    with pytest.raises(NotImplementedError, match="2368"):
        training.DeviceAdam(models.AE_Dropout_BN(24, 15), 1e-3, 5000)
