"""CPU-only checks of training on tables streamed from host memory: the C entry points are declared, bound and exported,
the placement decision (resident vs streamed, window size) under a given device budget, the checks on host tables, and
the no-CPU-fallback error."""
import ctypes
import os
import re
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from baler_b200 import _lib, build, engine
from baler_b200.modules import data_processing, training

SYMBOLS = ("bb_trainer_epoch_host", "bb_trainer_validate_host", "bb_ltrainer_epoch_host", "bb_ltrainer_validate_host")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_stream_symbols_declared_bound_and_exported():
    build.build()
    hdr = open(os.path.join(ROOT, "include", "baler_b200.h")).read()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in SYMBOLS:
        assert name + "(" in hdr and name in _lib.exported_symbols() and (" T " + name) in out, name


def test_null_trainer_is_an_invalid_argument():
    lib = _lib.lib()
    x = np.zeros((8, 24), dtype=np.float32)
    out, hyper = ctypes.c_double(), engine.make_hyper()
    for name in ("bb_trainer_epoch_host", "bb_ltrainer_epoch_host"):
        assert getattr(lib, name)(None, x.ctypes.data, _lib.BB_F32, 8, 4, ctypes.byref(hyper), 4, ctypes.byref(out), None) == -1
    for name in ("bb_trainer_validate_host", "bb_ltrainer_validate_host"):
        assert getattr(lib, name)(None, x.ctypes.data, _lib.BB_F32, 8, 4, 4, ctypes.byref(out), None) == -1


def _cfg(**kw):
    base = dict(precision=None, data_dimension=1, model_type="dense", model_name="AE")
    base.update(kw)
    return SimpleNamespace(**base)


@pytest.fixture
def no_upload(monkeypatch):
    """the resident branch without a device: _to_device_table returns a marker"""
    monkeypatch.setattr(training, "_to_device_table", lambda data, config: "resident")


@pytest.mark.parametrize("n_rows,batch", [(10_000, 512), (10_037, 512), (9001, 4096), (601, 200)])
def test_placement_under_a_budget(no_upload, n_rows, batch):
    table = np.ones((n_rows, 24), dtype=np.float32)
    row = 24 * 4
    table_ds, win, used = training._place_table(table, _cfg(), batch, table.nbytes)
    assert table_ds == "resident" and win is None and used == table.nbytes
    budget = table.nbytes - 1
    table_ds, win, used = training._place_table(table, _cfg(), batch, budget)
    assert isinstance(table_ds, np.ndarray) and table_ds.flags.c_contiguous and table_ds.shape == (n_rows, 24)
    assert win % batch == 0 and win >= batch and 2 * win * row <= budget and used == 2 * win * row
    assert win + batch > min(budget // 2, training.STREAM_WINDOW_MAX_BYTES) // row  # the largest such multiple
    dl = training.DeviceBatches(table_ds, batch, win)
    assert len(dl) == (n_rows + batch - 1) // batch  # the ragged last batch counts
    # a second table streams through the same windows
    _, win2, _ = training._place_table(table, _cfg(), batch, 0, win)
    assert win2 == win


def test_placement_keeps_the_training_dtype_and_shape(no_upload):
    t64 = np.random.default_rng(0).random((1000, 24))
    arr, win, _ = training._place_table(t64, _cfg(precision="fp64"), 100, 100_000)
    assert arr.dtype == np.float64 and win == 200
    arr, _, _ = training._place_table(t64, _cfg(), 100, 50_000)
    assert arr.dtype == np.float32 and np.array_equal(arr, t64.astype(np.float32))
    snaps = np.zeros((50, 5, 5), dtype=np.float32)
    arr, win, _ = training._place_table(snaps, _cfg(data_dimension=2, model_type="convolutional", model_name="Conv_AE"), 10, 2000)
    assert arr.shape == (50, 25) and win == 10


def test_window_sizes():
    assert training.stream_window_rows(96, 512, 1 << 40) * 96 <= training.STREAM_WINDOW_MAX_BYTES
    assert training.stream_window_rows(96, 512, 2 * 96 * 1024) == 1024
    assert training.stream_window_rows(96, 512, 2 * 96 * 1023) == 512
    with pytest.raises(MemoryError):
        training.stream_window_rows(96, 512, 2 * 96 * 511)


def test_host_table_checks():
    x = np.zeros((100, 24), dtype=np.float32)
    assert engine._host_table(x, 50, 10)[1] == _lib.BB_F32
    assert engine._host_table(x.astype(np.float64), 10, 10)[1] == _lib.BB_F64
    for bad_window in (None, 0, 5, 15):
        with pytest.raises(ValueError):
            engine._host_table(x, bad_window, 10)
    for bad_table in (x[:, ::2], x.astype(np.float16), x.reshape(100, 2, 12), np.asfortranarray(x)):
        with pytest.raises(ValueError):
            engine._host_table(bad_table, 10, 10)


def test_row_chunks_cover_the_table(monkeypatch):
    monkeypatch.setattr(data_processing, "PREPROCESS_CHUNK_BYTES", 1000)
    flat = np.arange(37 * 24, dtype=np.float32).reshape(37, 24)
    chunks = data_processing._row_chunks(flat)
    assert [r0 for r0, _ in chunks] == list(range(0, 37, 10)) and all(c.flags.c_contiguous for _, c in chunks)
    assert np.array_equal(np.concatenate([c for _, c in chunks]), flat)
    assert len(data_processing._row_chunks(flat[:0])) == 1


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        engine.Trainer([np.zeros((2, 2))] * 8, [np.zeros(2)] * 8, 2, 2, 4)
    with pytest.raises(RuntimeError):
        training.device_table_budget()


def test_sources_name_no_batched_memcpy():
    """the library copies with cudaMemcpyAsync; the batched-copy family is not used anywhere in the sources"""
    family = re.compile("Memcpy(3D)?" + "Batch")
    for d in ("baler_b200", "include", "tools", "tests", "oracle"):
        for root, _, files in os.walk(os.path.join(ROOT, d)):
            for f in files:
                if f.endswith((".cu", ".cuh", ".h", ".py", ".sh", ".c", ".cpp")):
                    assert not family.search(open(os.path.join(root, f), errors="ignore").read()), f
