"""CPU-only checks of error_report = True: the numpy mirror against records worked out by hand (NaN and inf rows, x = 0,
constant and integer columns, the float64 un-normalisation), merges of split tables equal to one pass, a gloo world-size-2
merge in rank order, the config validation before any file is read, the C ABI's argument checks and the no-CPU-fallback
error."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import error_report_ref as ref
from baler_b200 import _lib, build, error_report
from baler_b200.modules import helper


def _same(a, b):
    for k in ("count", "nonfinite_x", "nonfinite_y", "response_count", "int_mismatch", "err_max_row", "hist"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    for k in ("x_min", "x_max", "err_max_abs"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    for k in ("sum_e", "sum_e2", "sum_r", "sum_r2"):
        np.testing.assert_allclose(getattr(a, k), getattr(b, k), rtol=1e-13, atol=1e-300, err_msg=k)


def test_hand_computed_record():
    nan, inf = np.nan, np.inf
    # columns: 0 ordinary, 1 with NaN / inf rows and x = 0, 2 constant, 3 integer
    x = np.array([[1.0, 0.0, 5.0, 3.0],
                  [2.0, nan, 5.0, 4.0],
                  [4.0, 2.0, 5.0, 7.0],
                  [-1.0, inf, 5.0, 1.0]])
    y = np.array([[1.5, 0.25, 5.0, 3.9],
                  [2.0, 1.0, 5.0, 4.2],
                  [3.0, nan, 5.0, -6.9],
                  [-1.5, 1.0, 5.0, 1.0]])
    rec = ref.record(x, y, row0=10, scale_range=np.array([2.0, 0.0, np.nan, 4.0]), int_mask=np.array([0, 0, 0, 1]))
    assert list(rec.count) == [4, 1, 4, 4]
    assert list(rec.nonfinite_x) == [0, 2, 0, 0] and list(rec.nonfinite_y) == [0, 1, 0, 0]
    assert list(rec.x_min) == [-1.0, 0.0, 5.0, 1.0] and list(rec.x_max) == [4.0, 2.0, 5.0, 7.0]
    # column 0: e = 0.5, 0, -1, -0.5
    assert rec.sum_e[0] == -1.0 and rec.sum_e2[0] == 1.5 and rec.err_max_abs[0] == 1.0 and rec.err_max_row[0] == 12
    assert rec.response_count[0] == 4 and rec.sum_r[0] == 50.0 + 0.0 - 25.0 + 50.0
    # |e| / 2 = 0.25, 0, 0.5, 0.25 -> bins (0.1, 1] three times, [0, 1e-9] once
    assert list(rec.hist[0]) == [1, 0, 0, 0, 0, 0, 0, 0, 0, 3, 0]
    # column 1: only row 0 is finite on both sides; x = 0 there, so no response; range 0 -> 1
    assert rec.sum_e[1] == 0.25 and rec.err_max_row[1] == 10 and rec.response_count[1] == 0
    assert list(rec.hist[1]) == [0] * 9 + [1, 0]
    # column 2: constant, exact everywhere: the first row attains the maximum 0; range NaN -> 1
    assert rec.sum_e2[2] == 0 and rec.err_max_abs[2] == 0 and rec.err_max_row[2] == 10 and rec.hist[2][0] == 4
    # column 3: trunc(y) = 3, 4, -6, 1: e = 0, 0, -13, 0; one mismatch; |e| / 4 = 3.25 -> the last bin
    assert rec.int_mismatch[3] == 1 and rec.sum_e[3] == -13.0 and rec.err_max_row[3] == 12
    assert list(rec.hist[3]) == [3] + [0] * 9 + [1]
    assert rec.int_mismatch[:3].sum() == 0
    rep = error_report.finalize(rec, np.array(list("abcd")), error_report.scale_range(np.array([[0] * 4, [2, 0, np.nan, 4]]), 4),
                                4, "float64", "auto")
    assert rep["err_mean"][0] == -0.25 and rep["err_rms"][0] == np.sqrt(1.5 / 4)
    assert rep["response_mean"][0] == 18.75 and np.isnan(rep["response_mean"][1])
    assert list(rep["scale_range"]) == [2.0, 1.0, 1.0, 4.0]
    text = error_report.summary(rep)
    assert "worst columns" in text and text.index("    d ") < text.index("    a ")


def test_nothing_finite_and_post_operations():
    x = np.array([[np.nan, 1.0], [np.inf, 2.0]])
    y = np.array([[0.5, 0.5], [0.5, 0.75]])
    rec = ref.record(x, y, post=(np.array([0.0, 1e9]), np.array([1.0, 4.0])))
    assert list(rec.count) == [0, 2] and rec.err_max_row[0] == -1 and rec.err_max_abs[0] == 0
    assert rec.x_min[0] == np.inf and rec.x_max[0] == -np.inf
    # y * 4 + 1e9 in two roundings, then - x
    assert rec.sum_e[1] == ((0.5 * 4 + 1e9) - 1.0) + ((0.75 * 4 + 1e9) - 2.0)
    rep = error_report.finalize(rec, np.array(["p", "q"]), np.ones(2), 2, "q4", "fp32")
    assert np.isnan(rep["x_min"][0]) and np.isnan(rep["err_rms"][0]) and np.isnan(rep["err_max_abs"][0])
    assert rep["err_max_row"][0] == -1


def test_histogram_edges_are_inclusive_above():
    x = np.zeros((11, 1))
    y = np.array([0.0, 1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1, 1.0])[:, None]
    assert list(ref.record(x, y).hist[0]) == [2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0]
    assert list(ref.record(x, y * 1.5).hist[0]) == [1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1]


def _table(n=1000, c=7, seed=0):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, c)) * rng.uniform(0.1, 100, c)
    y = x + rng.standard_normal((n, c)) * rng.uniform(1e-8, 1e-1, c)
    x[3, 2], y[5, 4], x[7, 1] = np.nan, np.inf, 0.0
    x[::97, 0], y[::97, 0] = 1.0, 6.0  # equal maxima in several rows: the smallest row must win
    x[:, 6] = 2.5
    return x, y


@pytest.mark.parametrize("cuts", [[500], [1, 999], [128, 256, 700], list(range(50, 1000, 50))])
def test_merge_of_split_tables_equals_one_pass(cuts):
    x, y = _table()
    mask = np.array([0, 0, 1, 0, 0, 0, 1])
    whole = ref.record(x, y, scale_range=np.arange(1, 8.0), int_mask=mask)
    bounds = [0] + cuts + [len(x)]
    parts = [ref.record(x[a:b], y[a:b], row0=a, scale_range=np.arange(1, 8.0), int_mask=mask)
             for a, b in zip(bounds[:-1], bounds[1:])]
    merged = error_report.merge(parts)
    _same(merged, whole)
    assert merged.err_max_row[0] == 0
    assert error_report.merge([merged, error_report.Record.empty(7)]) == merged


def test_words_round_trip():
    x, y = _table(200)
    rec = ref.record(x, y)
    ni = 6
    words = np.zeros((error_report.N_FIELDS, 7), np.int64)
    for i, k in enumerate(("count", "nonfinite_x", "nonfinite_y", "response_count", "int_mismatch", "err_max_row")):
        words[i] = getattr(rec, k)
    words[ni:ni + 11] = rec.hist.T
    for i, k in enumerate(("x_min", "x_max", "sum_e", "sum_e2", "err_max_abs", "sum_r", "sum_r2")):
        words[ni + 11 + i] = getattr(rec, k).view(np.int64)
    assert error_report.Record.from_words(words.reshape(-1), 7) == rec
    assert error_report.N_FIELDS == _lib.BB_ERROR_STATS_FIELDS == 24


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_main(rank, world, port, path):
    import torch.distributed as dist
    from baler_b200 import sharded
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    try:
        x, y = _table(1001, seed=3)
        lo, hi = sharded.row_range(len(x), rank, world)
        mine = error_report.merge([ref.record(x[a:min(a + 100, hi)], y[a:min(a + 100, hi)], row0=a)
                                   for a in range(lo, hi, 100)])
        parts = sharded.gather_objects_to_rank0(mine)
        if rank == 0:
            np.savez(path, **{k: getattr(error_report.merge(parts), k) for k in ("count", "hist", "sum_e", "err_max_row")})
    finally:
        dist.destroy_process_group()


def test_gloo_two_rank_merge_equals_one_pass(tmp_path):
    import torch.multiprocessing as mp
    path = str(tmp_path / "merged.npz")
    mp.spawn(_rank_main, args=(2, _free_port(), path), nprocs=2, join=True)
    x, y = _table(1001, seed=3)
    whole = ref.record(x, y)
    got = np.load(path)
    assert np.array_equal(got["count"], whole.count) and np.array_equal(got["hist"], whole.hist)
    assert np.array_equal(got["err_max_row"], whole.err_max_row)
    np.testing.assert_allclose(got["sum_e"], whole.sum_e, rtol=1e-13, atol=1e-300)


@pytest.mark.parametrize("value", ["yes", 1, 0, None, 1.0, [True]])
def test_non_bool_error_report_is_refused_before_any_file(tmp_path, value):
    from baler_b200 import baler
    cfg = SimpleNamespace(error_report=value, precision="auto", latent_dtype=None, apply_normalization=True,
                          input_path=str(tmp_path / "missing.npz"), save_error_bounded_deltas=False)
    with pytest.raises(ValueError, match="error_report must be True or False"):
        helper.compress(str(tmp_path / "missing.pt"), cfg)
    with pytest.raises(ValueError, match="error_report must be True or False"):
        baler.perform_compression(str(tmp_path / "output"), cfg, False)
    assert os.listdir(tmp_path) == []
    assert error_report.enabled(SimpleNamespace()) is False
    assert error_report.enabled(SimpleNamespace(error_report=np.bool_(True))) is True


def test_normalised_report_needs_the_training_features(tmp_path):
    cfg = SimpleNamespace(error_report=True, precision="auto", apply_normalization=True,
                          input_path=str(tmp_path / "missing.npz"))
    with pytest.raises(ValueError, match="training features"):
        helper.compress(str(tmp_path / "missing.pt"), cfg)
    assert os.listdir(tmp_path) == []


def test_integer_columns_mask():
    cfg = SimpleNamespace(type_list=["float64", "int", "float32", "int64", "uint8"])
    assert list(error_report.int_columns(cfg, (5,))) == [0, 1, 0, 1, 1]
    assert error_report.int_columns(SimpleNamespace(type_list=["float64"] * 3), (3,)) is None
    assert error_report.int_columns(SimpleNamespace(), (3,)) is None
    # 2-D dense rows: type_list indexes the snapshot's first axis, as decompressed[:, index] does
    assert list(error_report.int_columns(SimpleNamespace(type_list=["float", "int"]), (2, 3))) == [0, 0, 0, 1, 1, 1]


def test_c_abi_argument_checks():
    build.build()
    lib = _lib.lib()
    p = 4096  # (any non-NULL value: every refusal happens before a pointer is used)
    ok = dict(ctx=p, x=p, xt=_lib.BB_F32, y=p, yt=_lib.BB_F32, n=10, c=3, row0=0, pmin=None, prng=None, scale=None,
              mask=None, rec=p)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.bb_error_stats(a["ctx"], a["x"], a["xt"], a["y"], a["yt"], a["n"], a["c"], a["row0"], a["pmin"],
                                  a["prng"], a["scale"], a["mask"], a["rec"], None)
    for bad in (dict(ctx=None), dict(x=None), dict(y=None), dict(rec=None), dict(rec=p + 4), dict(n=-1), dict(c=0),
                dict(row0=-1), dict(xt=_lib.BB_F16), dict(yt=_lib.BB_F16), dict(xt=7), dict(pmin=p), dict(prng=p),
                dict(x=p + 4, xt=_lib.BB_F64), dict(y=p + 2), dict(scale=p + 4), dict(pmin=p + 4, prng=p)):
        assert call(**bad) == -1, bad  # BB_ERR_INVALID


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from baler_b200 import engine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        engine.error_stats(torch.zeros((4, 3)), torch.zeros((4, 3)))
