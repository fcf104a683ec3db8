"""error_report = True on the device: bb_error_stats against the numpy mirror (tests/error_report_ref.py) for every dtype
pair, widths 1 to 2500, with the float64 un-normalisation, integer columns and the histogram range; bit-identical re-runs;
chunkings that agree; no spills.  Through the CLI: the report compress writes equals the mirror's record of the input and
the decompressed.npz decompress then writes, for the CMS model with float64 / float16 / q4 / q8 latents, fp32, fp64 on a
float64 table, integer type_list columns, Conv_AE on 5x5 blocks and CFD_dense_AE on 50x50 snapshots; the compressed files
(and the delta files) are the same with the report on and off; the 2-rank run gives the one-process report.
The test tables stay inside the split16 kernels' fp16 range: a chunk that trips that guard is re-run on the fp32 kernel, which
the C pipeline may decide on another row range, so its latent bits could differ with the report on."""
import gzip
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import error_report_ref as ref
from conftest import ROOT, randomise_bn2d, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import build, engine, error_report, synth
from test_gpu_latent_q8 import TYPE_LIST, _free_port, _workspace

pytestmark = pytest.mark.gpu


def _check_record(got, want, x, y):
    for k in ("count", "nonfinite_x", "nonfinite_y", "response_count", "int_mismatch", "err_max_row", "hist"):
        assert np.array_equal(getattr(got, k), getattr(want, k)), (k, getattr(got, k), getattr(want, k))
    for k in ("x_min", "x_max", "err_max_abs"):
        assert np.array_equal(getattr(got, k), getattr(want, k)), k
    # sums within 1e-12 of sum |e| and sum e^2 (the summation orders differ)
    e = np.asarray(y, np.float64) - np.asarray(x, np.float64)
    e[~np.isfinite(e)] = 0.0
    assert (np.abs(got.sum_e - want.sum_e) <= 1e-12 * np.abs(e).sum(axis=0) + 1e-300).all()
    assert (np.abs(got.sum_e2 - want.sum_e2) <= 1e-12 * (e * e).sum(axis=0) + 1e-300).all()
    # the response r = 100 e / x over x != 0: sum r within 1e-12 of sum |r|
    xx = np.asarray(x, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where((xx != 0) & np.isfinite(xx), 100.0 * e / xx, 0.0)
    r[~np.isfinite(r)] = 0.0
    assert (np.abs(got.sum_r - want.sum_r) <= 1e-12 * np.abs(r).sum(axis=0) + 1e-300).all()
    np.testing.assert_allclose(got.sum_r2, want.sum_r2, rtol=1e-11, atol=0)


def _awkward(n, c, dtype, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((n, c)) * rng.uniform(0.1, 50, c)).astype(dtype)
    y = (x + rng.standard_normal((n, c)) * rng.uniform(1e-7, 1e-1, c)).astype(dtype)
    if n > 10:
        x[n // 2, 0], y[n // 3, c - 1], x[1, c // 2] = np.nan, np.inf, 0.0
        x[:, c // 3], y[:, c // 3] = 3.0, 3.0  # a constant, exact column
        x[::7, 0], y[::7, 0] = 1.0, 9.0  # equal maxima: the smallest row wins
    return x, y


@pytest.mark.parametrize("xt,yt", [(np.float32, np.float32), (np.float32, np.float64), (np.float64, np.float32),
                                   (np.float64, np.float64)])
@pytest.mark.parametrize("n,c", [(1, 1), (1000, 1), (4099, 24), (777, 255), (777, 256), (301, 257), (3000, 1000),
                                 (257, 2500)])
def test_kernel_equals_mirror(xt, yt, n, c):
    x, y = _awkward(n, c, np.float64, n + c)
    x, y = x.astype(xt), y.astype(yt)
    rng = np.random.default_rng(c)
    scale = rng.uniform(0.5, 20, c)
    scale[0] = 0.0  # -> 1
    mask = (rng.random(c) < 0.3).astype(np.uint8)
    got = engine.error_stats(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), row0=17,
                             scale_range=torch.from_numpy(scale).cuda(), int_mask=torch.from_numpy(mask).cuda())
    want = ref.record(x, y, row0=17, scale_range=scale, int_mask=mask)
    yy = np.asarray(y, np.float64).copy()
    yy[:, mask.astype(bool)] = np.trunc(yy[:, mask.astype(bool)])
    _check_record(got, want, x, yy)


def test_kernel_post_operations_equal_mirror():
    """y * range + min in float64 (a table beyond F32_OFFSET_LIMIT): offsets of 1e9 with a spread of a few units"""
    n, c = 5000, 6
    rng = np.random.default_rng(5)
    mn, rg = 1e9 + rng.uniform(0, 100, c), rng.uniform(1, 5, c)
    x = mn + rng.random((n, c)) * rg
    y = ((x - mn) / rg + rng.standard_normal((n, c)) * 1e-4).astype(np.float32)
    got = engine.error_stats(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), post_min=torch.from_numpy(mn).cuda(),
                             post_range=torch.from_numpy(rg).cuda(), scale_range=torch.from_numpy(rg).cuda())
    want = ref.record(x, y, post=(mn, rg), scale_range=rg)
    _check_record(got, want, x, (y.astype(np.float64) * rg) + mn)


def test_reruns_are_bit_identical_and_chunkings_agree():
    x, y = _awkward(3_000_001, 24, np.float32, 1)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    a, b = engine.error_stats(xd, yd), engine.error_stats(xd, yd)
    for k in ("sum_e", "sum_e2", "sum_r", "sum_r2", "x_min", "x_max", "err_max_abs"):
        assert getattr(a, k).tobytes() == getattr(b, k).tobytes(), k
    assert a == b
    for chunk in (1 << 20, 100_003, 4096):
        parts = [engine.error_stats(xd[r:r + chunk].contiguous(), yd[r:r + chunk].contiguous(), row0=r)
                 for r in range(0, len(x), chunk)]
        m = error_report.merge(parts)
        for k in ("count", "nonfinite_x", "nonfinite_y", "response_count", "err_max_row", "hist", "x_min", "x_max", "err_max_abs"):
            assert np.array_equal(getattr(m, k), getattr(a, k)), (chunk, k)
        for k in ("sum_e", "sum_e2", "sum_r", "sum_r2"):
            np.testing.assert_allclose(getattr(m, k), getattr(a, k), rtol=1e-13, atol=0, err_msg=k)


def test_kernel_has_no_spills(tmp_path):
    src = os.path.join(build.CSRC, "bb_error_stats.cu")
    r = subprocess.run([build.NVCC] + build.FLAGS + ["-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "es.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    kernels = re.findall(r"Compiling entry function '(\w*error_stats\w*)'", r.stderr)
    assert len(kernels) == 5  # 4 dtype pairs + the fold
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert len(spills) >= 5 and all(s == ("0", "0") for s in spills), r.stderr


# ---------------------------------------------------------------- the CLI


def _report_vs_files(out, cfg, x, features, int_mask=None):
    """error_report.npz against the mirror's record of the input rows and decompressed.npz"""
    from baler_b200 import baler
    baler.perform_decompression(out, cfg, False)
    y = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    x, y = np.asarray(x).reshape(len(x), -1), y.reshape(len(x), -1)
    rep = np.load(os.path.join(out, "compressed_output", "error_report.npz"))
    got = error_report.Record(**{k: rep[k] for k in ("count", "nonfinite_x", "nonfinite_y", "response_count", "int_mismatch",
                                                     "err_max_row", "hist", "sum_e", "sum_e2")},
                              x_min=np.where(np.isnan(rep["x_min"]), np.inf, rep["x_min"]),
                              x_max=np.where(np.isnan(rep["x_max"]), -np.inf, rep["x_max"]),
                              err_max_abs=np.where(np.isnan(rep["err_max_abs"]), 0.0, rep["err_max_abs"]),
                              sum_r=np.where(rep["response_count"] > 0, rep["response_mean"] * rep["response_count"], 0.0),
                              sum_r2=np.where(rep["response_count"] > 0, rep["response_rms"] ** 2 * rep["response_count"], 0.0))
    want = ref.from_files(x, y, features=features, int_mask=int_mask)
    _check_record(got, want, x, y)
    assert int(rep["rows"]) == len(x) and np.array_equal(rep["hist_edges"], error_report.HIST_EDGES)
    assert np.array_equal(rep["scale_range"], error_report.scale_range(features, x.shape[1]))
    return rep, x, y


def _compressed_arrays(out):
    comp = np.load(os.path.join(out, "compressed_output", "compressed.npz"))
    arrays = {k: comp[k].copy() for k in comp.files}
    for name in ("compressed_deltas.npz.gz", "compressed_batch_index_metadata.npz.gz"):
        p = os.path.join(out, "compressed_output", name)
        if os.path.exists(p):
            arrays[name] = repr(np.load(gzip.GzipFile(p, "r"), allow_pickle=True).tolist())
    return arrays


def _same_files(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        if isinstance(a[k], str):
            assert a[k] == b[k], k
        else:
            assert a[k].dtype == b[k].dtype and a[k].tobytes() == b[k].tobytes(), k


CMS_CASES = {  # name: (latent_dtype, precision, float64 table, type_list)
    "float64": (None, "auto", False, None),
    "float16": ("float16", "auto", False, None),
    "q4": ("q4", "auto", False, None),
    "q8": ("q8", "auto", False, None),
    "fp32": ("float32", "fp32", False, None),
    "fp64_float64_table": (None, "fp64", True, None),
    "int_columns": (None, "auto", False, TYPE_LIST),
}


@pytest.mark.parametrize("case", sorted(CMS_CASES))
def test_cli_cms_report_equals_mirror_of_decompressed(golden, tmp_path, monkeypatch, capsys, case):
    from baler_b200 import baler
    latent, precision, f64, types = CMS_CASES[case]
    table = synth.cms_table(300_001, seed=21)  # (two pipeline chunks of bb_compress_host / bb_decompress_host)
    if f64:
        table = table.astype(np.float64) * 1.0000001
    feats = orc.find_minmax(synth.cms_table(50_000, seed=22).astype(table.dtype))  # training features of another sample
    extra = dict(latent_dtype=latent, precision=precision)
    if types is not None:
        extra["type_list"] = types
    out, cfg = _workspace(tmp_path, monkeypatch, sub_sd(golden("ae_cms.npz"), "sd"), table, feats, **extra)
    baler.perform_compression(out, cfg, False)
    plain = _compressed_arrays(out)
    cfg.error_report = True
    capsys.readouterr()
    baler.perform_compression(out, cfg, False)
    printed = capsys.readouterr().out
    assert "err_rms / range: mean" in printed and "worst columns" in printed
    _same_files(plain, _compressed_arrays(out))  # the report changes no byte of the latent
    mask = error_report.int_columns(cfg, (24,))
    rep, x, y = _report_vs_files(out, cfg, table, feats, mask)
    assert list(rep["names"]) == list(synth.CMS_NAMES)
    assert str(rep["precision"]) == precision and str(rep["latent_dtype"]) == (latent or "float64")
    if types is not None:
        it = np.array([t == "int" for t in TYPE_LIST])
        assert np.array_equal(rep["int_mismatch"] > 0, it & (rep["int_mismatch"] > 0)) and rep["int_mismatch"][it].sum() > 0


def test_cli_deltas_files_equal_with_report(golden, tmp_path, monkeypatch):
    from baler_b200 import baler
    g = golden("eb_deltas.npz")
    table, bound = g["table"], float(g["bound"])
    feats = orc.find_minmax(table)
    out, cfg = _workspace(tmp_path, monkeypatch, sub_sd(golden("ae_cms.npz"), "sd"), table, feats,
                          save_error_bounded_deltas=True, error_bounded_requirement=bound, batch_size=256, latent_dtype="q3")
    baler.perform_compression(out, cfg, False)
    plain = _compressed_arrays(out)
    assert "compressed_deltas.npz.gz" in plain
    cfg.error_report = True
    baler.perform_compression(out, cfg, False)
    _same_files(plain, _compressed_arrays(out))
    rep = np.load(os.path.join(out, "compressed_output", "error_report.npz"))
    assert "before error-bounded deltas" in str(rep["scope"]) and rep["count"].sum() > 0


def test_cli_conv_ae_blocks(golden, tmp_path, monkeypatch):
    from baler_b200 import baler
    from baler_b200.modules import helper, models
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CFD_workspace", "P")
    snaps = synth.cfd_snapshots(40)
    path = os.path.join("workspaces", "CFD_workspace", "data", "CFD_blocks.npz")
    np.savez(path, data=snaps, names=np.array(["snapshot"]))
    out = os.path.join("workspaces", "CFD_workspace", "P", "output")
    torch.manual_seed(0)
    m = models.Conv_AE(50, 250)
    m.load_state_dict(randomise_bn2d(m.state_dict()))
    torch.save(m.state_dict(), os.path.join(out, "compressed_output", "model.pt"))

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name, model_type = 2, 10, False, "Conv_AE", "convolutional"
        batch_size, custom_norm, extra_compression, separate_model_saving = 600, True, False, False
        save_error_bounded_deltas, convert_to_blocks, error_report = False, [1, 5, 5], True

    baler.perform_compression(out, cfg, False)
    rep, _, _ = _report_vs_files(out, cfg, snaps.reshape(-1, 25), None)
    assert len(rep["names"]) == 25 and rep["count"].sum() == snaps.size


def test_cli_cfd_dense_snapshots(tmp_path, monkeypatch):
    from baler_b200 import baler
    from baler_b200.modules import helper, models
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CFD_workspace", "D")
    snaps = synth.cfd_snapshots(3000)
    path = os.path.join("workspaces", "CFD_workspace", "data", "snaps.npz")
    np.savez(path, data=snaps, names=np.array(["snapshot"]))
    out = os.path.join("workspaces", "CFD_workspace", "D", "output")
    torch.manual_seed(0)
    torch.save(models.CFD_dense_AE(2500, 25).state_dict(), os.path.join(out, "compressed_output", "model.pt"))
    feats = orc.find_minmax(snaps)
    np.save(os.path.join(out, "training", "normalization_features.npy"), feats)

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name, model_type = 2, 100, True, "CFD_dense_AE", "dense"
        batch_size, custom_norm, extra_compression, separate_model_saving = 500, False, False, False
        save_error_bounded_deltas, convert_to_blocks, error_report = False, False, True

    baler.perform_compression(out, cfg, False)
    rep, _, _ = _report_vs_files(out, cfg, snaps, feats)
    assert len(rep["names"]) == 2500 and rep["count"].sum() == snaps.size


_CFG = """
def set_config(c):
    c.input_path = {path!r}
    c.data_dimension, c.compression_ratio, c.apply_normalization, c.model_name = 1, 1.6, True, "AE"
    c.batch_size, c.custom_norm, c.extra_compression, c.separate_model_saving = 512, False, False, False
    c.save_error_bounded_deltas, c.convert_to_blocks, c.latent_dtype, c.error_report = False, False, {latent!r}, True
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("latent", [None, "q4"])
def test_torchrun_two_ranks_report_equals_one_process(golden, tmp_path, latent):
    sd = sub_sd(golden("ae_cms.npz"), "sd")
    table = synth.cms_table(30011, seed=44)
    reports = {}
    for world in (1, 2):
        wd = tmp_path / ("w%d" % world)
        proj = wd / "workspaces" / "WS" / "P"
        for d in ("config", "output/compressed_output", "output/decompressed_output", "output/training"):
            os.makedirs(proj / d)
        os.makedirs(wd / "workspaces" / "WS" / "data")
        data = str(wd / "workspaces" / "WS" / "data" / "d.npz")
        np.savez(data, data=table, names=synth.CMS_NAMES)
        torch.save({k: torch.from_numpy(v) for k, v in sd.items()}, proj / "output" / "compressed_output" / "model.pt")
        np.save(proj / "output" / "training" / "normalization_features.npy", orc.find_minmax(table))
        (proj / "config" / "P_config.py").write_text(_CFG.format(path=data, latent=latent))
        launch = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port",
                  str(_free_port())] if world == 2 else [sys.executable]
        r = subprocess.run(launch + ["-m", "baler_b200", "--project", "WS", "P", "--mode", "compress"], cwd=wd,
                           env=dict(os.environ, PYTHONPATH=ROOT), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        reports[world] = dict(np.load(proj / "output" / "compressed_output" / "error_report.npz"))
    a, b = reports[1], reports[2]
    for k in ("count", "nonfinite_x", "nonfinite_y", "hist", "err_max_row", "err_max_abs", "int_mismatch", "x_min", "x_max"):
        assert np.array_equal(a[k], b[k], equal_nan=a[k].dtype.kind == "f"), k
    np.testing.assert_allclose(b["sum_e"], a["sum_e"], rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(b["sum_e2"], a["sum_e2"], rtol=1e-12, atol=0)
