"""latent_dtype "q8" on the device: codes and parameters bit-equal to the numpy mirror (tests/latent_q8_ref.py) applied to the
device's own float32 latent, on every codec the host pipelines take; decompression bit-equal to decode of the mirror's
dequantised latent; the step / 2 bound; the CLI round trip; error-bounded deltas; the 2-rank file."""
import gzip
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

import latent_q8_ref as ref
from conftest import ROOT, randomise_bn2d, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import engine, latent_q8, synth
from baler_b200.modules import models

pytestmark = pytest.mark.gpu
TYPE_LIST = ["float64"] * 12 + ["int"] * 7 + ["float64"] * 3 + ["int"] * 2


def _ae(golden):
    m = models.AE(24, 15)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sub_sd(golden("ae_cms.npz"), "sd").items()})
    return m.eval().codec(), lambda n, seed: synth.cms_table(n, seed=seed)


def _chain_tc(golden):
    rng = np.random.default_rng(1)
    dims = [24, 64, 48, 32, 12]

    def layers(ds):
        return [(rng.standard_normal((o, i)) / np.sqrt(i), 0.1 * rng.standard_normal(o), "leaky" if k < len(ds) - 2 else "none")
                for k, (i, o) in enumerate(zip(ds[:-1], ds[1:]))]
    return engine.DenseCodec(layers(dims), layers(dims[::-1])), lambda n, seed: synth.cms_table(n, seed=seed)


def _conv(golden):
    torch.manual_seed(0)
    m = models.Conv_AE(5, 250)
    m.load_state_dict(randomise_bn2d(m.state_dict()))
    blocks = golden("conv_ae.npz")["blocks"].reshape(600, 25)
    return m.eval().codec(5, 5), lambda n, seed: np.ascontiguousarray(blocks[np.random.default_rng(seed).integers(0, 600, n)])


def _cfd(golden):
    torch.manual_seed(0)
    m = models.CFD_dense_AE(2500, 25).eval()
    return m.codec(), lambda n, seed: np.random.default_rng(seed).standard_normal((n, 2500)).astype(np.float32)


CODECS = {  # name: (builder, precision)
    "ae_chain_tc4": (_ae, "auto"),
    "chain_tc_4_layers": (_chain_tc, "auto"),
    "ae_fp32": (_ae, "fp32"),
    "ae_fast": (_ae, "fast"),
    "conv_ae_layered": (_conv, "auto"),
    "cfd_dense_2500_layered": (_cfd, "auto"),
}


def _pinned(shape, dtype):
    return torch.empty(shape, dtype=dtype, pin_memory=True).numpy()


def _check(codec, x, precision, pinned=False):
    mn, mx = np.nanmin(x, axis=0), np.nanmax(x, axis=0)  # (a NaN row normalises to NaN, the others as usual)
    feats = np.stack([mn, mx - mn]).astype(np.float32)
    n = len(x)
    if pinned:
        xp = _pinned(x.shape, torch.float32)
        xp[:] = x
        x = xp
        out = latent_q8.Q8Latent(_pinned((n, codec.z_dim), torch.uint8), _pinned((latent_q8.n_blocks(n), codec.z_dim), torch.float32),
                                 _pinned((latent_q8.n_blocks(n), codec.z_dim), torch.float32))
    else:
        out = None
    q, _ = codec.compress_host_q8(x, features=feats, precision=precision, out=out)
    z, _ = codec.compress_host(x, features=feats, z_dtype=np.float32, precision=precision)  # the device's own latent
    want = ref.quantize(z)
    for got, w, name in zip(q, want, ("codes", "lo", "step")):
        assert got.dtype == w.dtype and got.shape == w.shape, name
        assert np.array_equal(got.view(np.uint8), w.view(np.uint8)), (name, int((got.view(np.uint8) != w.view(np.uint8)).sum()))
    # the device-level entry points give the same bits
    zd = torch.from_numpy(z).cuda()
    qd = codec.quantize_q8(zd)
    assert all(np.array_equal(a.cpu().numpy().view(np.uint8), b.view(np.uint8)) for a, b in zip(qd, want))
    back = ref.dequantize(*want)
    assert np.array_equal(codec.dequantize_q8(qd).cpu().numpy().view(np.uint32), back.view(np.uint32))
    # latent error within step / 2 element by element
    fin = np.isfinite(z)
    err = np.abs(back.astype(np.float64) - z.astype(np.float64))
    assert (err[fin] <= ref.error_bound(z, want[2])[fin]).all()
    # decompression = decode of the mirror's dequantised latent on the same precision, fused un-normalisation included
    y = codec.decompress_host_q8(q, features=feats, y_dtype=np.float32, precision=precision)
    y_ref = codec.decompress_host(back, features=feats, y_dtype=np.float32, precision=precision)
    assert np.array_equal(y.view(np.uint32), y_ref.view(np.uint32))
    return q, z


@pytest.mark.parametrize("name", sorted(CODECS))
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
def test_codes_bit_equal_to_mirror(golden, name, n):
    build, precision = CODECS[name]
    codec, make = build(golden)
    _check(codec, make(n, seed=n), precision)


@pytest.mark.parametrize("pinned", [False, True])
def test_several_pipeline_chunks(golden, pinned):
    """5,000,001 rows: 16 pipeline chunks of whole blocks and a ragged last block, pinned and pageable buffers"""
    codec, make = _ae(golden)
    x = make(5_000_001, seed=3)
    x[123_457, 4] = np.nan  # a NaN row stays NaN
    q, z = _check(codec, x, "auto", pinned)
    assert (q.codes[123_457] == 255).any()


def test_tc4_range_fallback_keeps_the_format(golden):
    """the split16 range guard re-runs the rows on the fp32 kernel; the q8 result is then the fp32 one"""
    codec, make = _ae(golden)
    x = make(1000, seed=9)
    x[10, 3] = 1e30
    feats = orc.find_minmax(make(1000, seed=9)).astype(np.float32)
    q, _ = codec.compress_host_q8(x, features=feats)
    q32, _ = codec.compress_host_q8(x, features=feats, precision="fp32")
    assert all(np.array_equal(a.view(np.uint8), b.view(np.uint8)) for a, b in zip(q, q32))


def test_fp64_is_refused(golden):
    codec, make = _ae(golden)
    with pytest.raises(NotImplementedError, match="q8"):
        codec.compress_host_q8(make(10, seed=1), precision="fp64")
    from baler_b200 import _lib
    x = make(10, seed=1)
    q = latent_q8.empty(10, 15)
    assert _lib.lib().bb_compress_host_q8(codec.handle, x.ctypes.data, 10, None, 0, q.codes.ctypes.data, q.lo.ctypes.data,
                                          q.step.ctypes.data, _lib.BB_PREC_FP64) == -2  # BB_ERR_UNSUPPORTED


# ---------------------------------------------------------------- the CLI


def _workspace(tmp_path, monkeypatch, sd, table, feats, **extra):
    from baler_b200.modules import helper
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CMS_workspace", "CMS_project_v1")
    path = os.path.join("workspaces", "CMS_workspace", "data", "example_CMS_data.npz")
    np.savez(path, data=table, names=synth.CMS_NAMES)
    out = os.path.join("workspaces", "CMS_workspace", "CMS_project_v1", "output")
    torch.save({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}, os.path.join(out, "compressed_output", "model.pt"))
    np.save(os.path.join(out, "training", "normalization_features.npy"), feats)

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name = 1, 1.6, True, "AE"
        batch_size, custom_norm, extra_compression, separate_model_saving = 512, False, False, False
        save_error_bounded_deltas, convert_to_blocks, precision, latent_dtype = False, False, "auto", "q8"
    for k, v in extra.items():
        setattr(cfg, k, v)
    return out, cfg


def test_cli_train_compress_decompress_info(tmp_path, monkeypatch, capsys):
    from baler_b200 import baler
    from baler_b200.modules import helper
    from test_gpu_train_fp64 import _cfg, _project
    table = synth.cms_table(20_000, seed=31)
    out, path = _project(tmp_path, monkeypatch, table)
    cfg = _cfg(helper, path, precision="auto", latent_dtype="q8", type_list=TYPE_LIST, l1=False, activation_extraction=False)
    torch.manual_seed(0)
    baler.perform_training(out, cfg, False)
    baler.perform_compression(out, cfg, False)
    comp = np.load(os.path.join(out, "compressed_output", "compressed.npz"))
    assert sorted(comp.files) == sorted(["data", "latent_min", "latent_step", "latent_block_rows", "names",
                                         "normalization_features"])
    assert comp["data"].dtype == np.uint8 and comp["data"].shape == (20_000, 15)
    assert comp["latent_min"].dtype == comp["latent_step"].dtype == np.float32
    assert comp["latent_min"].shape == comp["latent_step"].shape == (157, 15) and int(comp["latent_block_rows"]) == 128
    q8_bytes = os.stat(os.path.join(out, "compressed_output", "compressed.npz")).st_size
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    assert dec.shape == table.shape and np.isfinite(dec).all()
    it = [c for c, t in enumerate(TYPE_LIST) if t == "int"]
    assert np.array_equal(dec[:, it], np.trunc(dec[:, it]))
    # the same decode outside the CLI, then the reference's truncation: identical
    from baler_b200.modules import data_processing
    m = data_processing.load_model(models.AE, os.path.join(out, "compressed_output", "model.pt"), n_features=24, z_dim=15)
    y = m.eval().codec().decompress_host_q8(latent_q8.from_npz(comp), features=np.load(
        os.path.join(out, "training", "normalization_features.npy")).reshape(2, -1), y_dtype=dec.dtype)
    y[:, it] = np.trunc(y[:, it])
    assert np.array_equal(y, dec)
    capsys.readouterr()
    baler.print_info(out, cfg)
    info = capsys.readouterr().out
    assert "Compressed file size: %s MB" % round(q8_bytes / (1024 * 1024), 4) in info
    cfg.latent_dtype = "float64"  # the same model's float64 latent, for the size comparison
    baler.perform_compression(out, cfg, False)
    f64_bytes = os.stat(os.path.join(out, "compressed_output", "compressed.npz")).st_size
    assert q8_bytes < f64_bytes / 7  # 15.9 against 120 bytes per row


def test_error_bounded_deltas_correct_the_quantised_reconstruction(golden, tmp_path, monkeypatch):
    """save_error_bounded_deltas with q8: the deltas are taken against decode(dequantise(quantise(encode(x)))), so every
    stored hit, applied by decompress, lands within float16 rounding of the input"""
    from baler_b200 import baler
    g = golden("eb_deltas.npz")
    table, bound, bs = g["table"], float(g["bound"]), 256
    feats = orc.find_minmax(table)
    out, cfg = _workspace(tmp_path, monkeypatch, sub_sd(golden("ae_cms.npz"), "sd"), table, feats,
                          save_error_bounded_deltas=True, error_bounded_requirement=bound, batch_size=bs)
    baler.perform_compression(out, cfg, False)
    comp = np.load(os.path.join(out, "compressed_output", "compressed.npz"))
    assert comp["data"].dtype == np.uint8
    index = np.load(gzip.GzipFile(os.path.join(out, "compressed_output", "compressed_batch_index_metadata.npz.gz"), "r"),
                    allow_pickle=True)
    hits = [(int(r) + bs * int(b), int(c)) for b, (rows, cols) in zip(index[0], index[1]) for r, c in zip(rows, cols)]
    assert hits
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    r, c = np.array(hits).T
    x_n = (table[r, c].astype(np.float64) - feats[0][c]) / feats[1][c]
    y_n = (dec[r, c].astype(np.float64) - feats[0][c]) / feats[1][c]
    # float16(y) - float16(x) removed from y: what remains is the float16 rounding of x and of y (|y| <= ~1.5 here)
    assert (np.abs(y_n - x_n) <= 2.0 ** -11 * (np.abs(x_n) + 2.0) + 1e-6).all(), float(np.abs(y_n - x_n).max())


_CFG = """
def set_config(c):
    c.input_path = {path!r}
    c.data_dimension, c.compression_ratio, c.apply_normalization, c.model_name = 1, 1.6, True, "AE"
    c.batch_size, c.custom_norm, c.extra_compression, c.separate_model_saving = 512, False, False, False
    c.save_error_bounded_deltas, c.convert_to_blocks, c.latent_dtype = False, False, "q8"
"""


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_torchrun_two_ranks_write_the_file_of_one_process(golden, tmp_path):
    sd = sub_sd(golden("ae_cms.npz"), "sd")
    n = 30011
    table = synth.cms_table(n, seed=44)
    files = {}
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
        (proj / "config" / "P_config.py").write_text(_CFG.format(path=data))
        for mode in ("compress", "decompress"):
            launch = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port",
                      str(_free_port())] if world == 2 else [sys.executable]
            r = subprocess.run(launch + ["-m", "baler_b200", "--project", "WS", "P", "--mode", mode], cwd=wd,
                               env=dict(os.environ, PYTHONPATH=ROOT), capture_output=True, text=True, timeout=600)
            assert r.returncode == 0, r.stderr[-3000:]
        comp = np.load(proj / "output" / "compressed_output" / "compressed.npz")
        files[world] = [comp[k].tobytes() for k in ("data", "latent_min", "latent_step")]
        files[world].append(np.load(proj / "output" / "decompressed_output" / "decompressed.npz")["data"].tobytes())
    assert files[1] == files[2]
