"""latent_dtype "q2" ... "q8" on the device: packed codes and parameters bit-equal to the numpy mirror
(tests/latent_packed_ref.py) for every b, on the device entry points at several latent widths and on every codec the host
pipelines take; decompression bit-equal to decode of the mirror's dequantised latent; bits = 8 equal to the 8-bit entry
points byte for byte; the CLI round trip at "q4"; error-bounded deltas at "q3"; the 2-rank file."""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import latent_packed_ref as ref
from conftest import ROOT, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import _lib, latent_q8, synth
from test_gpu_latent_q8 import CODECS, TYPE_LIST, _ae, _free_port, _pinned, _workspace

pytestmark = pytest.mark.gpu
BITS = list(range(2, 9))


def _mirror(z, bits):
    codes, lo, step = ref.quantize(z, bits)
    return ref.pack(codes, bits), lo, step, ref.dequantize(codes, lo, step, bits)


def _same(got, want, what):
    got = np.asarray(got)
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, got.shape, want.dtype, want.shape)
    a, b = got.view(np.uint8), want.view(np.uint8)
    assert np.array_equal(a, b), (what, int((a != b).sum()))


@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("z_dim", [1, 15, 31, 33, 250])
@pytest.mark.parametrize("n", [1, 127, 128, 129, 4099])
def test_device_entry_points_bit_equal_to_mirror(golden, bits, z_dim, n):
    """bb_latent_quantize_packed / bb_latent_dequantize_packed on a latent with awkward values in it"""
    codec, _ = _ae(golden)  # (only its context is used: the widths here are not the model's)
    rng = np.random.default_rng(1000 * bits + z_dim + n)
    z = (rng.standard_normal((n, z_dim)) * rng.uniform(0.01, 100, z_dim)).astype(np.float32)
    z[n // 2, 0] = np.nan
    if z_dim > 2:
        z[:, 1] = 0.5  # a constant column
        z[n // 3, 2] = -np.inf
    zd = torch.from_numpy(z).cuda()
    nb, w = latent_q8.n_blocks(n), latent_q8.row_bytes(z_dim, bits)
    codes = torch.full((n, w), 0xAA, dtype=torch.uint8, device="cuda")
    lo, step = (torch.empty((nb, z_dim), dtype=torch.float32, device="cuda") for _ in range(2))
    back = torch.empty_like(zd)
    lib = _lib.lib()
    assert lib.bb_latent_quantize_packed(codec.ctx.handle, zd.data_ptr(), n, z_dim, bits, codes.data_ptr(), lo.data_ptr(),
                                         step.data_ptr(), None) == 0
    assert lib.bb_latent_dequantize_packed(codec.ctx.handle, bits, codes.data_ptr(), lo.data_ptr(), step.data_ptr(), n, z_dim,
                                           back.data_ptr(), None) == 0
    torch.cuda.synchronize()
    want = _mirror(z, bits)
    for got, w_, what in zip((codes, lo, step, back), want, ("codes", "lo", "step", "dequantised")):
        _same(got.cpu().numpy(), w_, what)


def _check(codec, x, bits, precision, pinned=False):
    mn, mx = np.nanmin(x, axis=0), np.nanmax(x, axis=0)
    feats = np.stack([mn, mx - mn]).astype(np.float32)
    n = len(x)
    out = None
    if pinned:
        xp = _pinned(x.shape, torch.float32)
        xp[:] = x
        x = xp
        nb, w = latent_q8.n_blocks(n), latent_q8.row_bytes(codec.z_dim, bits)
        out = latent_q8.PackedLatent(_pinned((n, w), torch.uint8), _pinned((nb, codec.z_dim), torch.float32),
                                     _pinned((nb, codec.z_dim), torch.float32), bits)
    q, _ = codec.compress_host_packed(x, bits, features=feats, precision=precision, out=out)
    z, _ = codec.compress_host(x, features=feats, z_dtype=np.float32, precision=precision)  # the device's own latent
    packed, lo, step, back = _mirror(z, bits)
    assert q.bits == bits
    for got, want, what in zip(q[:3], (packed, lo, step), ("codes", "lo", "step")):
        _same(got, want, what)
    y = codec.decompress_host_packed(q, features=feats, y_dtype=np.float32, precision=precision)
    y_ref = codec.decompress_host(back, features=feats, y_dtype=np.float32, precision=precision)
    _same(y, y_ref, "decompressed")
    return q, z


@pytest.mark.parametrize("bits", BITS)
@pytest.mark.parametrize("name", sorted(CODECS))
@pytest.mark.parametrize("n", [1, 129, 4099])
def test_codecs_bit_equal_to_mirror(golden, bits, name, n):
    build, precision = CODECS[name]
    codec, make = build(golden)
    _check(codec, make(n, seed=n + bits), bits, precision)


@pytest.mark.parametrize("bits", [2, 5, 8])
@pytest.mark.parametrize("n", [262_143, 262_144, 262_145])
def test_around_one_pipeline_chunk(golden, bits, n):
    codec, make = _ae(golden)
    _check(codec, make(n, seed=n), bits, "auto")


@pytest.mark.parametrize("bits,pinned", [(3, False), (3, True), (4, True), (7, False)])
def test_several_pipeline_chunks(golden, bits, pinned):
    """5,000,001 rows: 16 pipeline chunks of whole blocks and a ragged last block, pinned and pageable buffers"""
    codec, make = _ae(golden)
    x = make(5_000_001, seed=3)
    x[123_457, 4] = np.nan  # a NaN row stays NaN
    q, _ = _check(codec, x, bits, "auto", pinned)
    assert (ref.unpack(q.codes[123_457:123_458], 15, bits) == 2 ** bits - 1).any()


def test_bits8_gives_the_q8_bytes(golden):
    """bb_compress_host_packed(bits = 8) and bb_compress_host_q8 write the same bytes, and both decompress alike"""
    codec, make = _ae(golden)
    x = make(300_001, seed=12)
    lib = _lib.lib()
    a, b = latent_q8.empty(len(x), 15), latent_q8.empty(len(x), 15)
    feats = [orc.find_minmax(x).astype(np.float32) for _ in range(2)]
    assert lib.bb_compress_host_q8(codec.handle, x.ctypes.data, len(x), feats[0].ctypes.data, 1, a.codes.ctypes.data,
                                   a.lo.ctypes.data, a.step.ctypes.data, _lib.BB_PREC_AUTO) == 0
    assert lib.bb_compress_host_packed(codec.handle, x.ctypes.data, len(x), feats[1].ctypes.data, 1, 8, b.codes.ctypes.data,
                                       b.lo.ctypes.data, b.step.ctypes.data, _lib.BB_PREC_AUTO) == 0
    for u, v, what in zip(a, b, ("codes", "lo", "step")):
        _same(u, v, what)
    y = [np.empty((len(x), 24), np.float32) for _ in range(2)]
    assert lib.bb_decompress_host_q8(codec.handle, a.codes.ctypes.data, a.lo.ctypes.data, a.step.ctypes.data, len(x),
                                     feats[0].ctypes.data, y[0].ctypes.data, _lib.BB_F32, _lib.BB_PREC_AUTO) == 0
    assert lib.bb_decompress_host_packed(codec.handle, 8, a.codes.ctypes.data, a.lo.ctypes.data, a.step.ctypes.data, len(x),
                                         feats[0].ctypes.data, y[1].ctypes.data, _lib.BB_F32, _lib.BB_PREC_AUTO) == 0
    _same(y[0], y[1], "decompressed")


def test_bits_out_of_range_and_fp64_are_refused(golden):
    codec, make = _ae(golden)
    x = make(300, seed=1)
    lib = _lib.lib()
    zd = torch.from_numpy(np.zeros((300, 15), np.float32)).cuda()
    buf = torch.zeros((300, 15), dtype=torch.uint8, device="cuda")
    par = torch.zeros((3, 15), dtype=torch.float32, device="cuda")
    for bits in (0, 1, 9, 16, -8):
        q = latent_q8.empty_packed(300, 15, 8)
        assert lib.bb_compress_host_packed(codec.handle, x.ctypes.data, 300, None, 0, bits, q.codes.ctypes.data,
                                           q.lo.ctypes.data, q.step.ctypes.data, _lib.BB_PREC_AUTO) == -1  # BB_ERR_INVALID
        y = np.empty((300, 24), np.float32)
        assert lib.bb_decompress_host_packed(codec.handle, bits, q.codes.ctypes.data, q.lo.ctypes.data, q.step.ctypes.data,
                                             300, None, y.ctypes.data, _lib.BB_F32, _lib.BB_PREC_AUTO) == -1
        assert lib.bb_latent_quantize_packed(codec.ctx.handle, zd.data_ptr(), 300, 15, bits, buf.data_ptr(), par.data_ptr(),
                                             par.data_ptr(), None) == -1
        assert lib.bb_latent_dequantize_packed(codec.ctx.handle, bits, buf.data_ptr(), par.data_ptr(), par.data_ptr(), 300,
                                               15, zd.data_ptr(), None) == -1
    for bits in (2, 5):
        q = latent_q8.empty_packed(300, 15, bits)
        assert lib.bb_compress_host_packed(codec.handle, x.ctypes.data, 300, None, 0, bits, q.codes.ctypes.data,
                                           q.lo.ctypes.data, q.step.ctypes.data, _lib.BB_PREC_FP64) == -2  # UNSUPPORTED
        with pytest.raises(NotImplementedError, match="latent_dtype='q%d'" % bits):
            codec.compress_host_packed(x, bits, precision="fp64")
        with pytest.raises(NotImplementedError, match="latent_dtype='q%d'" % bits):
            codec.decompress_host_packed(q, precision="fp64")


def test_tc4_range_fallback_keeps_the_format(golden):
    """the split16 range guard re-runs the rows on the fp32 kernel; the packed result is then the fp32 one"""
    codec, make = _ae(golden)
    x = make(1000, seed=9)
    x[10, 3] = 1e30
    feats = orc.find_minmax(make(1000, seed=9)).astype(np.float32)
    for bits in (3, 6):
        q, _ = codec.compress_host_packed(x, bits, features=feats)
        q32, _ = codec.compress_host_packed(x, bits, features=feats, precision="fp32")
        for a, b, what in zip(q[:3], q32[:3], ("codes", "lo", "step")):
            _same(a, b, what)


# ---------------------------------------------------------------- the CLI


def test_cli_train_compress_decompress_info_q4(tmp_path, monkeypatch, capsys):
    from baler_b200 import baler
    from baler_b200.modules import data_processing, helper, models
    from test_gpu_train_fp64 import _cfg, _project
    n = 20_000
    table = synth.cms_table(n, seed=31)
    out, path = _project(tmp_path, monkeypatch, table)
    cfg = _cfg(helper, path, precision="auto", latent_dtype="q4", type_list=TYPE_LIST, l1=False, activation_extraction=False)
    torch.manual_seed(0)
    baler.perform_training(out, cfg, False)
    baler.perform_compression(out, cfg, False)
    comp_path = os.path.join(out, "compressed_output", "compressed.npz")
    comp = np.load(comp_path)
    assert sorted(comp.files) == sorted(["data", "latent_min", "latent_step", "latent_block_rows", "latent_bits", "names",
                                         "normalization_features"])
    assert comp["data"].dtype == np.uint8 and comp["data"].shape == (n, 8)  # ceil(15 * 4 / 8)
    assert comp["latent_min"].shape == comp["latent_step"].shape == (157, 15) and int(comp["latent_bits"]) == 4
    q4_bytes = os.stat(comp_path).st_size
    payload = n * 8 + 2 * 157 * 15 * 4  # ceil(z b / 8) + 2 * 4 z / 128 bytes per row (8.94 for z = 15 at 4 bits)
    rest = q4_bytes - sum(comp[k].nbytes for k in ("names", "normalization_features"))
    assert payload <= rest <= payload + 4096  # (npy headers and zip records)
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    assert dec.shape == table.shape and np.isfinite(dec).all()
    it = [c for c, t in enumerate(TYPE_LIST) if t == "int"]
    m = data_processing.load_model(models.AE, os.path.join(out, "compressed_output", "model.pt"), n_features=24, z_dim=15)
    y = m.eval().codec().decompress_host_packed(latent_q8.read(comp), features=np.load(
        os.path.join(out, "training", "normalization_features.npy")).reshape(2, -1), y_dtype=dec.dtype)
    y[:, it] = np.trunc(y[:, it])
    assert np.array_equal(y, dec)
    capsys.readouterr()
    baler.print_info(out, cfg)
    assert "Compressed file size: %s MB" % round(q4_bytes / (1024 * 1024), 4) in capsys.readouterr().out
    cfg.latent_dtype = "q8"  # the same model's 8-bit file: 7 bytes more per row, no latent_bits key
    baler.perform_compression(out, cfg, False)
    comp8 = np.load(comp_path)
    assert "latent_bits" not in comp8.files and comp8["data"].shape == (n, 15)
    assert abs(os.stat(comp_path).st_size - q4_bytes - 7 * n) < 1024


def test_error_bounded_deltas_correct_the_q3_reconstruction(golden, tmp_path, monkeypatch):
    """save_error_bounded_deltas with q3: the deltas are taken against decode(dequantise(quantise(encode(x)))), so every
    stored hit, applied by decompress, lands within float16 rounding of the input"""
    from baler_b200 import baler
    g = golden("eb_deltas.npz")
    table, bound, bs = g["table"], float(g["bound"]), 256
    feats = orc.find_minmax(table)
    out, cfg = _workspace(tmp_path, monkeypatch, sub_sd(golden("ae_cms.npz"), "sd"), table, feats,
                          save_error_bounded_deltas=True, error_bounded_requirement=bound, batch_size=bs, latent_dtype="q3")
    baler.perform_compression(out, cfg, False)
    comp = np.load(os.path.join(out, "compressed_output", "compressed.npz"))
    assert comp["data"].shape == (len(table), 6) and int(comp["latent_bits"]) == 3
    index = np.load(gzip.GzipFile(os.path.join(out, "compressed_output", "compressed_batch_index_metadata.npz.gz"), "r"),
                    allow_pickle=True)
    hits = [(int(r) + bs * int(b), int(c)) for b, (rows, cols) in zip(index[0], index[1]) for r, c in zip(rows, cols)]
    assert hits
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    r, c = np.array(hits).T
    x_n = (table[r, c].astype(np.float64) - feats[0][c]) / feats[1][c]
    y_n = (dec[r, c].astype(np.float64) - feats[0][c]) / feats[1][c]
    assert (np.abs(y_n - x_n) <= 2.0 ** -11 * (np.abs(x_n) + 2.0) + 1e-6).all(), float(np.abs(y_n - x_n).max())


_CFG = """
def set_config(c):
    c.input_path = {path!r}
    c.data_dimension, c.compression_ratio, c.apply_normalization, c.model_name = 1, 1.6, True, "AE"
    c.batch_size, c.custom_norm, c.extra_compression, c.separate_model_saving = 512, False, False, False
    c.save_error_bounded_deltas, c.convert_to_blocks, c.latent_dtype = False, False, "q4"
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_torchrun_two_ranks_write_the_file_of_one_process_q4(golden, tmp_path):
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
        files[world] = [comp[k].tobytes() for k in ("data", "latent_min", "latent_step", "latent_bits")]
        files[world].append(np.load(proj / "output" / "decompressed_output" / "decompressed.npz")["data"].tobytes())
    assert files[1] == files[2]
