"""precision "fp64": the float64 chain against the reference's float64 numbers.

Tolerance 1e-12 on max|d|/max|ref| and on ||d||2/||ref||2 (the float64 arithmetic of the reference in another summation
order differs by ~1e-15); column min / max and the features are bit-exact; integer columns after the reference's
truncation are equal."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_l2, rel_max, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import engine, synth
from baler_b200.modules import models

pytestmark = pytest.mark.gpu
TOL = 1e-12
TYPE_LIST = ["float64"] * 12 + ["int"] * 7 + ["float64"] * 3 + ["int"] * 2


def close(a, ref, tol=TOL):
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    assert a.shape == ref.shape
    assert rel_max(a, ref) <= tol and rel_l2(a, ref) <= tol, (rel_max(a, ref), rel_l2(a, ref))


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def ae(golden):
    g = golden("ae_cms.npz")
    m = models.AE(24, 15)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sub_sd(g, "sd").items()})
    return m.eval(), sub_sd(g, "sd"), g


def test_ae_cms_golden(ae):
    """float32 table normalised in float32 (bit-equal to numpy), then the float64 chain; decode and fused un-normalisation"""
    m, _, g = ae
    codec = m.codec()
    mn, rg = cuda(g["norm_features"][0]), cuda(g["norm_features"][1])
    z = codec.encode(cuda(g["x_raw"]), mn, rg, out_dtype=torch.float64, precision="fp64")
    assert z.dtype == torch.float64
    close(z, g["latent"])
    lat = cuda(g["latent"].astype(np.float64))
    close(codec.decode(lat), g["recon"])
    close(codec.decode(lat, mn, rg), g["unnorm"])


def test_dropout_bn_eval_fp64(golden):
    g = golden("ae_dbn.npz")
    m = models.AE_Dropout_BN(24, 15)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sub_sd(g, "sd0").items()})
    codec = m.eval().codec()
    close(codec.encode(cuda(g["x_norm"][:256].astype(np.float64))), g["latent_eval"])
    close(codec.decode(cuda(g["latent_eval"].astype(np.float64))), g["recon_eval"])


def _cli_workspace(tmp_path, monkeypatch, sd, table, feats, **extra):
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
        save_error_bounded_deltas, convert_to_blocks, precision = False, False, "fp64"
    for k, v in extra.items():
        setattr(cfg, k, v)
    return out, cfg


def test_cli_roundtrip_equals_reference_files(golden, tmp_path, monkeypatch):
    """--mode compress / decompress with precision "fp64" on the workspace whose files the reference wrote
    (tests/golden/cli_roundtrip.npz): latent and float columns to 1e-12, integer columns equal"""
    from baler_b200 import baler
    g = golden("cli_roundtrip.npz")
    out, cfg = _cli_workspace(tmp_path, monkeypatch, sub_sd(g, "sd"), synth.cms_table(4096, seed=17), g["norm_features"],
                              type_list=TYPE_LIST)
    baler.perform_compression(out, cfg, False)
    comp = np.load(os.path.join(out, "compressed_output", "compressed.npz"))
    assert comp["data"].dtype == np.float64 and comp["data"].shape == (4096, 15)
    assert comp["normalization_features"].tobytes() == g["comp_norm_features"].tobytes()
    close(comp["data"], g["compressed"])
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    ref = g["decompressed"]
    assert dec.dtype == np.float64 and dec.shape == ref.shape
    fl = [c for c, t in enumerate(TYPE_LIST) if t != "int"]
    it = [c for c, t in enumerate(TYPE_LIST) if t == "int"]
    close(dec[:, fl], ref[:, fl])
    assert np.array_equal(dec[:, it], ref[:, it]), int((dec[:, it] != ref[:, it]).sum())


def test_cli_float64_table_with_large_offsets_fp64(ae, tmp_path, monkeypatch):
    """the float64 file with a 1e9 event counter: normalised and un-normalised in float64 on the device (the host float64
    normalisation around the float32 kernels is not used)"""
    from baler_b200 import baler
    from baler_b200.modules import data_processing

    def no_host_path(*a, **k):
        raise AssertionError("host float64 normalisation used")
    monkeypatch.setattr(data_processing, "normalize_float64_host", no_host_path)
    _, sd, _ = ae
    n = 4096
    table = synth.cms_table(n, seed=29).astype(np.float64)
    table[:, 5] = 1.0e9 + np.arange(n) % 977
    table[:, 11] = -4.0e7 + 0.25 * table[:, 11]
    feats = orc.find_minmax(table)
    out, cfg = _cli_workspace(tmp_path, monkeypatch, sd, table, feats)
    baler.perform_compression(out, cfg, False)
    z = np.load(os.path.join(out, "compressed_output", "compressed.npz"))["data"]
    z_ref = orc.compress(sd, table)
    assert z.dtype == np.float64
    close(z, z_ref)
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    ref = orc.decompress(sd, z_ref, feats)
    assert dec.dtype == np.float64 and dec.shape == ref.shape
    assert (np.abs(dec - ref) / feats[1]).max() <= TOL


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("F,Z", [(1, 1), (7, 5), (24, 15), (31, 31), (64, 40), (100, 63), (256, 160)])
def test_ragged_shapes_vs_numpy_chain(F, Z, dtype):
    torch.manual_seed(F * 1000 + Z)
    m = models.AE(F, Z).eval()
    sd = {k: v.numpy() for k, v in m.state_dict().items()}
    codec = m.codec()
    rng = np.random.default_rng(F + Z)
    table = (rng.standard_normal((100003, F)) * rng.uniform(0.5, 50.0, F) + rng.uniform(-100, 100, F)).astype(dtype)
    mn_np, mx_np = table.min(0), table.max(0)
    rg_np = mx_np - mn_np  # one subtraction in the table's dtype, as find_minmax
    mn, rg = cuda(mn_np), cuda(rg_np)
    for n in (0, 1, 2, 31, 32, 33, 1000, 100003):
        x = table[:n]
        z = codec.encode(cuda(x), mn, rg, out_dtype=torch.float64, precision="fp64")
        assert z.dtype == torch.float64 and z.shape == (n, Z)
        y = codec.decode(z, mn, rg)
        assert y.dtype == torch.float64 and y.shape == (n, F)
        if n == 0:
            continue
        xn = ((x - mn_np) / rg_np).astype(np.float64)  # numpy: normalised in the table's dtype, then widened
        close(z, orc.ae_encode(sd, xn))
        zd = z.cpu().numpy()
        close(y, orc.renormalize(orc.ae_decode(sd, zd), mn_np.astype(np.float64), rg_np.astype(np.float64)))
        y32 = codec.decode(z.float(), precision="fp64")  # float32 latent in, float32 rows out
        assert y32.dtype == torch.float32
        close(y32, orc.ae_decode(sd, zd.astype(np.float32).astype(np.float64)), 1e-6)


def test_colminmax_f64_bit_exact():
    rng = np.random.default_rng(4)
    for n, c in ((1, 24), (7, 24), (1000, 24), (100003, 24), (4099, 25), (513, 3), (20, 200), (3001, 2000)):
        t = rng.standard_normal((n, c)) * rng.uniform(0.1, 1e9, c) + 1e9
        mn, mx = engine.colminmax(cuda(t))
        assert mn.dtype == torch.float64
        assert mn.cpu().numpy().tobytes() == t.min(0).tobytes() and mx.cpu().numpy().tobytes() == t.max(0).tobytes()
    t = rng.standard_normal((5001, 24))
    t[17, 3] = np.nan
    t[:, 7] = 0.0
    t[100, 7] = -0.0  # order-preserving keys: -0 < +0
    t[:, 9] = -0.0
    flat = cuda(np.concatenate([[0.0], t.ravel()]))
    view = flat[1:].view(5001, 24)  # 8-byte aligned only: the scalar path
    for x in (cuda(t), view):
        mn, mx = (v.cpu().numpy() for v in engine.colminmax(x))
        assert np.isnan(mn[3]) and np.isnan(mx[3])  # numpy: NaN propagates, per column
        assert np.signbit(mn[7]) and not np.signbit(mx[7]) and np.signbit(mn[9]) and np.signbit(mx[9])
        ok = [c for c in range(24) if c not in (3, 7, 9)]
        assert mn[ok].tobytes() == t.min(0)[ok].tobytes() and mx[ok].tobytes() == t.max(0)[ok].tobytes()


def test_host_pipeline_bits_do_not_depend_on_chunks_or_buffers(ae):
    """a multi-chunk host pipeline call gives the bits of one device-resident call; pinned and pageable buffers agree"""
    m, _, _ = ae
    codec = m.codec()
    n = (1 << 20) + 777  # 4 pipeline chunks and a ragged tail
    t32 = synth.cms_table(n, seed=41)
    t64 = t32.astype(np.float64) * 1.0000001 + 3.0
    z64, f64 = codec.compress_host(t64, recompute_minmax=True, z_dtype=np.float64, precision="fp64")
    assert f64.dtype == np.float64 and f64.tobytes() == orc.find_minmax(t64).tobytes()
    zd = codec.encode(cuda(t64), cuda(f64[0]), cuda(f64[1]))
    assert z64.tobytes() == zd.cpu().numpy().tobytes()
    y64 = codec.decompress_host(z64, features=f64, y_dtype=np.float64, precision="fp64")
    assert y64.tobytes() == codec.decode(zd, cuda(f64[0]), cuda(f64[1])).cpu().numpy().tobytes()
    z32, f32 = codec.compress_host(t32, recompute_minmax=True, z_dtype=np.float64, precision="fp64")
    assert f32.dtype == np.float32 and f32.tobytes() == orc.find_minmax(t32).tobytes()
    zd32 = codec.encode(cuda(t32), cuda(f32[0]), cuda(f32[1]), out_dtype=torch.float64, precision="fp64")
    assert z32.tobytes() == zd32.cpu().numpy().tobytes()
    y32 = codec.decompress_host(z32, features=f32, y_dtype=np.float64, precision="fp64")
    assert y32.tobytes() == codec.decode(zd32, cuda(f32[0]), cuda(f32[1])).cpu().numpy().tobytes()
    pin = torch.empty(t64.shape, dtype=torch.float64, pin_memory=True).numpy()
    pin[...] = t64
    zp = torch.empty(z64.shape, dtype=torch.float64, pin_memory=True).numpy()
    codec.compress_host(pin, features=f64, precision="fp64", out=zp)
    assert zp.tobytes() == z64.tobytes()
    yp = torch.empty(y64.shape, dtype=torch.float64, pin_memory=True).numpy()
    codec.decompress_host(zp, features=f64, precision="fp64", out=yp)
    assert yp.tobytes() == y64.tobytes()


def test_trim_releases_and_repacks(ae):
    m, _, g = ae
    codec = m.codec()
    x = cuda(g["x_norm"].astype(np.float64))
    z1 = codec.encode(x)
    codec.trim()
    assert torch.equal(codec.encode(x), z1)


_CFG = """
def set_config(c):
    c.input_path = {path!r}
    c.data_dimension, c.compression_ratio, c.apply_normalization, c.model_name = 1, 1.6, True, "AE"
    c.batch_size, c.custom_norm, c.extra_compression, c.separate_model_saving = 512, False, False, False
    c.save_error_bounded_deltas, c.convert_to_blocks, c.precision = False, False, "fp64"
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_torchrun_two_ranks_write_the_files_of_one_process(ae, tmp_path):
    """2-rank torchrun compress / decompress with "fp64" writes the bytes one process writes (row shards, one min / max
    exchange in the table's dtype)"""
    _, sd, _ = ae
    n = 30011
    table = synth.cms_table(n, seed=43).astype(np.float64)
    table[:, 5] = 1.0e9 + np.arange(n) % 977
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
        files[world] = [np.load(proj / "output" / p)["data"].tobytes()
                        for p in ("compressed_output/compressed.npz", "decompressed_output/decompressed.npz")]
    assert files[1] == files[2]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]
