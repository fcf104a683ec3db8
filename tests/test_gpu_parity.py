"""Parity of the CUDA path (through the C ABI) with the oracle and the golden vectors.

Tolerance of the float path (BASELINE.json north_star, SURVEY 8d): max|d|/max|ref| <= 1e-5 and
||d||2/||ref||2 <= 1e-5 per tensor against the float64 reference; normalisation and column min/max are
bit-exact float32."""
import os

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_l2, rel_max, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import engine, synth
from baler_b200.modules import models

pytestmark = pytest.mark.gpu
TOL = 1e-5
TYPE_LIST = ["float64"] * 12 + ["int"] * 7 + ["float64"] * 3 + ["int"] * 2


def close(a, ref, tol=TOL):
    assert a.shape == ref.shape
    assert rel_max(a, ref) <= tol and rel_l2(a, ref) <= tol, (rel_max(a, ref), rel_l2(a, ref))


@pytest.fixture(scope="module")
def ae(golden):
    g = golden("ae_cms.npz")
    m = models.AE(24, 15)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sub_sd(g, "sd").items()})
    return m.eval(), sub_sd(g, "sd"), g


def precisions(codec):
    return ["fp32"] + (["split16"] if codec.auto_precision == "split16" else [])


# ------------------------------------------------------------------ column statistics / normalisation
@pytest.mark.parametrize("n,c", [(1, 24), (7, 24), (1000, 24), (100003, 24), (4099, 25), (513, 3), (20, 200)])
def test_colminmax_bit_exact(n, c):
    rng = np.random.default_rng(n * 31 + c)
    t = (rng.normal(size=(n, c)) * rng.uniform(0.1, 1e4, size=c)).astype(np.float32)
    mn, mx = engine.colminmax(torch.from_numpy(t).cuda())
    assert np.array_equal(mn.cpu().numpy(), t.min(0)) and np.array_equal(mx.cpu().numpy(), t.max(0))


def test_colminmax_unaligned_and_nan():
    t = synth.cms_table(5001)
    flat = torch.from_numpy(np.concatenate([[0.0], t.ravel()]).astype(np.float32)).cuda()
    view = flat[1:].view(5001, 24)  # 4-byte aligned only: scalar path
    mn, mx = engine.colminmax(view)
    assert np.array_equal(mn.cpu().numpy(), t.min(0)) and np.array_equal(mx.cpu().numpy(), t.max(0))
    t[17, 3] = np.nan
    mn, mx = engine.colminmax(torch.from_numpy(t).cuda())
    assert np.isnan(mn[3].item()) and np.isnan(mx[3].item())  # numpy min/max propagate NaN
    assert np.array_equal(np.delete(mx.cpu().numpy(), [0, 1, 2, 3]), np.delete(t.max(0), [0, 1, 2, 3]))


def test_normalize_renormalize_bit_exact(golden):
    g = golden("ae_cms.npz")
    table = synth.cms_table(20000)
    x = torch.from_numpy(table).cuda()
    mn, mx = engine.colminmax(x)
    rg = mx - mn
    assert np.array_equal(np.stack([mn.cpu().numpy(), rg.cpu().numpy()]), g["norm_features"])
    norm = engine.normalize_table(x, mn, rg).cpu().numpy()
    assert np.array_equal(norm, orc.normalize(table)) and np.array_equal(norm[:256], g["x_norm"])
    y = torch.from_numpy(g["recon"].astype(np.float32)).cuda()
    un = engine.normalize_table(y, mn, rg, inverse=True).cpu().numpy()
    close(un, g["unnorm"], 2e-7)


def test_host_helpers_match_reference_known_answers():
    # /root/reference/tests/test_data_processing.py:52-121 by value, through the drop-in functions
    from baler_b200.modules import data_processing as dp

    for data, exp in (([[1, 2, 3], [4, 5, 6], [7, 8, 9]], [[1, 2, 3], [6, 6, 6]]),
                      ([[-1, -2, -3], [-4, -5, -6], [-7, -8, -9]], [[-7, -8, -9], [6, 6, 6]]),
                      ([[0, 0, 0], [1, 1, 1], [2, 2, 2]], [[0, 0, 0], [2, 2, 2]])):
        assert np.array_equal(dp.find_minmax(np.array(data)), np.array(exp))
    np.testing.assert_almost_equal(dp.normalize([1, 2, 3, 4, 5], False), [0.0, 0.25, 0.5, 0.75, 1.0])
    np.testing.assert_almost_equal(dp.normalize([1, 2, 3, 4, 5], True), [1, 2, 3, 4, 5])
    np.testing.assert_allclose(dp.renormalize_std(np.array([0.1, 0.2, 0.3, 0.4, 0.5]), 1, 2), [1.2, 1.4, 1.6, 1.8, 2.0], rtol=1e-6)
    data = np.array([[-1, 2], [-0.5, 6], [0, 10], [1, 18]], dtype=np.float64)
    norm = (data - data.min(0)) / (data.max(0) - data.min(0))
    np.testing.assert_allclose(dp.renormalize_func(norm, [-1, 2], [2, 16]), data, rtol=1e-6)


# ------------------------------------------------------------------ encode / decode
def test_encode_decode_golden(ae):
    m, sd, g = ae
    codec = m.codec()
    feats = torch.from_numpy(g["norm_features"]).cuda()
    x = torch.from_numpy(g["x_raw"]).cuda()
    for p in precisions(codec):
        z = codec.encode(x, feats[0].contiguous(), feats[1].contiguous(), precision=p)
        close(z.cpu().numpy(), g["latent"])
        y = codec.decode(torch.from_numpy(g["latent"].astype(np.float32)).cuda(), precision=p)
        close(y.cpu().numpy(), g["recon"])
        y2 = codec.decode(z, feats[0].contiguous(), feats[1].contiguous(), precision=p)
        close(y2.cpu().numpy(), g["unnorm"])


@pytest.mark.parametrize("n", [1, 2, 79, 80, 81, 160, 1000, 11840, 11841, 200000])
def test_encode_decode_vs_oracle_ragged(ae, n):
    m, sd, _ = ae
    codec = m.codec()
    x = orc.normalize(synth.cms_table(max(n, 1000), seed=n))[:n]  # ranges from >= 1000 rows: no zero range
    zr = orc.ae_encode(sd, x)
    yr = orc.ae_decode(sd, zr)
    for p in precisions(codec):
        z = codec.encode(torch.from_numpy(x).cuda(), precision=p)
        close(z.cpu().numpy(), zr)
        y = codec.decode(z, precision=p)
        close(y.cpu().numpy(), yr)


def test_empty_input(ae):
    m, _, _ = ae
    z = m.codec().encode(torch.empty((0, 24), dtype=torch.float32, device="cuda"))
    assert z.shape == (0, 15)
    y = m.codec().decode(z)
    assert y.shape == (0, 24)
    zh, _ = m.codec().compress_host(np.empty((0, 24), dtype=np.float32))
    assert zh.shape == (0, 15)


def test_unnormalised_input_range(ae):
    """apply_normalization=False feeds raw values (|x| up to ~1e3): the range guard of the split path
    must either pass the tolerance or fall back, never return garbage"""
    m, sd, _ = ae
    x = synth.cms_table(4096, seed=5)
    zr = orc.ae_encode(sd, x.astype(np.float64))
    z = m.codec().encode(torch.from_numpy(x).cuda(), precision="auto")
    close(z.cpu().numpy(), zr)


def test_fp16_latent_opt_in(ae):
    m, sd, g = ae
    codec = m.codec()
    x = torch.from_numpy(g["x_norm"]).cuda()
    z16 = codec.encode(x, out_dtype=torch.float16)
    assert z16.dtype == torch.float16
    close(z16.float().cpu().numpy(), g["latent"], 1e-3)  # fp16 storage: 2^-11 relative, labelled opt-in
    y = codec.decode(z16)
    close(y.cpu().numpy(), orc.ae_decode(sd, z16.float().cpu().numpy().astype(np.float64)))


def test_model_protocol(ae):
    m, sd, g = ae
    z = m.encode(torch.from_numpy(g["x_norm"]).double())  # reference feeds float64 tensors (helper.py:565)
    assert z.dtype == torch.float64 and z.is_cuda
    close(z.cpu().numpy(), g["latent"])
    close(m(torch.from_numpy(g["x_norm"])).cpu().numpy(), g["recon"])
    close(m.decode(g["latent"]).cpu().numpy(), g["recon"])


def test_dropout_bn_eval(golden):
    g = golden("ae_dbn.npz")
    m = models.AE_Dropout_BN(24, 15)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sub_sd(g, "sd0").items()})
    m.eval()
    close(m.encode(g["x_norm"][:256]).cpu().numpy(), g["latent_eval"])
    close(m.decode(g["latent_eval"]).cpu().numpy(), g["recon_eval"])
    with pytest.raises(NotImplementedError):
        m.train().forward(g["x_norm"][:8])


# ------------------------------------------------------------------ host pipeline (what helper.compress calls)
def test_compress_decompress_host_roundtrip(ae):
    m, sd, _ = ae
    codec = m.codec()
    table = synth.cms_table(30011, seed=3)
    z, feats = codec.compress_host(table, recompute_minmax=True, z_dtype=np.float64)
    assert z.dtype == np.float64 and np.array_equal(feats, orc.find_minmax(table))
    zr = orc.compress(sd, table)
    close(z, zr)
    z32, _ = codec.compress_host(table, features=feats, z_dtype=np.float32)
    assert np.array_equal(z32.astype(np.float64), z)  # given features == recomputed features, widening is exact
    y = codec.decompress_host(z, features=feats, y_dtype=np.float64)
    close(y, orc.decompress(sd, zr, feats))
    y_plain = codec.decompress_host(z32, y_dtype=np.float32)
    close(y_plain, orc.ae_decode(sd, zr))


@pytest.mark.parametrize("n", [1, 7, 1000, 30011])
def test_compress_host_statistics_match_the_kernel(ae, n, monkeypatch):
    """the column min / max that bb_compress_host finds on host threads while the table uploads (resident path) equals the
    device kernel's - bit for bit, incl. -0 < +0 and NaN propagation per column - and the streaming two-pass path"""
    m, _, _ = ae
    codec = m.codec()
    rng = np.random.default_rng(n)
    table = synth.cms_table(n, seed=5)
    table[rng.integers(0, n, size=max(1, n // 50)), rng.integers(0, 24, size=max(1, n // 50))] = 0.0
    table[rng.integers(0, n, size=max(1, n // 80)), rng.integers(0, 24, size=max(1, n // 80))] = -0.0
    z1, feats = codec.compress_host(table, recompute_minmax=True, z_dtype=np.float32)
    mn, mx = engine.colminmax(torch.from_numpy(table).cuda())
    ref = np.stack([mn.cpu().numpy(), (mx - mn).cpu().numpy()])
    assert feats.tobytes() == ref.tobytes()
    for hook in ("BALER_B200_NO_RESIDENT", "BALER_B200_DEVICE_MINMAX"):  # the two device-side statistics paths
        monkeypatch.setenv(hook, "1")
        z2, feats2 = codec.compress_host(table, recompute_minmax=True, z_dtype=np.float32)
        assert feats2.tobytes() == feats.tobytes() and z2.tobytes() == z1.tobytes()
        monkeypatch.delenv(hook)
    if n >= 1000:  # numpy semantics: a NaN makes that column's min and max NaN, and only that column's
        table[n // 3, 5] = np.nan
        table[n - 1, 23] = np.nan
        _, fn = codec.compress_host(table, recompute_minmax=True, z_dtype=np.float32)
        bad = np.zeros(24, dtype=bool)
        bad[[5, 23]] = True
        assert np.isnan(fn[:, bad]).all() and fn[:, ~bad].tobytes() == feats[:, ~bad].tobytes()


def test_host_pipeline_multi_chunk(ae):
    """more rows than one pipeline chunk (2^21): slots, events and ragged tail; checked on sampled rows"""
    m, sd, _ = ae
    n = (1 << 22) + 12345
    rng = np.random.default_rng(9)
    base = synth.cms_table(1 << 16, seed=21)
    table = np.ascontiguousarray(base[rng.integers(0, len(base), size=n)])
    z, feats = m.codec().compress_host(table, recompute_minmax=True, z_dtype=np.float32)
    assert np.array_equal(feats, orc.find_minmax(table))
    idx = np.unique(np.concatenate([np.arange(64), (1 << 21) + np.arange(-64, 64), (1 << 22) + np.arange(-64, 64),
                                    np.arange(n - 64, n), rng.integers(0, n, size=4096)]))
    xn = ((table[idx] - feats[0]) / feats[1]).astype(np.float64)
    close(z[idx], orc.ae_encode(sd, xn))
    y = m.codec().decompress_host(z, features=feats, y_dtype=np.float32)
    close(y[idx], orc.renormalize(orc.ae_decode(sd, z[idx].astype(np.float64)), feats[0], feats[1]))


def test_full_size_table_properties(ae):
    """BASELINE configs[1]: 100M x 24 on one GPU - size-independent properties instead of a full oracle pass:
    shard independence (any row range encodes to the same bits as inside the full pass), sampled rows against
    the oracle, decode(encode(x)) against the oracle forward."""
    m, sd, _ = ae
    codec = m.codec()
    free, _ = torch.cuda.mem_get_info()
    n = 100_000_000 if free > 40e9 else 10_000_000
    g = torch.Generator(device="cuda").manual_seed(20260101)
    x = torch.rand((n, 24), dtype=torch.float32, device="cuda", generator=g)
    z = codec.encode(x)
    for lo, hi in ((0, 1000), (n // 2 + 13, n // 2 + 80 * 1000 + 7), (n - 4321, n)):
        assert torch.equal(codec.encode(x[lo:hi].contiguous()), z[lo:hi])
    idx = torch.randint(0, n, (8192,), device="cuda", generator=g)
    xs = x[idx].cpu().numpy().astype(np.float64)
    close(z[idx].cpu().numpy(), orc.ae_encode(sd, xs))
    y = codec.decode(z)
    close(y[idx].cpu().numpy(), orc.ae_forward(sd, xs))
    mn, mx = engine.colminmax(x)
    assert torch.equal(mn, x.min(0).values) and torch.equal(mx, x.max(0).values)


def test_billion_row_table_in_chunks(ae):
    """BASELINE configs[4] at one GPU (SURVEY 8d: T1B in 8 chunks of 125M rows; the 96 GB table plus its 60 GB latent and
    96 GB reconstruction do not fit 180 GB at once): pass 1 combines the chunks' column min / max into the file's
    features, pass 2 encodes + decodes every chunk with them.  Chunks are regenerated from their seeds, never stored.
    Properties: the combined features equal the min / max of all rows (exact), sampled rows of every chunk match the
    oracle with the GLOBAL features, a row range inside a chunk encodes to the same bits as on its own, and the
    reconstruction of the whole table stays within the model's error everywhere (checksum of per-chunk maxima)."""
    m, sd, _ = ae
    codec = m.codec()
    free, _ = torch.cuda.mem_get_info()
    chunk, n_chunks = (125_000_000, 8) if free > 60e9 else (2_000_000, 4)
    scale = torch.linspace(0.5, 3.0, 24, device="cuda")

    def make(i):
        g = torch.Generator(device="cuda").manual_seed(20260101 + i)
        x = torch.rand((chunk, 24), dtype=torch.float32, device="cuda", generator=g)
        return x.mul_(scale).add_(float(i) * 0.125)  # every chunk has its own range: the features must be global

    mn = torch.full((24,), float("inf"), device="cuda")
    mx = -mn
    for i in range(n_chunks):
        x = make(i)
        cmn, cmx = engine.colminmax(x)
        assert torch.equal(cmn, x.min(0).values) and torch.equal(cmx, x.max(0).values)
        mn, mx = torch.minimum(mn, cmn), torch.maximum(mx, cmx)
        del x
    rg = mx - mn
    feats = [mn.cpu().numpy().astype(np.float64), rg.cpu().numpy().astype(np.float64)]
    worst = []
    for i in range(n_chunks):
        x = make(i)
        z = codec.encode(x, mn, rg)
        g = torch.Generator(device="cuda").manual_seed(99 + i)
        idx = torch.randint(0, chunk, (2048,), device="cuda", generator=g)
        xs = x[idx].cpu().numpy()
        xn = ((xs - mn.cpu().numpy()) / rg.cpu().numpy()).astype(np.float64)  # float32 normalisation, as helper.normalize
        close(z[idx].cpu().numpy(), orc.ae_encode(sd, xn))
        lo = chunk // 3 + 5
        assert torch.equal(codec.encode(x[lo:lo + 70_001].contiguous(), mn, rg), z[lo:lo + 70_001])
        y = codec.decode(z, mn, rg)
        close(y[idx].cpu().numpy(), orc.renormalize(orc.ae_decode(sd, z[idx].cpu().numpy().astype(np.float64)), feats[0], feats[1]))
        worst.append(float((y - x).abs_().max()))
        assert bool(torch.isfinite(y).all())
        del x, y, z
    ref_err = np.abs(orc.renormalize(orc.ae_forward(sd, xn), feats[0], feats[1]) - xs).max()
    assert max(worst) < 50 * max(ref_err, 1e-3)  # no chunk went through different features or a stale buffer


def test_cli_roundtrip_matches_reference_files(golden, tmp_path, monkeypatch):
    """--mode compress / decompress on a workspace whose model.pt was trained by the reference: the files we
    write must match the files the reference wrote (tests/golden/cli_roundtrip.npz)."""
    from baler_b200 import baler
    from baler_b200.modules import helper

    g = golden("cli_roundtrip.npz")
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CMS_workspace", "CMS_project_v1")
    table = synth.cms_table(4096, seed=17)
    path = os.path.join("workspaces", "CMS_workspace", "data", "example_CMS_data.npz")
    np.savez(path, data=table, names=synth.CMS_NAMES)
    out = os.path.join("workspaces", "CMS_workspace", "CMS_project_v1", "output")
    torch.save({k: torch.from_numpy(v) for k, v in sub_sd(g, "sd").items()}, os.path.join(out, "compressed_output", "model.pt"))
    np.save(os.path.join(out, "training", "normalization_features.npy"), g["norm_features"])

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name = 1, 1.6, True, "AE"
        batch_size, custom_norm, extra_compression, separate_model_saving = 512, False, False, False
        save_error_bounded_deltas, convert_to_blocks, type_list = False, False, TYPE_LIST

    baler.perform_compression(out, cfg, False)
    comp = np.load(os.path.join(out, "compressed_output", "compressed.npz"))
    assert comp["data"].dtype == np.float64 and comp["data"].shape == (4096, 15)
    assert list(comp["names"]) == list(synth.CMS_NAMES)
    assert np.array_equal(comp["normalization_features"], g["comp_norm_features"])
    close(comp["data"], g["compressed"])
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    ref = g["decompressed"]
    assert dec.dtype == np.float64 and dec.shape == ref.shape
    fl = [c for c, t in enumerate(TYPE_LIST) if t != "int"]
    it = [c for c, t in enumerate(TYPE_LIST) if t == "int"]
    close(dec[:, fl], ref[:, fl])
    mism = dec[:, it] != ref[:, it]  # truncation is discontinuous (SURVEY F10): counted +-1 budget
    assert np.all(dec[:, it] == np.trunc(dec[:, it]))
    assert mism.mean() <= 1e-3 and np.all(np.abs(dec[:, it] - ref[:, it])[mism] == 1), mism.mean()
    np.save(os.path.join(out, "training", "loss_data.npy"), g["loss_data"])
    baler.print_info(out, type("c", (), {"input_path": path}))


def test_cli_float64_table_with_large_offsets(ae, tmp_path, monkeypatch):
    """a float64 file with an event-counter column (offset 1e9, spread ~1e3) and a shifted column: the reference normalises
    and un-normalises it in float64 (numpy); float32 would keep 64 / 977 of the counter's resolution.  --mode compress /
    decompress must match the oracle's float64 pipeline: the latent to 1e-5, the reconstruction to 1e-5 of each column's
    range (data_processing.F32_OFFSET_LIMIT: host float64 (re)normalisation around the float32 kernels)."""
    from baler_b200 import baler
    from baler_b200.modules import helper

    m, sd, _ = ae
    n = 4096
    table = synth.cms_table(n, seed=29).astype(np.float64)
    table[:, 5] = 1.0e9 + np.arange(n) % 977
    table[:, 11] = -4.0e7 + 0.25 * table[:, 11]
    feats = orc.find_minmax(table)
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CMS_workspace", "CMS_project_v1")
    path = os.path.join("workspaces", "CMS_workspace", "data", "example_CMS_data.npz")
    np.savez(path, data=table, names=synth.CMS_NAMES)
    out = os.path.join("workspaces", "CMS_workspace", "CMS_project_v1", "output")
    torch.save(m.state_dict(), os.path.join(out, "compressed_output", "model.pt"))
    np.save(os.path.join(out, "training", "normalization_features.npy"), feats)

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name = 1, 1.6, True, "AE"
        batch_size, custom_norm, extra_compression, separate_model_saving = 512, False, False, False
        save_error_bounded_deltas, convert_to_blocks = False, False

    baler.perform_compression(out, cfg, False)
    z = np.load(os.path.join(out, "compressed_output", "compressed.npz"))["data"]
    z_ref = orc.compress(sd, table)
    close(z, z_ref)
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    ref = orc.decompress(sd, z_ref, feats)
    assert dec.dtype == np.float64 and dec.shape == ref.shape
    assert (np.abs(dec - ref) / feats[1]).max() <= 1e-5


def test_host_pipeline_streaming_path(ae, monkeypatch):
    """tables that do not fit next to their latent in HBM (BASELINE configs[4]: 1B rows = 96 GB) are read from the host
    twice - once for the column min / max, once for the encode - instead of staying resident between the passes; the
    test hook forces that path on a small table and the result must equal the resident path bit for bit"""
    m, sd, _ = ae
    n = (1 << 20) + 777
    table = synth.cms_table(n, seed=31)
    z_res, f_res = m.codec().compress_host(table, recompute_minmax=True, z_dtype=np.float32)
    monkeypatch.setenv("BALER_B200_NO_RESIDENT", "1")
    z_str, f_str = m.codec().compress_host(table, recompute_minmax=True, z_dtype=np.float32)
    assert np.array_equal(f_res, f_str) and np.array_equal(f_res, orc.find_minmax(table))
    assert np.array_equal(z_res, z_str)
    z64, _ = m.codec().compress_host(table, recompute_minmax=True, z_dtype=np.float64)
    assert z64.dtype == np.float64 and np.array_equal(z64, z_res.astype(np.float64))


def test_error_bounded_deltas_vs_reference(golden, tmp_path, monkeypatch):
    """config.save_error_bounded_deltas: hits, float16 deltas and their re-application against what the reference
    functions produced for the same model and rows (tests/golden/eb_deltas.npz, batches of 256 rows, bound 25 %).
    The reconstruction here differs from the float64 one by ~1e-6, so elements within that distance of the bound may flip:
    counted budget."""
    import gzip
    from baler_b200 import baler
    from baler_b200.modules import helper
    g, ga = golden("eb_deltas.npz"), golden("ae_cms.npz")
    table, bound, bs = g["table"], float(g["bound"]), 256
    ref_hits = {}
    for b in range(2):
        for r, c, d in zip(g["rows%d" % b], g["cols%d" % b], g["deltas%d" % b]):
            ref_hits[(int(r) + bs * b, int(c))] = d
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CMS_workspace", "CMS_project_v1")
    path = os.path.join("workspaces", "CMS_workspace", "data", "example_CMS_data.npz")
    np.savez(path, data=table, names=synth.CMS_NAMES)
    out = os.path.join("workspaces", "CMS_workspace", "CMS_project_v1", "output")
    torch.save({k: torch.from_numpy(v) for k, v in sub_sd(ga, "sd").items()}, os.path.join(out, "compressed_output", "model.pt"))
    feats = orc.find_minmax(table)
    np.save(os.path.join(out, "training", "normalization_features.npy"), feats)

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name = 1, 1.6, True, "AE"
        batch_size, custom_norm, extra_compression, separate_model_saving = bs, False, False, False
        save_error_bounded_deltas, error_bounded_requirement, convert_to_blocks = True, bound, False

    baler.perform_compression(out, cfg, False)
    deltas = np.load(gzip.GzipFile(os.path.join(out, "compressed_output", "compressed_deltas.npz.gz"), "r"), allow_pickle=True)
    index = np.load(gzip.GzipFile(os.path.join(out, "compressed_output", "compressed_batch_index_metadata.npz.gz"), "r"), allow_pickle=True)
    assert list(index[0]) == [0, 1] and len(deltas) == 2  # one entry per batch, as upstream writes them
    got = {}
    for b in range(2):
        rows, cols = index[1][b]
        assert np.all(np.diff(rows * 24 + cols) > 0)  # np.where order: row-major
        for r, c, d in zip(rows, cols, deltas[b]):
            got[(int(r) + bs * b, int(c))] = d
    both = set(got) & set(ref_hits)
    assert len(set(got) ^ set(ref_hits)) <= 0.005 * len(ref_hits), (len(got), len(ref_hits))
    off = [k for k in both if got[k] != ref_hits[k]]
    assert len(off) <= 0.01 * len(both)
    # the delta is float16(y) - float16(x) with x, y in [0, 1]: a reconstruction that differs in the 7th digit can round
    # to the neighbouring float16, which moves the delta by one float16 ulp of y
    assert all(abs(float(got[k]) - float(ref_hits[k])) <= 2.0 ** -10 for k in off)
    # decompression applies the deltas: compare with the reference's corrected reconstruction, un-normalised
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    fixed = np.concatenate([g["fixed0"], g["fixed1"]])
    ref = orc.renormalize(fixed, feats[0], feats[1])
    same = np.ones(dec.shape, dtype=bool)
    for r, c in set(got) ^ set(ref_hits):
        same[r, c] = False
    scale = np.abs(ref).max(axis=0)
    assert (np.abs(dec - ref)[same] <= 1e-3 * np.broadcast_to(scale, dec.shape)[same]).all()  # float16 deltas: 2^-11 relative


def test_bench_dump_outputs(ae, tmp_path):
    """bench.py --dump-outputs: the features of the last timed step and its latent and reconstruction at the sampled rows,
    the same whatever --steps (which sets the number of timed steps), equal to the oracle's compress / decompress"""
    import json
    import subprocess
    import sys

    sd = ae[1]
    n = 300_000  # more rows than the dump samples
    runs = []
    for steps in (1, 3):
        out = tmp_path / ("steps%d" % steps)
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
               "--rows", str(n), "--no-sweep", "--no-cpu", "--no-modes", "--no-e2e", "--no-train", "--no-cfd",
               "--dump-outputs", str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip().splitlines()[-1])
        assert d["steps"] == steps and d["gpu_launches"] == 3 * steps
        files = {p.name[:-4]: np.load(p) for p in out.iterdir()}
        assert sorted(files) == ["features", "latent", "reconstruction", "rows"]
        assert all(a.dtype in (np.float32, np.float64) for a in files.values())
        assert sum(a.nbytes for a in files.values()) <= 64 << 20
        runs.append(files)
    for k in runs[0]:
        assert np.array_equal(runs[0][k], runs[1][k]), k
    got = runs[0]
    rows = got["rows"].astype(np.int64)
    assert len(rows) < n and np.all(np.diff(rows) > 0)
    table = synth.cms_table_device(n, seed=synth.CMS_SEED).cpu().numpy()
    feats = orc.find_minmax(table)
    assert np.array_equal(got["features"], feats)
    z_ref = orc.compress(sd, table)[rows]
    close(got["latent"], z_ref)
    close(got["reconstruction"], orc.decompress(sd, z_ref, feats))
