"""precision "fp64" training: the float64 step against the reference's float64 training.

Bounds are those tests/test_oracle_golden.py uses for float64 against float64 (or wider where noted): the float64
arithmetic of the reference in another summation order agrees to ~1e-14."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_max, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import engine, synth
from baler_b200.modules import models

pytestmark = pytest.mark.gpu
NAMES = models.AE.names
TYPE_LIST = ["float64"] * 12 + ["int"] * 7 + ["float64"] * 3 + ["int"] * 2


def flat(sd_like):
    return np.concatenate([np.concatenate([np.asarray(sd_like[n + ".weight"]).ravel(), np.asarray(sd_like[n + ".bias"]).ravel()])
                           for n in NAMES]).astype(np.float64)


def split(v):
    """flat trainer layout -> {name: array} (shapes of the AE(24, 15) state dict)"""
    out, off = {}, 0
    shapes = orc.init_ae_shapes(24, 15)
    for n in NAMES:
        for part, shape in ((".weight", shapes[n]), (".bias", (shapes[n][0],))):
            size = int(np.prod(shape))
            out[n + part] = np.asarray(v[off:off + size]).reshape(shape)
            off += size
    return out


def trainer(sd, max_batch=512):
    tr = engine.Trainer([sd[n + ".weight"] for n in NAMES], [sd[n + ".bias"] for n in NAMES], 24, 15, max_batch)
    tr.set_precision("fp64")
    assert tr.precision == "fp64"
    return tr


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("tag,l1", [("mse", False), ("l1", True)])
def test_step_loss_grads_adam(golden, tag, l1):
    g = golden("ae_train.npz")
    sd0 = sub_sd(g, "sd0")
    x = cuda(g["x_norm"])
    tr = trainer(sd0)
    h = engine.make_hyper(lr=1e-3, reg_param=0.001, l1=l1)
    ref_losses = g["losses_" + tag]
    losses = []
    for step in range(3):
        tr.loss_accum.zero_()
        tr.step(x[step * 512:(step + 1) * 512].contiguous(), h)
        losses.append(tr.loss_accum.item())
        if step == 0:
            gv = tr.grads_view().cpu().numpy()
            assert gv.dtype == np.float64
            assert abs(gv[-1] - ref_losses[0]) <= 1e-12 * ref_losses[0], (gv[-1], ref_losses[0])
            got, ref = split(gv[:-1]), sub_sd(g, "g_" + tag)
            for k in ref:
                assert rel_max(got[k], ref[k]) <= 1e-11, (k, rel_max(got[k], ref[k]))
        if step in (0, 2):
            p = split(tr.params_view().cpu().numpy())
            ref = sub_sd(g, "sd%d_%s" % (step + 1, tag))
            for k in ref:  # the UPDATE: Adam's g / (|g| + eps)
                assert rel_max(p[k] - sd0[k], ref[k] - sd0[k]) <= 1e-8, (step, k, rel_max(p[k] - sd0[k], ref[k] - sd0[k]))
    np.testing.assert_allclose(losses, ref_losses, rtol=1e-11)
    w, b = tr.get_params()
    assert w[0].dtype == np.float64 and w[0].shape == (200, 24) and b[7].shape == (24,)
    p = split(tr.params_view().cpu().numpy())
    assert all(np.array_equal(w[i], p[n + ".weight"]) and np.array_equal(b[i], p[n + ".bias"]) for i, n in enumerate(NAMES))


@pytest.mark.parametrize("rows", [1, 7, 63, 65, 100, 448])
def test_ragged_batches_vs_oracle(golden, rows):
    g = golden("ae_train.npz")
    sd0 = sub_sd(g, "sd0")
    x = g["x_norm"][:rows]
    loss, _, _, grads = orc.ae_loss_and_grads(sd0, x.astype(np.float64))
    tr = trainer(sd0)
    tr.step(cuda(x), engine.make_hyper(), phase=1)
    got = tr.grads_view().cpu().numpy()
    assert abs(got[-1] - loss) <= 1e-12 * loss, (got[-1], loss)
    if rows == 100:
        assert abs(got[-1] - float(g["loss_ragged100"])) <= 1e-12 * loss
    ref = flat(grads)
    assert rel_max(got[:-1], ref) <= 1e-11, rel_max(got[:-1], ref)
    assert np.array_equal(tr.params_view().cpu().numpy(), flat(sd0))  # phase 1 leaves the float64 master alone


def test_float32_and_float64_input_give_the_same_bits(golden):
    g = golden("ae_train.npz")
    sd0 = sub_sd(g, "sd0")
    x32 = cuda(g["x_norm"][:512])
    x64 = x32.double()
    h = engine.make_hyper(lr=1e-3, reg_param=0.001, l1=True)
    a, b = trainer(sd0), trainer(sd0)
    for _ in range(2):
        a.step(x32, h)
        b.step(x64, h)
    assert torch.equal(a.grads_view(), b.grads_view()) and torch.equal(a.params_view(), b.params_view())
    assert a.loss_accum.item() == b.loss_accum.item()
    assert a.validate(x32, 512) == b.validate(x64, 512)
    assert a.epoch(x32, 128, h) == b.epoch(x64, 128, h)
    assert torch.equal(a.params_view(), b.params_view())


def test_phases_and_reproducibility(golden):
    g = golden("ae_train.npz")
    sd0 = sub_sd(g, "sd0")
    x = cuda(g["x_norm"][:512])
    h = engine.make_hyper()
    a, b = trainer(sd0), trainer(sd0)
    a.step(x, h, phase=0)
    b.step(x, h, phase=1)
    b.step(x, h, phase=2)
    assert torch.equal(a.params_view(), b.params_view()) and a.loss_accum.item() == b.loss_accum.item()
    # two half batches, gradients summed (what the SUM all-reduce of two ranks leaves) == one full batch
    c, d = trainer(sd0), trainer(sd0)
    h2 = engine.make_hyper(world_size=2)
    c.step(x[:256].contiguous(), h2, phase=1)
    d.step(x[256:].contiguous(), h2, phase=1)
    summed = (c.grads_view() + d.grads_view()).cpu().numpy()
    full = b.grads_view().cpu().numpy()
    assert rel_max(summed, full) <= 1e-13, rel_max(summed, full)
    # two identical runs are bitwise equal
    runs = []
    for _ in range(2):
        t = trainer(sd0)
        t.epoch(cuda(g["x_norm"]), 512, engine.make_hyper(lr=1e-3, reg_param=0.001, l1=True))
        runs.append(t.params_view().clone())
    assert torch.equal(runs[0], runs[1])


def test_fit_curve_validate_and_activations(golden):
    g, g0 = golden("ae_fit.npz"), golden("ae_train.npz")
    sd0 = sub_sd(g0, "sd0")
    xn = orc.normalize(synth.cms_table(4096, seed=11))
    x = cuda(xn)
    tr = trainer(sd0)
    h = engine.make_hyper(lr=1e-3)
    losses = [tr.epoch(x, 512, h) for _ in range(3)]
    np.testing.assert_allclose(losses, g["loss_data"][0], rtol=1e-11)
    w, b = tr.get_params()
    sd = {n + ".weight": w[i] for i, n in enumerate(NAMES)}
    sd.update({n + ".bias": b[i] for i, n in enumerate(NAMES)})
    ref = sub_sd(g, "sd_final")
    worst = max(rel_max(sd[k], ref[k]) for k in ref)
    assert worst <= 1e-10, worst
    x64 = xn.astype(np.float64)
    val = tr.validate(x, 512)
    ref_val = np.mean([orc.mse_sum_loss(orc.ae_forward(sd, x64[i:i + 512]), x64[i:i + 512]) for i in range(0, 4096, 512)])
    assert abs(val - ref_val) <= 1e-12 * ref_val, (val, ref_val)
    # activation means of the last forward pass (validate's last batch) from the oracle's float64 forward
    h_ = x64[3584:]
    means = []
    for i, n in enumerate(NAMES[:7]):
        h_ = orc.linear(h_, sd[n + ".weight"], sd[n + ".bias"])
        if i != 3:
            h_ = orc.leaky_relu(h_)
            means.append(h_.mean(axis=0))
    act = tr.activation_means()
    for i, m in enumerate(means):
        assert np.isnan(act[i, len(m):]).all()
        assert rel_max(act[i, :len(m)], m) <= 1e-12, (i, rel_max(act[i, :len(m)], m))
    print("ae_fit: loss rel %.2e, weights rel_max %.2e, validate rel %.2e, activation means rel_max %.2e"
          % (np.max(np.abs(np.array(losses) / g["loss_data"][0] - 1)), worst, abs(val / ref_val - 1),
             max(rel_max(act[i, :len(m)], m) for i, m in enumerate(means))))


def _cfg(helper, path, **extra):
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
    return cfg


def _project(tmp_path, monkeypatch, table):
    from baler_b200.modules import helper
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CMS_workspace", "CMS_project_v1")
    path = os.path.join("workspaces", "CMS_workspace", "data", "example_CMS_data.npz")
    np.savez(path, data=table, names=synth.CMS_NAMES)
    return os.path.join("workspaces", "CMS_workspace", "CMS_project_v1", "output"), path


def test_train_compress_decompress_reproduce_the_reference_files(golden, tmp_path, monkeypatch):
    """--mode train, compress, decompress with precision "fp64" from torch.manual_seed(0) give the files the reference's
    CLI wrote for the same workspace (tests/golden/cli_roundtrip.npz)"""
    from baler_b200 import baler
    from baler_b200.modules import helper
    g = golden("cli_roundtrip.npz")
    out, path = _project(tmp_path, monkeypatch, synth.cms_table(4096, seed=17))
    cfg = _cfg(helper, path, type_list=TYPE_LIST)
    torch.manual_seed(0)
    baler.perform_training(out, cfg, False)
    loss = np.load(os.path.join(out, "training", "loss_data.npy"))
    np.testing.assert_allclose(loss, g["loss_data"], rtol=1e-11)
    feats = np.load(os.path.join(out, "training", "normalization_features.npy"))
    assert feats.dtype == g["norm_features"].dtype and np.array_equal(feats, g["norm_features"])
    sd = torch.load(os.path.join(out, "compressed_output", "model.pt"))
    ref = sub_sd(g, "sd")
    assert list(sd.keys()) == list(ref.keys())
    for k in ref:
        assert sd[k].dtype == torch.float64 and rel_max(sd[k].numpy(), ref[k]) <= 1e-10, (k, rel_max(sd[k].numpy(), ref[k]))
    act, ref_act = np.load(os.path.join(out, "training", "activations.npy")), g["activations"]
    assert act.shape == ref_act.shape and np.array_equal(np.isnan(act), np.isnan(ref_act))
    assert rel_max(np.nan_to_num(act), np.nan_to_num(ref_act)) <= 1e-10
    baler.perform_compression(out, cfg, False)
    z = np.load(os.path.join(out, "compressed_output", "compressed.npz"))["data"]
    assert z.dtype == np.float64 and rel_max(z, g["compressed"]) <= 1e-10, rel_max(z, g["compressed"])
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    ref_dec = g["decompressed"]
    fl = [c for c, t in enumerate(TYPE_LIST) if t != "int"]
    it = [c for c, t in enumerate(TYPE_LIST) if t == "int"]
    assert rel_max(dec[:, fl], ref_dec[:, fl]) <= 1e-10
    mism = dec[:, it] != ref_dec[:, it]  # truncation is discontinuous: isolated +-1 (as test_cli_roundtrip_golden)
    assert mism.mean() < 1e-4 and np.all(np.abs(dec[:, it] - ref_dec[:, it])[mism] == 1)
    print("cli_roundtrip: loss rel %.2e, model.pt rel_max %.2e, activations rel_max %.2e, latent rel_max %.2e, "
          "float columns rel_max %.2e, integer columns differing %d"
          % (np.max(np.abs(loss / g["loss_data"] - 1)), max(rel_max(sd[k].numpy(), ref[k]) for k in ref),
             rel_max(np.nan_to_num(act), np.nan_to_num(ref_act)), rel_max(z, g["compressed"]),
             rel_max(dec[:, fl], ref_dec[:, fl]), int(mism.sum())))


def test_float64_file_with_large_offsets_trains_in_float64(tmp_path, monkeypatch):
    """a float64 file with a 1e9 event counter: normalised in float64 on the device (bit-equal to numpy, the host float64
    normalisation unused), trained as a float64 table; the loss curve is the oracle's float64 training"""
    from baler_b200 import baler
    from baler_b200.modules import data_processing, helper, training

    def no_host_path(*a, **k):
        raise AssertionError("host float64 normalisation used")
    monkeypatch.setattr(data_processing, "normalize_float64_host", no_host_path)
    n = 4096
    table = synth.cms_table(n, seed=29).astype(np.float64)
    table[:, 5] = 1.0e9 + np.arange(n) % 977
    table[:, 11] = -4.0e7 + 0.25 * table[:, 11]
    out, path = _project(tmp_path, monkeypatch, table)
    cfg = _cfg(helper, path)
    xn = orc.normalize(table)
    tr_set, _, feats, _ = helper.process(path, False, 0, True, None, False, precision="fp64")
    assert tr_set.dtype == np.float64 and tr_set.tobytes() == xn.tobytes()
    assert feats.dtype == np.float64 and feats.tobytes() == orc.find_minmax(table).tobytes()
    seen = []
    to_dev = training._to_device_table
    monkeypatch.setattr(training, "_to_device_table", lambda d, c: seen.append(to_dev(d, c)) or seen[-1])
    torch.manual_seed(0)
    sd_init = {k: v.numpy().copy() for k, v in models.AE(24, 15).state_dict().items()}
    torch.manual_seed(0)
    baler.perform_training(out, cfg, False)
    assert seen and all(t.dtype == torch.float64 for t in seen)
    assert np.load(os.path.join(out, "training", "normalization_features.npy")).tobytes() == feats.tobytes()
    _, ref_loss = orc.train(sd_init, xn, 512, 2, lr=1e-3)
    np.testing.assert_allclose(np.load(os.path.join(out, "training", "loss_data.npy")), ref_loss, rtol=1e-11)


def test_float64_kernels_do_not_spill():
    """-Xptxas -v on the float64 training kernels: no local-memory spills"""
    from baler_b200 import build
    src = os.path.join(ROOT, "baler_b200", "csrc", "bb_train_f64.cu")
    r = subprocess.run([build.NVCC] + build.FLAGS + ["-Xptxas", "-v", "-c", src, "-o", os.devnull],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    props = [line for line in r.stderr.splitlines() if "spill stores" in line]
    assert len(props) >= 3 and all("0 bytes spill stores, 0 bytes spill loads" in line for line in props), props


_CFG = """
def set_config(c):
    c.input_path = {path!r}
    c.data_dimension, c.compression_ratio, c.apply_normalization, c.model_name = 1, 1.6, True, "AE"
    c.epochs, c.lr, c.batch_size, c.early_stopping, c.lr_scheduler = 2, 0.001, 512, True, True
    c.early_stopping_patience, c.min_delta, c.lr_scheduler_patience, c.custom_norm = 100, 0, 50, False
    c.reg_param, c.RHO, c.test_size, c.extra_compression = 0.001, 0.05, 0, False
    c.intermittent_model_saving, c.intermittent_saving_patience = False, 100
    c.l1, c.activation_extraction, c.deterministic_algorithm = True, False, False
    c.convert_to_blocks, c.separate_model_saving, c.save_error_bounded_deltas = False, False, False
    c.precision = "fp64"
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_torchrun_two_ranks_train_what_one_process_trains(tmp_path):
    """2-rank torchrun --mode train with "fp64" (phase 1, NCCL SUM of the float64 gradient + loss, phase 2) against one
    process on the same global batches"""
    table = synth.cms_table(6000, seed=47)
    res = {}
    for world in (1, 2):
        wd = tmp_path / ("w%d" % world)
        proj = wd / "workspaces" / "WS" / "P"
        for d in ("config", "output/compressed_output", "output/decompressed_output", "output/training"):
            os.makedirs(proj / d)
        os.makedirs(wd / "workspaces" / "WS" / "data")
        data = str(wd / "workspaces" / "WS" / "data" / "d.npz")
        np.savez(data, data=table, names=synth.CMS_NAMES)
        (proj / "config" / "P_config.py").write_text(_CFG.format(path=data))
        launch = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port",
                  str(_free_port())] if world == 2 else [sys.executable]
        r = subprocess.run(launch + ["-m", "baler_b200", "--project", "WS", "P", "--mode", "train"], cwd=wd,
                           env=dict(os.environ, PYTHONPATH=ROOT, BALER_B200_SEED="5"), capture_output=True, text=True,
                           timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        res[world] = (np.load(proj / "output" / "training" / "loss_data.npy"),
                      torch.load(proj / "output" / "compressed_output" / "model.pt"))
    np.testing.assert_allclose(res[2][0], res[1][0], rtol=1e-12)
    for k, v in res[1][1].items():
        assert rel_max(res[2][1][k].numpy(), v.numpy()) <= 1e-11, k


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]
