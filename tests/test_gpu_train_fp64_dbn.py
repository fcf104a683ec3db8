"""precision "fp64" training of AE_Dropout_BN: the float64 cooperative step against the reference's fixture and against
the torch twin of the reference's training loop (tests/dbn_reference.py), with the dropout masks drawn on the device
from torch's generator (dropout_stream = "torch")."""
import json
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_max, sub_sd
from dbn_reference import DROPOUT_P, fit, validate, twin_from_state
from oracle import baler_oracle as orc
from baler_b200 import _lib, engine, synth
from baler_b200.modules import models, training

pytestmark = pytest.mark.gpu
LIN = models.AE_Dropout_BN.enc_names + models.AE_Dropout_BN.dec_names
BN = models.AE_Dropout_BN.bn_names
WIDTHS = (200, 100, 50, 15)
# A run of the reference's own training is sensitive to rounding: scaling one weight matrix of the twin by (1 + 1e-15)
# moves its 3-epoch loss curve by ~4e-10, its validate losses by ~2e-8 and its tensors by up to ~5e-7 of their max|.|
# (most on biases feeding a LeakyReLU + BatchNorm or a BatchNorm, whose gradient is near or below Adam's eps = 1e-8, so
# m / (sqrt(v) + eps) amplifies its rounding, and on the running means that track them).  Another summation order
# cannot be closer than that, so every quantity is gated at SPREAD x the twin's own spread under that perturbation
# (at least FLOOR).
SPREAD, FLOOR = 100.0, 1e-12


def record(name, **values):
    """measured errors as one JSON line on stdout (pytest -rA shows it with the test's result)"""
    print(json.dumps({"test": name, **values}, default=float))


def dbn_trainer(sd, max_batch=512, precision="fp64"):
    bn = {k: [sd[b + "." + k] for b in BN] for k in ("weight", "bias", "running_mean", "running_var")}
    bn["num_batches_tracked"] = [int(sd[b + ".num_batches_tracked"]) for b in BN]
    tr = engine.Trainer([sd[n + ".weight"] for n in LIN], [sd[n + ".bias"] for n in LIN], 24, 15, max_batch, bn=bn)
    tr.set_precision(precision)
    assert tr.precision == precision
    return tr


def flat(sd_like):
    lin = [np.concatenate([np.asarray(sd_like[n + ".weight"]).ravel(), np.asarray(sd_like[n + ".bias"]).ravel()]) for n in LIN]
    bn = [np.concatenate([np.asarray(sd_like[b + ".weight"]).ravel(), np.asarray(sd_like[b + ".bias"]).ravel()]) for b in BN]
    return np.concatenate(lin + bn).astype(np.float64)


def state_of(tr):
    """the trainer's parameters and BatchNorm buffers as a state dict"""
    w, b = tr.get_params()
    sd = {}
    for i, n in enumerate(LIN):
        sd[n + ".weight"], sd[n + ".bias"] = w[i], b[i]
    bn = tr.get_bn()
    for i, n in enumerate(BN):
        for k in ("weight", "bias", "running_mean", "running_var"):
            sd[n + "." + k] = bn[k][i]
        sd[n + ".num_batches_tracked"] = np.int64(bn["num_batches_tracked"][i])
    return sd


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def masks_of(g):
    return [cuda(g["mask%d" % i].astype(np.uint8)) for i in range(4)]


def test_golden_step_with_injected_masks(golden):
    g = golden("ae_dbn.npz")
    sd0, sd1, gref = sub_sd(g, "sd0"), sub_sd(g, "sd1"), sub_sd(g, "g")
    tr = dbn_trainer(sd0)
    tr.set_dropout(masks=masks_of(g))
    tr.step(cuda(g["x_norm"][:512]), engine.make_hyper(lr=1e-3))
    loss, ref_loss = tr.loss_accum.item(), float(g["loss_train"])
    gv = tr.grads_view().cpu().numpy()
    assert gv.dtype == np.float64 and abs(gv[-1] - ref_loss) <= 1e-12 * ref_loss and abs(loss - ref_loss) <= 1e-12 * ref_loss
    ref = flat(gref)
    gscale = np.abs(ref).max()
    gerr = np.abs(gv[:-1] - ref).max() / gscale
    assert gerr <= 1e-11, gerr
    sd = state_of(tr)
    serr = max(rel_max(sd[b + "." + k], sd1[b + "." + k]) for b in BN for k in ("running_mean", "running_var"))
    assert serr <= 1e-12, serr
    assert all(int(sd[b + ".num_batches_tracked"]) == int(sd1[b + ".num_batches_tracked"]) for b in BN)
    p, p1 = tr.params_view().cpu().numpy(), flat(sd1)
    live = np.abs(ref) > 1e-6 * gscale  # Adam moves a zero-gradient parameter by up to lr on rounding noise
    assert np.abs(p - p1)[live].max() <= 1e-9 and np.abs(p - p1).max() <= 1.001e-3
    rm, rv = tr.bn_running_views()
    assert rm.dtype == torch.float64 and rm.numel() == 50 + 100 + 200 + 24
    record("golden_step", loss_rel=abs(loss / ref_loss - 1), grad_rel=gerr, running_rel=serr,
           adam_live_abs=float(np.abs(p - p1)[live].max()))


def test_device_stream_draws_the_fixture_masks(golden):
    """after manual_seed(5) the device draws mask0..3: the step is bit-identical to the one with the fixture's masks"""
    g = golden("ae_dbn.npz")
    sd0 = sub_sd(g, "sd0")
    x = cuda(g["x_norm"][:512])
    h = engine.make_hyper(lr=1e-3)
    a, b = dbn_trainer(sd0), dbn_trainer(sd0)
    a.set_dropout(masks=masks_of(g))
    torch.manual_seed(5)
    b.set_dropout_torch()
    for t in (a, b):
        t.step(x, h, phase=1)
    assert torch.equal(a.grads_view(), b.grads_view())
    b.write_back_dropout_torch()
    got = torch.rand(8)
    torch.manual_seed(5)
    for w, p in zip(WIDTHS, DROPOUT_P):
        torch.empty(512, w, dtype=torch.float64).bernoulli_(1 - p)
    assert torch.equal(got, torch.rand(8))


@pytest.mark.parametrize("n_rows,batch", [(1100, 512), (1531, 100)])
def test_device_stream_over_an_epoch_equals_cpu_bernoulli(golden, n_rows, batch):
    """an epoch with a ragged last batch: the torch stream gives what injected CPU bernoulli_ masks give, bit for bit, and
    leaves the host generator where the CPU replay leaves it"""
    sd0 = sub_sd(golden("ae_dbn.npz"), "sd0")
    x = cuda(orc.normalize(synth.cms_table(n_rows, seed=41)))
    h = engine.make_hyper(lr=1e-3)
    a, b = dbn_trainer(sd0), dbn_trainer(sd0)
    torch.manual_seed(123)
    torch.rand(5)
    start = torch.get_rng_state()
    a.set_dropout_torch()
    la = a.epoch(x, batch, h)
    a.write_back_dropout_torch()
    after = torch.rand(8)
    torch.set_rng_state(start)
    lb, kept = 0.0, []
    for r0 in range(0, n_rows, batch):
        rows = min(batch, n_rows - r0)
        m = [torch.empty(rows, w, dtype=torch.float64).bernoulli_(1 - p).to(torch.uint8).cuda() for w, p in zip(WIDTHS, DROPOUT_P)]
        kept.append(m)
        b.set_dropout(masks=m)
        b.loss_accum.zero_()
        b.step(x[r0:r0 + rows].contiguous(), h)
        lb += b.loss_accum.item()
    assert torch.equal(torch.rand(8), after)
    assert torch.equal(a.params_view(), b.params_view())
    assert la == lb / len(kept)


def test_philox_masks_are_the_fp32_kernels(golden):
    g = golden("ae_dbn.npz")
    sd0 = sub_sd(g, "sd0")
    x = cuda(g["x_norm"][:512])
    out = {}
    for prec in ("fp32", "fp64"):
        tr = dbn_trainer(sd0, precision=prec)
        tr.set_dropout(seed=4321)
        tr.step(x, engine.make_hyper(lr=1e-3), phase=1)
        out[prec] = tr.grads_view().cpu().numpy().astype(np.float64)
    gscale = np.abs(out["fp64"][:-1]).max()
    assert np.abs(out["fp32"] - out["fp64"])[:-1].max() <= 1e-5 * gscale
    assert abs(out["fp32"][-1] - out["fp64"][-1]) <= 1e-5 * out["fp64"][-1]


def test_float32_and_float64_input_give_the_same_bits_and_runs_repeat(golden):
    sd0 = sub_sd(golden("ae_dbn.npz"), "sd0")
    x32 = cuda(orc.normalize(synth.cms_table(2048, seed=43)))
    h = engine.make_hyper(lr=1e-3)
    runs = []
    for x in (x32, x32.double(), x32):
        t = dbn_trainer(sd0)
        t.set_dropout(seed=9)
        t.epoch(x, 512, h)
        runs.append((t.params_view().clone(), t.bn_running_views()[1].clone(), t.validate(x, 512)))
    for r in runs[1:]:
        assert torch.equal(r[0], runs[0][0])
        assert torch.equal(r[1], runs[0][1])
        assert r[2] == runs[0][2]


def test_resident_limit(golden):
    sd0 = sub_sd(golden("ae_dbn.npz"), "sd0")
    h = engine.make_hyper(lr=1e-3)
    limit = 4 * torch.cuda.get_device_properties(0).multi_processor_count
    assert limit == training.fp64_dbn_max_batch()
    t = dbn_trainer(sd0, max_batch=limit + 1)
    t.set_dropout(seed=1)
    xl = cuda(orc.normalize(synth.cms_table(limit + 1, seed=44)))
    t.step(xl[:limit].contiguous(), h, phase=1)
    assert np.isfinite(t.grads_view().cpu().numpy()).all()
    with pytest.raises(_lib.BalerB200Error, match="bb_trainer_step"):
        t.step(xl, h, phase=1)


def _twin_fit(sd0, x64, batch, epochs, scale=1.0):
    sd = dict(sd0)
    sd["enc_nn.0.weight"] = sd0["enc_nn.0.weight"] * scale
    twin = twin_from_state(sd)
    opt = torch.optim.Adam(twin.parameters(), lr=1e-3)
    torch.manual_seed(7)
    return twin, [(fit(twin, opt, x64, batch), validate(twin, x64, batch)) for _ in range(epochs)]


def _spread(a, b):
    """per-entry relative difference of two twin runs: loss curves, then every state tensor"""
    (ta, la), (tb, lb) = a, b
    out = {"loss": [abs(y[0] / x[0] - 1) for x, y in zip(la, lb)], "val": [abs(y[1] / x[1] - 1) for x, y in zip(la, lb)]}
    sa, sb = ta.state_dict(), tb.state_dict()
    out.update({k: rel_max(sb[k].numpy(), sa[k].numpy()) for k in sa if not k.endswith("num_batches_tracked")})
    return out


def _twin_run(sd0, xn, batch, epochs):
    """the twin from sd0 and the trainer from sd0 through the same seeding: (twin, twin losses, trainer, trainer losses,
    the twin's own spread under a 1e-15 perturbation)"""
    x64 = torch.from_numpy(xn.astype(np.float64))
    twin, ref = _twin_fit(sd0, x64, batch, epochs)
    spread = _spread((twin, ref), _twin_fit(sd0, x64, batch, epochs, 1.0 + 1e-15))
    tr = dbn_trainer(sd0, max_batch=batch)
    x = cuda(xn)
    torch.manual_seed(7)
    got = []
    for _ in range(epochs):
        training.consume_loader_seed(xn.shape[0], batch)
        tr.set_dropout_torch()
        loss = tr.epoch(x, batch, engine.make_hyper(lr=1e-3))
        tr.write_back_dropout_torch()
        training.consume_loader_seed(xn.shape[0], batch)
        got.append((loss, tr.validate(x, batch)))
    return twin, ref, tr, got, spread


def _compare_states(sd, ref, spread, name):
    """every tensor within SPREAD x the twin's own spread of its max|.|; returns the errors"""
    errs = {}
    for k, v in ref.items():
        v = v.numpy() if torch.is_tensor(v) else v
        if k.endswith("num_batches_tracked"):
            assert int(sd[k]) == int(v), k
            continue
        errs[k] = rel_max(sd[k], v)
    record(name, errs=errs, spread={k: spread[k] for k in errs})
    bad = {k: (e, spread[k]) for k, e in errs.items() if e > max(SPREAD * spread[k], FLOOR)}
    assert not bad, bad
    return errs


def _check_curve(got, ref, spread, name):
    rel = [abs(g_ / r - 1) for g_, r in zip(got, ref)]
    record(name, rel=rel, spread=spread)
    assert all(e <= max(SPREAD * s, FLOOR) for e, s in zip(rel, spread)), (rel, spread)


@pytest.mark.parametrize("batch", [512, 500])
def test_three_epochs_against_the_torch_twin(golden, batch):
    sd0 = sub_sd(golden("ae_dbn.npz"), "sd0")
    xn = orc.normalize(synth.cms_table(4096, seed=47))
    twin, ref, tr, got, spread = _twin_run(sd0, xn, batch, 3)
    _check_curve([g_[0] for g_ in got], [r[0] for r in ref], spread["loss"], "twin_loss_%d" % batch)
    _check_curve([g_[1] for g_ in got], [r[1] for r in ref], spread["val"], "twin_validate_%d" % batch)
    _compare_states(state_of(tr), twin.state_dict(), spread, "twin_state_%d" % batch)


def test_cli_train_compress_decompress_against_the_twin(golden, tmp_path, monkeypatch):
    """--mode train / compress / decompress of AE_Dropout_BN with precision "fp64" and dropout_stream "torch" from
    manual_seed(0) against the twin driven through the same seeding"""
    from baler_b200 import baler
    from baler_b200.modules import helper
    from test_gpu_train_fp64 import TYPE_LIST, _cfg, _project
    table = synth.cms_table(3000, seed=17)
    out, path = _project(tmp_path, monkeypatch, table)
    cfg = _cfg(helper, path, model_name="AE_Dropout_BN", dropout_stream="torch", type_list=TYPE_LIST, l1=False,
               test_size=0.2, activation_extraction=False)
    # the twin: the same model initialisation (the CLI builds the model after the same seed), the same split
    # the twin starts from the model the CLI builds after manual_seed(0) and from the generator state that leaves
    torch.manual_seed(0)
    sd_init = {k: v.numpy().copy() for k, v in models.AE_Dropout_BN(24, 15).state_dict().items()}
    after_init = torch.get_rng_state()
    twin = twin_from_state(sd_init)
    torch.set_rng_state(after_init)
    tr_set, te_set, _, _ = helper.process(path, False, 0.2, True, None, False, precision="fp64")
    opt = torch.optim.Adam(twin.parameters(), lr=1e-3)
    xt, xv = torch.from_numpy(np.asarray(tr_set, np.float64)), torch.from_numpy(np.asarray(te_set, np.float64))

    def twin_cli(m, o):
        losses = [[], []]
        for _ in range(cfg.epochs):
            losses[0].append(fit(m, o, xt, 512))
            losses[1].append(validate(m, xv, 512))
        return losses
    ref_loss = twin_cli(twin, opt)
    sd_p = dict(sd_init)
    sd_p["enc_nn.0.weight"] = sd_init["enc_nn.0.weight"] * (1.0 + 1e-15)
    twin_p = twin_from_state(sd_p)
    torch.set_rng_state(after_init)
    ref_p = twin_cli(twin_p, torch.optim.Adam(twin_p.parameters(), lr=1e-3))
    spread = {"loss": [abs(b / a - 1) for a, b in zip(ref_loss[0], ref_p[0])],
              "val": [abs(b / a - 1) for a, b in zip(ref_loss[1], ref_p[1])]}
    spread.update({k: rel_max(twin_p.state_dict()[k].numpy(), v.numpy()) for k, v in twin.state_dict().items()
                   if not k.endswith("num_batches_tracked")})
    torch.manual_seed(0)
    baler.perform_training(out, cfg, False)
    loss = np.load(os.path.join(out, "training", "loss_data.npy"))
    _check_curve(loss[0], ref_loss[0], spread["loss"], "cli_loss")
    _check_curve(loss[1], ref_loss[1], spread["val"], "cli_validate")
    sd = torch.load(os.path.join(out, "compressed_output", "model.pt"))
    ref = twin.state_dict()
    assert set(sd.keys()) == set(ref.keys())
    _compare_states({k: v.numpy() for k, v in sd.items()}, ref, spread, "cli_model")
    baler.perform_compression(out, cfg, False)
    z = np.load(os.path.join(out, "compressed_output", "compressed.npz"))["data"]
    feats = orc.find_minmax(table)

    @torch.no_grad()
    def codec(m):
        m.eval()
        zm = m.enc_nn(torch.from_numpy(orc.normalize(table).astype(np.float64)))
        return zm.numpy(), m.dec_nn(zm).numpy() * feats[1].astype(np.float64) + feats[0].astype(np.float64)
    zr, yr = codec(twin)
    zp, yp = codec(twin_p)
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    fl = [c for c, t in enumerate(TYPE_LIST) if t != "int"]
    it = [c for c, t in enumerate(TYPE_LIST) if t == "int"]
    z_rel, y_rel = rel_max(z, zr), rel_max(dec[:, fl], yr[:, fl])
    z_spread, y_spread = rel_max(zp, zr), rel_max(yp[:, fl], yr[:, fl])
    mism = dec[:, it] != np.trunc(yr[:, it])
    record("cli", latent_rel=z_rel, recon_rel=y_rel, latent_spread=z_spread, recon_spread=y_spread,
           int_differing=int(mism.sum()))
    assert z_rel <= max(SPREAD * z_spread, FLOOR) and y_rel <= max(SPREAD * y_spread, FLOOR), (z_rel, y_rel, z_spread, y_spread)
    assert mism.mean() < 1e-4 and np.all(np.abs(dec[:, it] - np.trunc(yr[:, it]))[mism] == 1)


def test_dbn_kernels_do_not_spill():
    from baler_b200 import build
    for name in ("bb_train_f64.cu", "bb_dropout_mt.cu"):
        src = os.path.join(ROOT, "baler_b200", "csrc", name)
        r = subprocess.run([build.NVCC] + build.FLAGS + ["-Xptxas", "-v", "-c", src, "-o", os.devnull],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        assert "dbn_f64" in r.stderr or "mt_dropout" in r.stderr
        props = [line for line in r.stderr.splitlines() if "spill stores" in line]
        assert props and all("0 bytes spill stores, 0 bytes spill loads" in line for line in props), props
