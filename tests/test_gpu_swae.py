"""loss_function_swae at any batch size and on Conv_AE (bb_ltrainer_step_swae): batches above 2048 rows, whose projections
are sorted by a stable radix sort in global memory, against the float64 oracle; ties; Conv_AE's step against a float64
restatement and against a torch twin of upstream's loop (model(inputs), then model.encode(inputs): the encoder's
BatchNorm2d updates twice per step); the CLI; host tables; no spills."""
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, randomise_bn2d, rel_l2, rel_max, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import engine, synth
from baler_b200.modules import helper, models, training

pytestmark = pytest.mark.gpu
NAMES = models.AE.names
AE_ACTS = ["leaky", "leaky", "leaky", "none"] * 2
S = 2000
# a bias in front of a BatchNorm2d has a mathematically zero gradient (the mean subtraction removes it): both sides hold
# rounding noise there, which Adam turns into +-lr moves (DESIGN 4.6)
CONV_DEAD = ("q_z_conv.2.bias", "p_x_conv.0.bias", "p_x_conv.3.bias")
BN_AFTER_DEAD = {"q_z_conv.3": "q_z_conv.2.bias", "p_x_conv.1": "p_x_conv.0.bias", "p_x_conv.4": "p_x_conv.3.bias"}
CONV_BN = ("q_z_conv.3", "p_x_conv.1", "p_x_conv.4")


def _draws(rows, z, seed):
    g = torch.Generator().manual_seed(seed)
    prior = torch.randn((rows, z), generator=g)
    proj = torch.randn((S, z), generator=g)
    return prior, proj / proj.norm(dim=1, keepdim=True)


def _dense_step(sd, x, prior, proj, reg):
    tr = engine.LayeredTrainer([sd[n + ".weight"] for n in NAMES], [sd[n + ".bias"] for n in NAMES], AE_ACTS, x.shape[0])
    tr.step_swae(torch.from_numpy(x).cuda(), engine.make_hyper(lr=1e-3), prior.cuda(), proj.cuda(), latent_layer=3,
                 reg_weight=reg, phase=1)
    return tr, tr.grads_view().cpu().numpy().astype(np.float64)


def _flat_named(g):
    return np.concatenate([np.concatenate([np.ravel(g[n + ".weight"]), np.ravel(g[n + ".bias"])]) for n in NAMES])


@pytest.mark.parametrize("rows", [2048, 2049, 4096, 5001, 16384])
def test_large_batch_step_matches_oracle(golden, rows):
    """CFD_dense_AE(64, 10): loss and gradient of one step against the float64 oracle, at the reference's weight 100 and at
    100 B^2, where the sliced-Wasserstein term is a few % of the loss (100 / (B (B - 1)) makes it ~1e-7 of it)"""
    sd0 = sub_sd(golden("swae.npz"), "sd0")
    x = np.random.default_rng(rows).random((rows, 64), dtype=np.float32)
    prior, proj = _draws(rows, 10, rows)
    for reg in (100.0, 100.0 * rows * rows):
        _, flat = _dense_step(sd0, x, prior, proj, reg)
        loss, mse, _, grads = orc.ae_loss_and_grads(sd0, x, swae=(prior.numpy(), proj.numpy(), reg))
        if reg > 100.0:
            assert loss - mse > 0.01 * mse
        ref = _flat_named(grads)
        assert abs(flat[-1] - loss) <= 1e-5 * loss, (reg, flat[-1], loss)
        assert rel_max(flat[:-1], ref) <= 1e-5 and rel_l2(flat[:-1], ref) <= 1e-5, (reg, rel_max(flat[:-1], ref))


def test_ties_and_determinism(golden):
    """4096 rows made of 1024 rows four times over: every projection has exact ties.  The loss and the weight gradient
    (which does not depend on the order among tied rows) match the oracle's stable order; two runs are bit-identical"""
    sd0 = sub_sd(golden("swae.npz"), "sd0")
    x = np.tile(np.random.default_rng(1).random((1024, 64), dtype=np.float32), (4, 1))
    prior, proj = _draws(4096, 10, 2)
    reg = 100.0 * 4096 * 4096
    tr1, flat1 = _dense_step(sd0, x, prior, proj, reg)
    tr2, flat2 = _dense_step(sd0, x, prior, proj, reg)
    loss, _, _, grads = orc.ae_loss_and_grads(sd0, x, swae=(prior.numpy(), proj.numpy(), reg))
    assert abs(flat1[-1] - loss) <= 1e-5 * loss
    assert rel_max(flat1[:-1], _flat_named(grads)) <= 1e-5
    assert flat1.tobytes() == flat2.tobytes()
    h = engine.make_hyper(lr=1e-3)
    for tr in (tr1, tr2):
        tr.step_swae(torch.from_numpy(x).cuda(), h, prior.cuda(), proj.cuda(), latent_layer=3, reg_weight=reg, phase=2)
    assert torch.equal(tr1.params_view(), tr2.params_view())


def conv_swae_step(spec, x, prior, proj, latent_layer, reg_weight, loss_columns=1):
    """oracle.conv_chain_train_step with loss_function_swae: the sliced-Wasserstein term of layer `latent_layer`'s output
    (oracle.swd_term) added to the loss, and its latent gradient added to the decoder's at that layer's output (the sum of
    upstream's two backward passes).  Returns (loss, grads) as conv_chain_train_step."""
    x = np.asarray(x, dtype=np.float64)
    L = len(spec["weights"])
    dense, a, saved = [], x, []
    for l in range(L):
        k, n = spec["dims"][l], spec["dims"][l + 1]
        w = np.asarray(spec["weights"][l], dtype=np.float64)
        b = np.asarray(spec["biases"][l], dtype=np.float64)
        mp = spec["w_maps"][l]
        wd = w.reshape(n, k) if mp is None else np.where(mp >= 0, w.reshape(-1)[np.clip(mp, 0, None)], 0.0).reshape(n, k)
        dense.append(wd)
        z = a @ wd.T + np.repeat(b, n // b.size)
        bn = spec["bn"][l]
        xhat = rstd = None
        if bn is not None:
            c = bn.shape[1]
            zc = z.reshape(z.shape[0], c, n // c)
            mean, var = zc.mean(axis=(0, 2)), zc.var(axis=(0, 2))
            rstd = 1.0 / np.sqrt(var + orc.BN_EPS)
            xhat = (zc - mean[None, :, None]) * rstd[None, :, None]
            z = (xhat * bn[0][None, :, None] + bn[1][None, :, None]).reshape(z.shape)
        out = np.maximum(z, 0.0) if spec["acts"][l] == "relu" else z
        saved.append((a, out, xhat, rstd))
        a = out
    diff = a - x
    swd, dz_swd = orc.swd_term(saved[latent_layer][1], prior, proj, reg_weight)
    loss = float((diff * diff).sum() / loss_columns) + swd
    d = 2.0 * diff / loss_columns
    grads = [None] * L
    for l in reversed(range(L)):
        a_in, out, xhat, rstd = saved[l]
        n = spec["dims"][l + 1]
        if l == latent_layer:
            d = d + dz_swd
        if spec["acts"][l] == "relu":
            d = d * (out > 0)
        g = {}
        bn = spec["bn"][l]
        if bn is not None:
            c = bn.shape[1]
            dc = d.reshape(d.shape[0], c, n // c)
            g["gamma"], g["beta"] = (dc * xhat).sum(axis=(0, 2)), dc.sum(axis=(0, 2))
            m = dc.shape[0] * dc.shape[2]
            dc = (bn[0] * rstd)[None, :, None] * (dc - g["beta"][None, :, None] / m - xhat * g["gamma"][None, :, None] / m)
            d = dc.reshape(d.shape)
        gw, gb = d.T @ a_in, d.sum(axis=0)
        mp = spec["w_maps"][l]
        nb = np.asarray(spec["biases"][l]).size
        g["bias"] = gb.reshape(nb, n // nb).sum(axis=1)
        g["weight"] = gw if mp is None else np.bincount(mp[mp >= 0], weights=gw.reshape(-1)[mp >= 0],
                                                        minlength=np.asarray(spec["weights"][l]).size)
        grads[l] = g
        d = d @ dense[l]
    return loss, grads


def _conv_model(seed=0, z=10):
    torch.manual_seed(seed)
    m = models.Conv_AE(25, z)
    m.load_state_dict(randomise_bn2d(m.state_dict(), seed=seed + 2))
    return m


def _named_grads(m, sp, flat):
    out, off = {}, 0
    for (name, kind, pad, bn_name), w, b, bn in zip(m._CONV, sp["weights"], sp["biases"], sp["bn"]):
        for key, size in ((name + ".weight", w.size), (name + ".bias", b.size)) + \
                (((bn_name + ".weight", bn.shape[1]), (bn_name + ".bias", bn.shape[1])) if bn is not None else ()):
            out[key] = flat[off:off + size]
            off += size
    assert off == flat.size
    return out


@pytest.mark.parametrize("rows", [600, 4096])
def test_conv_ae_step_matches_float64_restatement(rows):
    """Conv_AE: loss and every gradient (kernels, channel biases, Linears, gamma / beta) of one SWAE step against the float64
    restatement, the dead biases excepted, at the reference's weight and at 100 B^2, where the term matters: 1e-5 of each
    tensor's largest at 600 blocks.  At 4096 blocks the MSE part alone differs by up to ~1e-4 in the encoder's Linears
    (measured at weight 100, where the sliced-Wasserstein term is ~1e-7 of the loss): among 8.2 M inputs of the 2000-wide
    ReLU some are zero to fp32 rounding and land on the other side than in float64 (the MSE step has the same property,
    DESIGN 4.6)."""
    m = _conv_model(5)
    sp = m.training_spec(5, 5)
    x = torch.rand((rows, 25), generator=torch.Generator().manual_seed(rows))
    prior, proj = _draws(rows, 10, 3)
    tol = 1e-5 if rows <= 600 else 3e-4
    for reg in (100.0, 100.0 * rows * rows):
        tr = engine.LayeredTrainer(sp["weights"], sp["biases"], sp["acts"], rows, dims=sp["dims"], w_maps=sp["w_maps"],
                                   bn=sp["bn"], loss_columns=1)
        tr.step_swae(x.cuda(), engine.make_hyper(lr=1e-3), prior.cuda(), proj.cuda(), latent_layer=m.latent_layer,
                     reg_weight=reg, phase=1)
        flat = tr.grads_view().cpu().numpy().astype(np.float64)
        loss, grads = conv_swae_step(sp, x.numpy(), prior.numpy(), proj.numpy(), m.latent_layer, reg)
        assert abs(flat[-1] - loss) <= 1e-5 * loss, (reg, flat[-1], loss)
        got = _named_grads(m, sp, flat[:-1])
        ref = {}
        for (name, kind, pad, bn_name), g in zip(m._CONV, grads):
            ref[name + ".weight"], ref[name + ".bias"] = g["weight"], g["bias"]
            if bn_name:
                ref[bn_name + ".weight"], ref[bn_name + ".bias"] = g["gamma"], g["beta"]
        # each tensor against its largest entry, or 1e-2 of the largest weight gradient for a tensor of tiny ones (as in
        # test_conv_ae_train_step_vs_oracle_ragged_batch)
        scale = max(float(np.abs(g["weight"]).max()) for g in grads)
        errs = {k: float(np.abs(got[k] - np.ravel(r)).max() / max(float(np.abs(r).max()), 1e-2 * scale))
                for k, r in ref.items() if k not in CONV_DEAD}
        assert max(errs.values()) <= tol, (reg, {k: e for k, e in errs.items() if e > tol})
        # the trainer counts the encoder's BatchNorm twice: upstream's second encode
        assert list(tr.bn_batches_tracked()[[1, 7, 8]]) == [2, 1, 1]


class _Twin(torch.nn.Module):
    """upstream's Conv_AE (models.py:316-407) for 5x5 blocks, module for module in Conv_AE._CONV's naming"""

    def __init__(self, z):
        super().__init__()
        nn = torch.nn
        self.q_z_conv = nn.Sequential(nn.Conv2d(1, 8, (2, 5), padding=1), nn.ReLU(), nn.Conv2d(8, 16, 3, padding=1),
                                      nn.BatchNorm2d(16), nn.ReLU(), nn.Conv2d(16, 32, 3, padding=0), nn.ReLU())
        self.q_z_lin = nn.Sequential(nn.Linear(128, 2000), nn.ReLU(), nn.Linear(2000, z), nn.ReLU())
        self.p_x_lin = nn.Sequential(nn.Linear(z, 2000), nn.ReLU(), nn.Linear(2000, 128), nn.ReLU())
        self.p_x_conv = nn.Sequential(nn.ConvTranspose2d(32, 16, 3, padding=0), nn.BatchNorm2d(16), nn.ReLU(),
                                      nn.ConvTranspose2d(16, 8, 3, padding=1), nn.BatchNorm2d(8), nn.ReLU(),
                                      nn.ConvTranspose2d(8, 1, (2, 5), padding=1))

    def encode(self, x):
        return self.q_z_lin(self.q_z_conv(x).flatten(1))

    def forward(self, x):
        return self.p_x_conv(self.p_x_lin(self.encode(x)).view(-1, 32, 4, 1))


def _swae_loss(x, z, recon, prior, proj, reg_weight=100.0):
    """utils.loss_function_swae (utils.py:27-91) with the draws given: sum-MSE / shape[1] + reg_weight / (B (B - 1)) x
    the mean squared difference of the batch-sorted projections of z and of the prior draws"""
    b = z.shape[0]
    swd = ((torch.sort(z @ proj.T, dim=0)[0] - torch.sort(prior @ proj.T, dim=0)[0]) ** 2).mean()
    return ((recon - x) ** 2).sum() / x.shape[1] + reg_weight / (b * (b - 1)) * swd


def _twin_steps(twin, opt, x, batch, z):
    """one reference epoch of fit with this loss: per batch model(inputs), model.encode(inputs), the draws in
    loss_function_swae's order from torch's global generator (randn_like(z), then 2000 normalised projections), Adam.
    Returns the batch losses."""
    twin.train()
    losses = []
    for r0 in range(0, x.shape[0], batch):
        xb = x[r0:r0 + batch].view(-1, 1, 5, 5)
        opt.zero_grad()
        recon = twin(xb)
        lat = twin.encode(xb)
        prior = torch.randn_like(lat)
        proj = torch.randn(S, z)
        proj = proj / proj.norm(dim=1).view(-1, 1)
        loss = _swae_loss(xb, lat, recon, prior, proj)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    return losses


def _running_mean_shift(history, twin_history, bn, steps, per_step):
    """what the dead bias in front of BatchNorm `bn` adds to the difference of the two running means: every batch mean
    contains the bias of that step, weighted in the final running mean by momentum 0.1 and the updates after it"""
    key = BN_AFTER_DEAD[bn]
    shift = 0.0
    for k in range(steps):  # history[k]: parameters before step k + 1
        w = sum(0.1 * 0.9 ** (j + per_step * (steps - 1 - k)) for j in range(per_step))
        shift = shift + w * (history[k][key].double() - twin_history[k][key].double())
    return shift.numpy()


def test_conv_ae_matches_torch_twin_of_upstream_loop():
    """DeviceAdam on Conv_AE with loss_function_swae (batches of 2500 blocks: the radix-sort path) against the twin after
    1 and 3 steps: running statistics, num_batches_tracked (2 per step for the encoder's BatchNorm2d), parameters"""
    z = 10
    m = _conv_model(7, z)
    twin = _Twin(z)
    twin.load_state_dict({k: v.clone() for k, v in m.state_dict().items()})
    table = torch.rand((5000, 25), generator=torch.Generator().manual_seed(8))
    batches = [table[:2500], table[2500:], table[:2500]]
    opt = training.DeviceAdam(m, 1e-3, 2500, block_hw=(5, 5), swae=True)
    history, ours = [{k: v.clone() for k, v in m.state_dict().items()}], []
    torch.manual_seed(11)
    for xb in batches:
        ours.append(opt.epoch_swae(xb.cuda(), 2500, z))
        opt.sync_model()
        history.append({k: v.clone() for k, v in m.state_dict().items()})
    torch.manual_seed(11)
    topt = torch.optim.Adam(twin.parameters(), lr=1e-3)
    twin_history = [{k: v.detach().clone() for k, v in twin.state_dict().items()}]
    theirs = []
    for xb in batches:
        theirs += _twin_steps(twin, topt, xb, 2500, z)
        twin_history.append({k: v.detach().clone() for k, v in twin.state_dict().items()})
    assert np.abs(np.array(ours) - theirs).max() <= 1e-5 * max(theirs), (ours, theirs)
    for steps in (1, 3):
        sd, tsd = history[steps], twin_history[steps]
        for bn in CONV_BN:
            per_step = 2 if bn == "q_z_conv.3" else 1
            assert int(sd[bn + ".num_batches_tracked"]) == int(tsd[bn + ".num_batches_tracked"]) == per_step * steps
            assert rel_max(sd[bn + ".running_var"].numpy(), tsd[bn + ".running_var"].numpy()) <= 1e-5, (steps, bn)
            shift = _running_mean_shift(history, twin_history, bn, steps, per_step)
            got = sd[bn + ".running_mean"].numpy().astype(np.float64) - shift
            assert rel_max(got, tsd[bn + ".running_mean"].numpy()) <= 1e-5, (steps, bn)
        errs = {k: rel_max(sd[k].numpy(), tsd[k].numpy()) for k in tsd
                if k.endswith((".weight", ".bias")) and k not in CONV_DEAD}
        # after one step 1e-5.  Three steps apart, fp32 on both sides: Adam moves an entry by ~lr * m / sqrt(v) whatever the
        # gradient's size, so entries whose gradient is cancellation noise differ by a fraction of lr = 1e-3 (observed
        # 1.8e-4 of a tensor's largest weight; test_conv_ae_train_steps_match_reference allows 2e-3 for the MSE loss)
        tol = 1e-5 if steps == 1 else 1e-3
        assert max(errs.values()) <= tol, (steps, {k: e for k, e in errs.items() if e > tol})


def _conv_workspace(tmp_path, monkeypatch, n_snap, **extra):
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CFD_workspace", "CFD_project_train")
    snaps = synth.cfd_snapshots(n_snap)
    snaps = (snaps - snaps.min()) / (snaps.max() - snaps.min())
    path = os.path.join("workspaces", "CFD_workspace", "data", "CFD_blocks.npz")
    np.savez(path, data=snaps, names=np.array(["snapshot"]))
    out = os.path.join("workspaces", "CFD_workspace", "CFD_project_train", "output")

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name, model_type = 2, 10, False, "Conv_AE", "convolutional"
        batch_size, custom_norm, extra_compression, separate_model_saving = 2500, True, False, False
        save_error_bounded_deltas, convert_to_blocks = False, [1, 5, 5]
        epochs, lr, reg_param, RHO, l1, test_size = 2, 1e-3, 0.001, 0.05, True, 0
        early_stopping, early_stopping_patience, min_delta = False, 100, 0
        lr_scheduler, lr_scheduler_patience = False, 50
        intermittent_model_saving, intermittent_saving_patience = False, 100
        activation_extraction, deterministic_algorithm = False, True
        custom_loss_function = "loss_function_swae"

    for k, v in extra.items():
        setattr(cfg, k, v)
    return cfg, out, snaps


def test_cli_conv_ae_swae_train_compress_decompress(tmp_path, monkeypatch):
    """--mode train of a Conv_AE workspace (5x5 blocks, batch 2500: one large and one ragged batch per epoch) with
    loss_function_swae: loss_data.npy's first epoch is the twin's, model.pt counts the twin's batches; compress and
    decompress run on it"""
    from baler_b200 import baler
    cfg, out, snaps = _conv_workspace(tmp_path, monkeypatch, 30)
    seen = {}
    real_train = training.train

    def spy(model, variables, train_data, test_data, project_path, config):
        seen.update(sd={k: v.clone() for k, v in model.state_dict().items()}, data=np.array(train_data), z=model.z_dim)
        return real_train(model, variables, train_data, test_data, project_path, config)

    monkeypatch.setattr(training, "train", spy)
    baler.perform_training(out, cfg, False)
    losses = np.load(os.path.join(out, "training", "loss_data.npy"))
    assert losses.shape == (2, 2) and np.isfinite(losses).all()
    assert list(np.load(os.path.join(out, "training", "final_layer.npy"))) == [500, 32, 4, 1]
    twin = _Twin(seen["z"])
    twin.load_state_dict(seen["sd"])
    topt = torch.optim.Adam(twin.parameters(), lr=1e-3)
    x = torch.from_numpy(seen["data"].reshape(-1, 25).astype(np.float32))
    assert x.shape[0] == 3000
    torch.manual_seed(0)
    first = np.mean(_twin_steps(twin, topt, x, 2500, seen["z"]))
    _twin_steps(twin, topt, x, 2500, seen["z"])
    assert abs(losses[0, 0] - first) <= 1e-5 * first, (losses[0, 0], first)
    sd = torch.load(os.path.join(out, "compressed_output", "model.pt"))
    for bn in CONV_BN:
        assert int(sd[bn + ".num_batches_tracked"]) == int(twin.state_dict()[bn + ".num_batches_tracked"])
    assert int(sd["q_z_conv.3.num_batches_tracked"]) == 8 and int(sd["p_x_conv.1.num_batches_tracked"]) == 4
    baler.perform_compression(out, cfg, False)
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    assert dec.shape == (30, 1, 50, 50) and np.isfinite(dec).all()


def test_cli_cfd_dense_swae_batch_4096(tmp_path, monkeypatch):
    """CFD_dense_AE on 1-D rows with loss_function_swae at batch 4096 (one large, one ragged batch) trains"""
    from baler_b200 import baler
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("WS", "P")
    path = os.path.join("workspaces", "WS", "data", "P_data.npz")
    table = np.random.default_rng(4).random((6000, 32)).astype(np.float32)
    np.savez(path, data=table, names=np.array(["c%d" % i for i in range(32)]))
    out = os.path.join("workspaces", "WS", "P", "output")

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name, model_type = 1, 2, False, "CFD_dense_AE", "dense"
        epochs, lr, batch_size, early_stopping, lr_scheduler = 3, 1e-3, 4096, False, False
        early_stopping_patience, min_delta, lr_scheduler_patience, custom_norm = 100, 0, 50, False
        reg_param, RHO, test_size, extra_compression = 0.001, 0.05, 0, False
        intermittent_model_saving, intermittent_saving_patience = False, 100
        l1, activation_extraction, deterministic_algorithm = True, False, True
        convert_to_blocks, separate_model_saving, save_error_bounded_deltas = False, False, False
        custom_loss_function = "loss_function_swae"

    baler.perform_training(out, cfg, False)
    losses = np.load(os.path.join(out, "training", "loss_data.npy"))
    assert losses.shape == (2, 3) and np.isfinite(losses).all() and losses[0, -1] < losses[0, 0]


def test_conv_ae_swae_host_table_equals_resident():
    """a Conv_AE SWAE epoch from a host table (one batch uploaded at a time) equals the resident one bit for bit, on the
    radix-sort path with a ragged last batch"""
    table = np.random.default_rng(9).random((5000, 25), dtype=np.float32)
    runs = []
    for host in (False, True):
        m = _conv_model(3)
        opt = training.DeviceAdam(m, 1e-3, 2100, block_hw=(5, 5), swae=True)
        torch.manual_seed(4)
        x = table if host else torch.from_numpy(table).cuda()
        losses = [opt.epoch_swae(x, 2100, 10) for _ in range(2)]
        tr = opt.trainer
        runs.append((losses, tr.params_view().cpu().numpy().tobytes(),
                     np.concatenate([b.ravel() for b in tr.get_bn() if b is not None]).tobytes(),
                     tr.bn_batches_tracked().tolist()))
    assert runs[0] == runs[1]
    assert runs[0][3][1] == 12 and runs[0][3][7] == 6


def test_swae_kernels_do_not_spill():
    """-Xptxas -v on the layer-by-layer trainer: the sliced-Wasserstein kernels and bn_fwd_kernel do not spill"""
    from baler_b200 import build
    src = os.path.join(ROOT, "baler_b200", "csrc", "bb_train_layered.cu")
    r = subprocess.run([build.NVCC] + build.FLAGS + ["-Xptxas", "-v", "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stderr.splitlines()
    props = {}
    for i, line in enumerate(lines):  # "Function properties for <mangled name>", then its stack / spill line
        for k in ("swd_radix_kernel", "swd_sort_kernel", "swd_fold_kernel", "bn_fwd_kernel"):
            if "Function properties for" in line and k in line:
                props[k] = lines[i + 1]
    assert len(props) == 4 and all("0 bytes spill stores, 0 bytes spill loads" in v for v in props.values()), props
