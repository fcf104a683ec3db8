"""2-D (CFD) models: Conv_AE on 5x5 blocks (dense-equivalent chain, layered GEMM path) and CFD_dense_AE on 50x50
snapshots, against fixtures produced by the reference modules (tests/golden/conv_ae.npz, cfd_dense.npz)."""
import os

import numpy as np
import pytest
import torch

from conftest import randomise_bn2d, rel_l2, rel_max
from baler_b200 import synth
from baler_b200.modules import helper, models

pytestmark = pytest.mark.gpu


def check_sums(model, g):
    for k, v in model.state_dict().items():
        ref = float(g["chk/" + k])
        assert abs(float(v.double().abs().sum()) - ref) <= 1e-6 * max(ref, 1.0), k


@pytest.mark.parametrize("precision", ["auto", "fp32"])
def test_conv_ae_eval_matches_reference(golden, precision):
    """the reference module's outputs on the tensor-core GEMM path (auto = split16: mma.sync hi / lo) and on the fp32 one"""
    g = golden("conv_ae.npz")
    torch.manual_seed(0)
    m = models.Conv_AE(5, 250)
    m.load_state_dict(randomise_bn2d(m.state_dict()))
    check_sums(m, g)  # same initial weights and BatchNorm statistics as the reference instance
    m.eval()
    assert m.codec(5, 5).auto_precision == "split16"
    x = torch.from_numpy(g["blocks"]).view(-1, 1, 5, 5)
    z = m.encode(x, precision=precision)
    assert z.shape == (600, 250) and z.dtype == torch.float32
    assert tuple(m.get_final_layer_dims()) == (600, 32, 4, 1)
    assert rel_max(z.cpu().numpy(), g["latent_eval"]) <= 1e-5 and rel_l2(z.cpu().numpy(), g["latent_eval"]) <= 1e-5
    y = m.decode(torch.from_numpy(g["latent_eval"]), precision=precision)
    assert y.shape == (600, 1, 5, 5)
    assert rel_max(y.cpu().numpy(), g["recon_eval"]) <= 1e-5 and rel_l2(y.cpu().numpy(), g["recon_eval"]) <= 1e-5
    with pytest.raises(RuntimeError, match="flattens"):
        m.encode(torch.zeros(4, 1, 50, 50))  # the shipped 50x50 CFD_project_still shape is invalid upstream too
    with pytest.raises(NotImplementedError):
        m.train().encode(x)


@pytest.mark.parametrize("tag,h,w,z_dim", [("b36", 3, 6, 9), ("b28", 2, 8, 4)])
def test_conv_ae_other_block_shapes(golden, tag, h, w, z_dim):
    """the other two block shapes the reference model accepts (their conv stack flattens to the hard-coded 128 values,
    SURVEY F7b): 3x6 blocks with z = 9, 2x8 blocks with z = 4, against the reference module's eval outputs"""
    g = golden("conv_shapes.npz")
    torch.manual_seed(0)
    m = models.Conv_AE(w, z_dim)
    m.load_state_dict(randomise_bn2d(m.state_dict()))
    for k, v in m.state_dict().items():
        ref = float(g[f"{tag}/chk/{k}"])
        assert abs(float(v.double().abs().sum()) - ref) <= 1e-6 * max(ref, 1.0), k
    m.eval()
    x = torch.from_numpy(g[f"{tag}/blocks"]).view(-1, 1, h, w)
    for precision in ("auto", "fp32"):
        z = m.encode(x, precision=precision)
        assert tuple(m.get_final_layer_dims()) == tuple(g[f"{tag}/final_layer"])
        assert rel_max(z.cpu().numpy(), g[f"{tag}/latent_eval"]) <= 1e-5
        y = m.decode(torch.from_numpy(g[f"{tag}/latent_eval"]), precision=precision)
        assert y.shape == g[f"{tag}/recon_eval"].shape
        assert rel_max(y.cpu().numpy(), g[f"{tag}/recon_eval"]) <= 1e-5


@pytest.mark.parametrize("precision", ["auto", "fp32"])
def test_cfd_dense_ae_2500_features(golden, precision):
    g = golden("cfd_dense.npz")
    torch.manual_seed(0)
    m = models.CFD_dense_AE(2500, 25)
    check_sums(m, g)
    m.eval()
    assert m.codec().auto_precision == "split16"  # W1 is 2 MB: layered GEMM path (tensor cores), not the fused kernels
    x = torch.from_numpy(synth.cfd_snapshots(60).reshape(60, 2500))
    z = m.encode(x, precision=precision)
    assert z.dtype == torch.float32
    assert rel_max(z.cpu().numpy(), g["latent"]) <= 1e-5 and rel_l2(z.cpu().numpy(), g["latent"]) <= 1e-5
    y = m.decode(torch.from_numpy(g["latent"]), precision=precision)
    assert rel_max(y.cpu().numpy(), g["recon"]) <= 1e-5 and rel_l2(y.cpu().numpy(), g["recon"]) <= 1e-5


@pytest.mark.parametrize("chunk", [None, "37888"])
def test_layered_path_ragged_rows_and_chunks(golden, chunk, monkeypatch):
    """more rows than one scratch chunk (32768 on the fp32 path; the tcgen05 path takes 8 row tiles per SM, or the 37888
    rows the tuning variable asks for) and a ragged tail on the GEMM path; Conv_AE blocks"""
    if chunk is not None:
        monkeypatch.setenv("BALER_B200_LAYER_CHUNK", chunk)
    g = golden("conv_ae.npz")
    torch.manual_seed(0)
    m = models.Conv_AE(5, 250)
    m.load_state_dict(randomise_bn2d(m.state_dict()))
    m.eval()
    base = g["blocks"].reshape(600, 25)
    n = 32768 * 2 + 77
    idx = np.arange(n) % 600
    for precision in ("auto", "fp32"):
        z = m.codec(5, 5).encode(torch.from_numpy(np.ascontiguousarray(base[idx])).cuda(), precision=precision)
        ref = g["latent_eval"][idx]
        assert rel_max(z.cpu().numpy(), ref) <= 1e-5
        assert torch.equal(z[:600], z[600:1200])  # independent rows: identical blocks give identical bits
        # ... and back (>= 148 row tiles per chunk: the tcgen05 GEMM keeps the A tile of the 2000-wide layers resident)
        y = m.codec(5, 5).decode(z, precision=precision)
        assert rel_max(y.cpu().numpy(), g["recon_eval"].reshape(600, 25)[idx]) <= 1e-5
        assert torch.equal(y[:600], y[600:1200])


@pytest.mark.parametrize("rows", [1, 127, 129, 5000, 20000])
@pytest.mark.parametrize("mode", ["tcgen05", "mma", "fp32"])
def test_layered_gemm_odd_shapes_vs_float64(rows, mode, monkeypatch):
    """the per-layer GEMMs (tcgen05 gemm_tc5_kernel; mma.sync dense_layer_tc_kernel; fp32 dense_layer_kernel, what
    precision "fp32" runs) on a chain with widths that are multiples of nothing, a long contraction (3001: partial
    accumulators) and ragged row counts (20000: enough row tiles for the resident-A mode of the 70 -> 1111 layer), against
    float64 numpy"""
    from baler_b200 import engine
    if mode == "mma":
        monkeypatch.setenv("BALER_B200_LAYERED_MMA", "1")
    rng = np.random.default_rng(17)
    dims_e, dims_d = [333, 3001, 17, 9], [9, 70, 1111, 333]
    acts = ["leaky", "relu", "none"]

    def layers(dims):
        return [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i]), 0.1 * rng.standard_normal(dims[i + 1]), acts[i])
                for i in range(len(dims) - 1)]

    enc, dec = layers(dims_e), layers(dims_d)
    codec = engine.DenseCodec(enc, dec)
    assert codec.auto_precision == "split16"
    x = rng.standard_normal((rows, 333)).astype(np.float32)

    def ref(v, ls):
        v = v.astype(np.float64)
        for w, b, a in ls:
            v = v @ w.T + b
            v = np.where(v > 0, v, 0.01 * v) if a == "leaky" else np.maximum(v, 0) if a == "relu" else v
        return v

    precision = "fp32" if mode == "fp32" else "auto"
    z = codec.encode(torch.from_numpy(x).cuda(), precision=precision)
    zr = ref(x, enc)
    assert rel_max(z.cpu().numpy(), zr) <= 1e-5 and rel_l2(z.cpu().numpy(), zr) <= 1e-5
    y = codec.decode(z, precision=precision)
    yr = ref(z.cpu().numpy(), dec)
    assert rel_max(y.cpu().numpy(), yr) <= 1e-5 and rel_l2(y.cpu().numpy(), yr) <= 1e-5


def test_trim_and_destroy_of_a_layered_model_leave_no_pending_cuda_error():
    """bb_model_trim releases the layered path's activation scratch of a live model (the next call allocates again and gives
    the same bits); bb_model_destroy must not release it a second time - a double cudaFree is not fatal, but it leaves an
    `invalid argument` for the next call that reads cudaGetLastError"""
    import gc
    from baler_b200 import engine
    rng = np.random.default_rng(1)

    def layers(dims):
        return [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i]), 0.1 * rng.standard_normal(dims[i + 1]), "relu")
                for i in range(len(dims) - 1)]

    codec = engine.DenseCodec(layers([333, 3001, 17, 9]), layers([9, 70, 1111, 333]))  # (too wide for the fused kernels)
    x = torch.randn(1000, 333, device="cuda")
    free0 = torch.cuda.mem_get_info()[0]
    y1 = codec.decode(codec.encode(x))
    torch.cuda.synchronize()
    held = free0 - torch.cuda.mem_get_info()[0]
    codec.trim()
    assert free0 - torch.cuda.mem_get_info()[0] < held  # the scratch went back
    y2 = codec.decode(codec.encode(x))
    assert torch.equal(y1, y2)
    del codec
    gc.collect()
    mn, mx = engine.colminmax(x)  # a launch that reports cudaGetLastError
    assert torch.equal(mn, x.min(dim=0).values) and torch.equal(mx, x.max(dim=0).values)
    # ... and the layered trainer, the call that tripped over the stale error
    tr = engine.LayeredTrainer([w for w, _, _ in layers([32, 64, 32])], [np.zeros(64), np.zeros(32)], ["relu", "none"], 64)
    tr.step(torch.rand(64, 32, device="cuda"), engine.make_hyper(lr=1e-3))


def test_layered_tensor_core_range_guard():
    """values beyond the fp16 range on the layered tensor-core path raise the sticky flag; AUTO callers re-run in fp32"""
    torch.manual_seed(0)
    m = models.CFD_dense_AE(2500, 25).eval()
    x = torch.from_numpy(synth.cfd_snapshots(8).reshape(8, 2500)).cuda() * 1.0e6
    codec = m.codec()
    z = codec.encode(x)                      # auto: trips, re-runs on the fp32 GEMMs
    z32 = codec.encode(x, precision="fp32")
    assert torch.isfinite(z).all() and torch.equal(z, z32)


def test_conv_cli_compress_decompress(golden, tmp_path, monkeypatch):
    """--mode compress / decompress for a convolutional project with convert_to_blocks = [1, 5, 5]"""
    from baler_b200 import baler

    g = golden("conv_ae.npz")
    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CFD_workspace", "CFD_project_blocks")
    snaps = synth.cfd_snapshots(6)
    path = os.path.join("workspaces", "CFD_workspace", "data", "CFD_blocks.npz")
    np.savez(path, data=snaps, names=np.array(["snapshot"]))
    out = os.path.join("workspaces", "CFD_workspace", "CFD_project_blocks", "output")
    torch.manual_seed(0)
    m = models.Conv_AE(50, 250)
    m.load_state_dict(randomise_bn2d(m.state_dict()))
    torch.save(m.state_dict(), os.path.join(out, "compressed_output", "model.pt"))

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name, model_type = 2, 10, False, "Conv_AE", "convolutional"
        batch_size, custom_norm, extra_compression, separate_model_saving = 600, True, False, False
        save_error_bounded_deltas, convert_to_blocks = False, [1, 5, 5]

    baler.perform_compression(out, cfg, False)
    comp = np.load(os.path.join(out, "compressed_output", "compressed.npz"))["data"]
    assert comp.shape == (600, 250) and comp.dtype == np.float32
    assert rel_max(comp, g["latent_eval"]) <= 1e-5
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    assert dec.shape == (6, 1, 50, 50) and dec.dtype == np.float32
    assert rel_max(dec.reshape(600, 25), g["recon_eval"].reshape(600, 25)) <= 1e-5


# ---- Conv_AE training (tests/golden/conv_train.npz: the reference's own steps, oracle/gen_golden.py::gen_conv_train)

CONV_BIG = ("q_z_lin.0.weight", "q_z_lin.2.weight", "p_x_lin.0.weight", "p_x_lin.2.weight")
# a bias in front of a BatchNorm2d has a mathematically zero gradient (the mean subtraction removes it): both sides hold
# rounding noise there, which Adam's first steps turn into +-lr moves.  It does not change the function.
CONV_DEAD = ("q_z_conv.2.bias", "p_x_conv.0.bias", "p_x_conv.3.bias")


def _conv_model():
    torch.manual_seed(0)
    m = models.Conv_AE(5, 250)
    m.load_state_dict(randomise_bn2d(m.state_dict()))
    return m


def _conv_trainer(m, max_batch=300):
    from baler_b200 import engine
    sp = m.training_spec(5, 5)
    tr = engine.LayeredTrainer(sp["weights"], sp["biases"], sp["acts"], max_batch, dims=sp["dims"], w_maps=sp["w_maps"],
                               bn=sp["bn"], loss_columns=1)
    return tr, sp


def _named_flat(m, sp, flat):
    """trainer's flat vector (layer after layer: weights | biases | gamma | beta) -> {state_dict key: float64 array}"""
    out, off = {}, 0
    for (name, kind, pad, bn_name), w, b, bn in zip(m._CONV, sp["weights"], sp["biases"], sp["bn"]):
        out[name + ".weight"] = flat[off:off + w.size]; off += w.size
        out[name + ".bias"] = flat[off:off + b.size]; off += b.size
        if bn is not None:
            c = bn.shape[1]
            out[bn_name + ".weight"] = flat[off:off + c]; off += c
            out[bn_name + ".bias"] = flat[off:off + c]; off += c
    assert off == flat.size
    return out


def _check_packed(g, prefix, named, tol, skip=()):
    scale = max(float(np.abs(g[f"{prefix}/{k}#sample" if k in CONV_BIG else f"{prefix}/{k}"]).max()) for k in named)
    bad = {}
    for k, a in named.items():
        if k in skip:
            continue
        a = np.asarray(a, dtype=np.float64).reshape(-1)
        if k in CONV_BIG:
            ref = g[f"{prefix}/{k}#sample"]
            if abs(np.sqrt((a * a).sum()) - float(g[f"{prefix}/{k}#norm"])) > tol * float(g[f"{prefix}/{k}#norm"]):
                bad[k + "#norm"] = np.sqrt((a * a).sum()) / float(g[f"{prefix}/{k}#norm"]) - 1
            a = a[::101]
        else:
            ref = g[f"{prefix}/{k}"].reshape(-1)
        floor = max(float(np.abs(ref).max()), 1e-2 * scale)
        err = float(np.abs(a - ref).max()) / floor
        if err > tol:
            bad[k] = err
    assert not bad, (prefix, bad)


def test_conv_ae_train_steps_match_reference(golden):
    """one training step of Conv_AE as training.fit runs it (train-mode BatchNorm2d, sum-MSE / 1 channel, backward, Adam):
    loss, every gradient and the parameters after 1 and 3 steps against the reference's own values"""
    from baler_b200 import engine
    g = golden("conv_train.npz")
    m = _conv_model()
    tr, sp = _conv_trainer(m)
    x = torch.from_numpy(g["blocks"]).cuda()
    h = engine.make_hyper(lr=1e-3)
    tr.step(x[:300].contiguous(), h, phase=1)
    grads = tr.grads_view().cpu().numpy().astype(np.float64)
    assert abs(grads[-1] - g["losses"][0]) <= 1e-5 * g["losses"][0]
    skip = CONV_DEAD
    _check_packed(g, "g0", _named_flat(m, sp, grads[:-1]), 1e-5, skip)
    tr.step(x[:300].contiguous(), h, phase=2)
    _check_packed(g, "sd1", _named_flat(m, sp, tr.params_view().cpu().numpy().astype(np.float64)), 1e-5, skip)
    tr.loss_accum.zero_()
    tr.step(x[300:].contiguous(), h)
    tr.step(x[:300].contiguous(), h)
    # fp32 on both sides and three steps apart: Adam moves an entry by ~lr * g / |g| whatever its size, so entries whose
    # gradient is cancellation noise (weights behind mostly-dead ReLU units) differ by a fraction of lr = 1e-3 (observed
    # 5e-5 absolute on p_x_lin.0, 9e-4 of the tensor's largest weight); the one-step gates above are the 1e-5 ones
    _check_packed(g, "sd3", _named_flat(m, sp, tr.params_view().cpu().numpy().astype(np.float64)), 2e-3, skip)
    assert abs(tr.loss_accum.item() - g["losses"][1:].sum()) <= 1e-4 * g["losses"][1:].sum()
    bn = tr.get_bn()
    for (name, kind, pad, bn_name), b4 in zip(m._CONV, bn):
        if bn_name is not None:
            # the batch mean contains the dead bias in front of the BatchNorm (see CONV_DEAD): +-lr per step of noise
            assert np.abs(b4[2] - g[f"sd3/{bn_name}.running_mean"]).max() <= 1e-3
            assert rel_max(b4[3], g[f"sd3/{bn_name}.running_var"]) <= 1e-4
    # eval mode (running statistics): the validation loss of the first 300 blocks
    assert abs(tr.validate(x[:300].contiguous(), 300) - float(g["eval_loss"])) <= 1e-3 * float(g["eval_loss"])


def test_conv_ae_training_through_the_training_module(golden, tmp_path):
    """training.train on a convolutional 2-D project: loss_data.npy within 1 % of the reference's two epochs from the same
    initial weights, final_layer.npy as the reference writes it, and the trained model's eval-mode reconstruction"""
    from types import SimpleNamespace
    from baler_b200.modules import training
    g = golden("conv_train.npz")
    blocks = g["blocks"].reshape(-1, 5, 5)
    cfg = SimpleNamespace(deterministic_algorithm=False, batch_size=300, data_dimension=2, model_type="convolutional",
                          model_name="Conv_AE", lr=1e-3, reg_param=0.001, early_stopping=False, early_stopping_patience=100,
                          min_delta=0, lr_scheduler=False, lr_scheduler_patience=50, epochs=2, test_size=0,
                          intermittent_model_saving=False, intermittent_saving_patience=100, RHO=0.05, l1=True,
                          activation_extraction=False)
    m = _conv_model()
    training.train(m, 5, blocks, blocks, str(tmp_path), cfg)
    losses = np.load(tmp_path / "loss_data.npy")
    assert losses.shape == (2, 2)
    assert np.abs(losses - g["loss_data"]).max() <= 1e-2 * np.abs(g["loss_data"]).max()
    assert np.abs(losses[0] - g["loss_data"][0]).max() <= 1e-4 * g["loss_data"][0, 0]
    assert list(np.load(tmp_path / "final_layer.npy")) == list(g["final_layer"]) == [300, 32, 4, 1]
    sd = m.state_dict()
    assert int(sd["p_x_conv.1.num_batches_tracked"]) == 4 == int(g["sd_final/p_x_conv.1.num_batches_tracked"])
    assert rel_max(sd["q_z_conv.3.running_var"].numpy(), g["sd_final/q_z_conv.3.running_var"]) <= 1e-3
    m.eval()
    y = m(torch.from_numpy(g["blocks"][:64]).view(-1, 1, 5, 5)).cpu().numpy().reshape(64, 25)
    # eval mode reads bias - running_mean of the three dead biases (CONV_DEAD): Adam moves them by +-lr per step on rounding
    # noise and the running mean follows with momentum 0.1, so after 4 steps the two sides differ by a few 1e-3 there
    # (observed 1.3e-2 of the largest output); the train-mode losses above, which do not see those biases, agree to 4e-6
    assert rel_max(y, g["recon_final"]) <= 4e-2 and rel_l2(y, g["recon_final"]) <= 4e-2


def test_conv_cli_train_compress_decompress(tmp_path, monkeypatch):
    """--mode train / compress / decompress of a convolutional project (convert_to_blocks = [1, 5, 5]): the files of the
    reference's train mode, then a round trip through the trained model"""
    from baler_b200 import baler

    monkeypatch.chdir(tmp_path)
    helper.create_new_project("CFD_workspace", "CFD_project_train")
    snaps = synth.cfd_snapshots(6)
    snaps = (snaps - snaps.min()) / (snaps.max() - snaps.min())
    path = os.path.join("workspaces", "CFD_workspace", "data", "CFD_blocks.npz")
    np.savez(path, data=snaps, names=np.array(["snapshot"]))
    out = os.path.join("workspaces", "CFD_workspace", "CFD_project_train", "output")

    class cfg(helper.Config):
        input_path = path
        data_dimension, compression_ratio, apply_normalization, model_name, model_type = 2, 10, False, "Conv_AE", "convolutional"
        batch_size, custom_norm, extra_compression, separate_model_saving = 200, True, False, False
        save_error_bounded_deltas, convert_to_blocks = False, [1, 5, 5]
        epochs, lr, reg_param, RHO, l1, test_size = 30, 1e-3, 0.001, 0.05, True, 0
        early_stopping, early_stopping_patience, min_delta = False, 100, 0
        lr_scheduler, lr_scheduler_patience = False, 50
        intermittent_model_saving, intermittent_saving_patience = False, 100
        activation_extraction, deterministic_algorithm = False, True

    baler.perform_training(out, cfg, False)
    losses = np.load(os.path.join(out, "training", "loss_data.npy"))
    assert losses.shape == (2, 30) and np.isfinite(losses).all() and losses[0, -1] < 0.2 * losses[0, 0]
    assert list(np.load(os.path.join(out, "training", "final_layer.npy"))) == [200, 32, 4, 1]
    sd = torch.load(os.path.join(out, "compressed_output", "model.pt"))
    assert len(sd) == 35 and sd["q_z_conv.5.weight"].shape == (32, 16, 3, 3) and sd["q_z_conv.5.weight"].dtype == torch.float32
    assert int(sd["q_z_conv.3.num_batches_tracked"]) == 90
    baler.perform_compression(out, cfg, False)
    baler.perform_decompression(out, cfg, False)
    dec = np.load(os.path.join(out, "decompressed_output", "decompressed.npz"))["data"]
    assert dec.shape == (6, 1, 50, 50)
    err = float(((dec.reshape(6, 50, 50) - snaps) ** 2).mean())
    assert err < 0.5 * float(((snaps - snaps.mean()) ** 2).mean())  # better than predicting the mean after 30 epochs


def test_conv_ae_train_step_vs_oracle_ragged_batch():
    """a ragged batch (77 blocks, trainer sized for 128) and other weights against the float64 restatement
    (oracle.conv_chain_train_step, itself pinned to the reference's step in tests/test_oracle_golden.py)"""
    from baler_b200 import engine
    from oracle import baler_oracle as orc
    torch.manual_seed(5)
    m = models.Conv_AE(5, 250)
    m.load_state_dict(randomise_bn2d(m.state_dict(), seed=9))
    tr, sp = _conv_trainer(m, max_batch=128)
    x = torch.rand((77, 25), generator=torch.Generator().manual_seed(6))
    tr.step(x.cuda(), engine.make_hyper(lr=1e-3), phase=1)
    flat = tr.grads_view().cpu().numpy().astype(np.float64)
    loss, grads, _ = orc.conv_chain_train_step(sp, x.numpy())
    assert abs(flat[-1] - loss) <= 1e-5 * loss
    got = _named_flat(m, sp, flat[:-1])
    scale = max(float(np.abs(g["weight"]).max()) for g in grads)
    for (name, kind, pad, bn_name), g in zip(m._CONV, grads):
        pairs = [(name + ".weight", g["weight"]), (name + ".bias", g["bias"])]
        if bn_name:
            pairs += [(bn_name + ".weight", g["gamma"]), (bn_name + ".bias", g["beta"])]
        for key, ref in pairs:
            ref = np.asarray(ref).reshape(-1)
            floor = max(float(np.abs(ref).max()), 1e-2 * scale)
            # a dead bias (exactly 0 in float64) holds fp32 cancellation noise of the 77 x 18 summed dZ values: ~5e-4 of floor
            assert np.abs(got[key] - ref).max() <= (5e-3 if key in CONV_DEAD else 1e-5) * floor, key
