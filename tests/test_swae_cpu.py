"""loss_function_swae without a device: which models and launches DeviceAdam accepts with it, where each model's latent
is, the arithmetic of a BatchNorm that a second encode updates twice, and the missing device as the only obstacle for
Conv_AE (no CPU fallback)."""
import numpy as np
import pytest
import torch

from baler_b200.modules import models, training

SWAE_REFUSAL = "loss_function_swae"


def test_conv_ae_swae_is_accepted_and_needs_the_device(monkeypatch):
    """Conv_AE + loss_function_swae passes the refusals and builds its layer-by-layer trainer, which without a device fails
    like every other compute path"""
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    torch.manual_seed(0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        training.DeviceAdam(models.Conv_AE(25, 10), 1e-3, 2500, block_hw=(5, 5), swae=True)


def test_dropout_and_several_processes_are_still_refused(monkeypatch):
    with pytest.raises(NotImplementedError, match=SWAE_REFUSAL):
        training.DeviceAdam(models.AE_Dropout_BN(24, 15), 1e-3, 64, swae=True)
    monkeypatch.setenv("WORLD_SIZE", "2")
    monkeypatch.setattr(training, "dist_env", lambda: (0, 2))
    for model, kw in ((models.CFD_dense_AE(64, 10), {}), (models.Conv_AE(25, 10), {"block_hw": (5, 5)})):
        with pytest.raises(NotImplementedError, match=SWAE_REFUSAL):
            training.DeviceAdam(model, 1e-3, 64, swae=True, **kw)


def test_latent_layer_of_each_model():
    """the layer whose output model.encode returns: en4 of the 8-Linear AEs, q_z_lin.2 of Conv_AE's training_spec"""
    assert models.AE(24, 15).latent_layer == 3 and models.AE.names[3] == "en4"
    assert models.CFD_dense_AE(64, 10).latent_layer == 3
    m = models.Conv_AE(25, 10)
    assert m.latent_layer == 4 and m._CONV[4][0] == "q_z_lin.2"
    sp = m.training_spec(5, 5)
    assert sp["dims"][m.latent_layer + 1] == 10 and sp["acts"][m.latent_layer] == "relu"


def _bn_train_forward(z, running_mean, running_var, momentum=0.1):
    """nn.BatchNorm2d's running-statistics update in float32, as torch applies it on one train-mode forward of z
    [rows, C, positions]: mean and unbiased variance over rows x positions"""
    z = np.asarray(z, dtype=np.float32)
    m = z.shape[0] * z.shape[2]
    mean = z.mean(axis=(0, 2), dtype=np.float64).astype(np.float32)
    var = z.var(axis=(0, 2), dtype=np.float64).astype(np.float32)
    unbiased = (var * np.float32(m) / np.float32(m - 1)).astype(np.float32)
    mom = np.float32(momentum)
    return ((np.float32(1) - mom) * running_mean + mom * mean).astype(np.float32), \
        ((np.float32(1) - mom) * running_var + mom * unbiased).astype(np.float32)


def test_second_encode_updates_running_statistics_twice():
    """the encoder's BatchNorm2d under upstream's model(inputs) then model.encode(inputs): two updates from the same batch
    statistics, r2 = 0.81 r0 + 0.19 stat; one forward of the same batch leaves 0.9 r0 + 0.1 stat; torch agrees"""
    rng = np.random.default_rng(3)
    z = rng.standard_normal((40, 16, 18)).astype(np.float32) * 2 + 0.5
    r0m, r0v = rng.standard_normal(16).astype(np.float32), (0.5 + rng.random(16)).astype(np.float32)
    once = _bn_train_forward(z, r0m, r0v)
    twice = _bn_train_forward(z, *once)
    mean = z.mean(axis=(0, 2), dtype=np.float64)
    var = z.var(axis=(0, 2), ddof=1, dtype=np.float64)
    assert np.abs(twice[0] - (0.81 * r0m + 0.19 * mean)).max() <= 1e-6 * max(1.0, np.abs(mean).max())
    assert np.abs(twice[1] - (0.81 * r0v + 0.19 * var)).max() <= 1e-6 * np.abs(var).max()
    bn = torch.nn.BatchNorm2d(16)
    bn.running_mean.copy_(torch.from_numpy(r0m))
    bn.running_var.copy_(torch.from_numpy(r0v))
    bn.train()
    zt = torch.from_numpy(z).view(40, 16, 18, 1)
    for _ in range(2):
        bn(zt)
    assert int(bn.num_batches_tracked) == 2
    assert np.abs(bn.running_mean.numpy() - twice[0]).max() <= 1e-6 * max(1.0, np.abs(mean).max())
    assert np.abs(bn.running_var.numpy() - twice[1]).max() <= 1e-6 * np.abs(var).max()


def test_load_trained_counts_batches_per_layer():
    """Conv_AE.load_trained adds one count per training_spec layer (SWAE: 2 per step for the encoder's BatchNorm2d, 1 for
    the decoder's), or one count for all"""
    torch.manual_seed(0)
    m = models.Conv_AE(25, 10)
    sp = m.training_spec(5, 5)
    counts = np.zeros(len(m._CONV), dtype=np.int64)
    counts[[1, 7, 8]] = (6, 3, 3)
    m.load_trained(sp["weights"], sp["biases"], sp["bn"], counts)
    sd = m.state_dict()
    assert [int(sd[k + ".num_batches_tracked"]) for k in ("q_z_conv.3", "p_x_conv.1", "p_x_conv.4")] == [6, 3, 3]
    m.load_trained(sp["weights"], sp["biases"], sp["bn"], 2)
    sd = m.state_dict()
    assert [int(sd[k + ".num_batches_tracked"]) for k in ("q_z_conv.3", "p_x_conv.1", "p_x_conv.4")] == [8, 5, 5]
