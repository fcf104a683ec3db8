"""Test infrastructure for float64 AE_Dropout_BN training (not product code).

- `bernoulli_masks`: numpy restatement of the dropout masks torch's CPU generator draws with bernoulli_(1 - p) on float64
  tensors: MT19937 continued from torch.Generator.get_state(), 2 words per element (first word high),
  keep = (random64 & (2^53 - 1)) * 2^-53 < 1 - p.
- `DbnTwin` / `fit` / `validate`: the reference's AE_Dropout_BN training loop (models.py:256-313, training.py:31-137) on
  torch CPU float64 with real nn.Linear / nn.Dropout / nn.LeakyReLU / nn.BatchNorm1d, torch.optim.Adam and
  DataLoader(shuffle=False), the loss as fit evaluates it (sum-MSE / n_cols).
"""
import numpy as np
import torch
from torch import nn

from baler_b200 import engine

DROPOUT_P = (0.5, 0.4, 0.3, 0.2)


def mt19937_from(generator=None):
    """numpy MT19937 positioned where torch's CPU generator is"""
    key, pos = engine.mt19937_from_torch_state((generator or torch.default_generator).get_state())
    g = np.random.MT19937(0)
    g.state = {"bit_generator": "MT19937", "state": {"key": key, "pos": pos}}
    return g


def bernoulli_masks(mt, rows, widths, ps=DROPOUT_P):
    """keep-masks (bool [rows, w]) of one batch in the reference's order, drawn from the numpy MT19937 `mt` (advanced)"""
    out = []
    for w, p in zip(widths, ps):
        n = rows * w
        words = mt.random_raw(2 * n).astype(np.uint64)
        r = ((words[0::2] << np.uint64(32)) | words[1::2]) & np.uint64((1 << 53) - 1)
        out.append((r.astype(np.float64) * 2.0 ** -53 < 1.0 - p).reshape(rows, w))
    return out


class DbnTwin(nn.Module):
    """reference models.py:256-313 (AE_Dropout_BN) in float64, module names as the reference's state dict"""

    def __init__(self, n_features, z_dim):
        super().__init__()
        self.enc_nn = nn.Sequential(
            nn.Linear(n_features, 200), nn.Dropout(p=0.5), nn.LeakyReLU(),
            nn.Linear(200, 100), nn.Dropout(p=0.4), nn.LeakyReLU(),
            nn.Linear(100, 50), nn.Dropout(p=0.3), nn.LeakyReLU(),
            nn.Linear(50, z_dim), nn.Dropout(p=0.2), nn.LeakyReLU())
        self.dec_nn = nn.Sequential(
            nn.Linear(z_dim, 50), nn.LeakyReLU(), nn.BatchNorm1d(50),
            nn.Linear(50, 100), nn.LeakyReLU(), nn.BatchNorm1d(100),
            nn.Linear(100, 200), nn.LeakyReLU(), nn.BatchNorm1d(200),
            nn.Linear(200, n_features), nn.BatchNorm1d(n_features), nn.ReLU())
        self.double()

    def forward(self, x):
        return self.dec_nn(self.enc_nn(x))


def twin_from_state(sd, n_features=24, z_dim=15):
    m = DbnTwin(n_features, z_dim)
    m.load_state_dict({k: torch.as_tensor(np.asarray(v)) for k, v in sd.items()})
    return m


def loss_fn(recon, x):
    return nn.functional.mse_loss(recon, x, reduction="sum") / x.shape[1]


def fit(model, opt, x, batch):
    """reference training.fit: one epoch, mean batch loss"""
    model.train()
    total, n = 0.0, 0
    for xb in torch.utils.data.DataLoader(x, batch_size=batch, shuffle=False, drop_last=False):
        opt.zero_grad()
        loss = loss_fn(model(xb), xb)
        loss.backward()
        opt.step()
        total += loss.item()
        n += 1
    return total / n


@torch.no_grad()
def validate(model, x, batch):
    """reference training.validate: eval mode, mean batch loss"""
    model.eval()
    total, n = 0.0, 0
    for xb in torch.utils.data.DataLoader(x, batch_size=batch, shuffle=False, drop_last=False):
        total += loss_fn(model(xb), xb).item()
        n += 1
    return total / n
