"""Model classes of the hot path with the reference's model protocol (reference
baler/modules/models.py): ctor `(n_features, z_dim)`, `encode / decode / forward`, `train / eval`,
`to`, `parameters`, `children`, `state_dict / load_state_dict(strict=False)`.

They are NOT torch.nn.Modules and do no torch math: the state dict (same keys, shapes and dtypes as
the reference, so `model.pt` files are interchangeable) lives on the host; `encode` / `decode`
run the fused CUDA chain of libbaler_b200 and training runs in `training.train` on a `bb_trainer`.
Initial weights are drawn with torch's own nn.Linear initialiser in the reference's construction
order, so `torch.manual_seed(s); AE(24, 15)` starts from the reference's weights.
"""
from collections import OrderedDict

import numpy as np
import torch

from .. import engine

BN_EPS = 1e-5


def _as_cuda_f32(x):
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(x)
    engine.require_cuda()
    return x.to(device="cuda", dtype=torch.float32).contiguous()


class _Layer:
    """What `model.children()` yields: a handle on one Linear's tensors (reference: nn.Linear)."""

    def __init__(self, sd, prefix):
        self._sd, self._prefix = sd, prefix

    @property
    def weight(self):
        return self._sd[self._prefix + ".weight"]

    @property
    def bias(self):
        return self._sd[self._prefix + ".bias"]


class _DenseBase:
    dtype = torch.float64
    hidden = (200, 100, 50)

    def __init__(self, n_features, z_dim, *args, **kwargs):
        self.n_features, self.z_dim = n_features, z_dim
        self.training = True
        self.activations = {}
        self._sd = OrderedDict()
        self._codec = None
        self._device = torch.device("cuda")
        self._build()

    # -- construction helpers
    def _linear(self, name, n_in, n_out):
        lin = torch.nn.Linear(n_in, n_out, dtype=self.dtype)  # consumes the RNG exactly like the reference
        self._sd[name + ".weight"] = lin.weight.detach().clone()
        self._sd[name + ".bias"] = lin.bias.detach().clone()

    # -- nn.Module-like protocol
    def state_dict(self):
        return OrderedDict((k, v.clone()) for k, v in self._sd.items())

    def load_state_dict(self, sd, strict=False):
        missing = [k for k in self._sd if k not in sd]
        unexpected = [k for k in sd if k not in self._sd]
        if strict and (missing or unexpected):
            raise RuntimeError("missing keys %s, unexpected keys %s" % (missing, unexpected))
        for k, v in sd.items():
            if k in self._sd:
                v = torch.as_tensor(v)
                if tuple(v.shape) != tuple(self._sd[k].shape):
                    raise RuntimeError("size mismatch for %s: %s vs %s" % (k, tuple(v.shape), tuple(self._sd[k].shape)))
                self._sd[k] = v.detach().to("cpu", self._sd[k].dtype).clone()
        self._codec = None
        return missing, unexpected

    def parameters(self):
        return [v for k, v in self._sd.items() if k.endswith(("weight", "bias"))]

    def named_parameters(self):
        return [(k, v) for k, v in self._sd.items() if k.endswith(("weight", "bias"))]

    def train(self, mode=True):
        self.training = bool(mode)
        return self

    def eval(self):
        return self.train(False)

    def to(self, device=None, *a, **k):
        return self

    def float(self):
        return self

    @property
    def type(self):
        return type(self).__name__

    def __call__(self, x):
        return self.forward(x)

    # -- compute
    def codec(self):
        if self._codec is None:
            enc, dec = self._chains()
            self._codec = engine.DenseCodec(enc, dec)
        return self._codec

    def _np(self, key):
        return self._sd[key].detach().cpu().numpy().astype(np.float64)

    def encode(self, x, precision="auto"):
        z = self.codec().encode(_as_cuda_f32(x).reshape(-1, self.n_features), precision=precision)
        return z.to(self.dtype)

    def decode(self, z, precision="auto"):
        y = self.codec().decode(_as_cuda_f32(z).reshape(-1, self.z_dim), precision=precision)
        return y.to(self.dtype)

    def forward(self, x):
        return self.decode(self.encode(x))


class AE(_DenseBase):
    """reference models.py:116-183 (float64 Linear stack 24-200-100-50-z and mirror, LeakyReLU between,
    none on latent / output)."""

    names = ("en1", "en2", "en3", "en4", "de1", "de2", "de3", "de4")
    latent_layer = 3  # the latent is the output of en4 (what loss_function_swae's model.encode returns)

    def _build(self):
        dims = (self.n_features,) + self.hidden + (self.z_dim,) + self.hidden[::-1] + (self.n_features,)
        for i, name in enumerate(self.names):
            self._linear(name, dims[i], dims[i + 1])

    def children(self):
        return [_Layer(self._sd, n) for n in self.names]

    def _chains(self):
        acts = ("leaky", "leaky", "leaky", "none")
        enc = [(self._np(n + ".weight"), self._np(n + ".bias"), a) for n, a in zip(self.names[:4], acts)]
        dec = [(self._np(n + ".weight"), self._np(n + ".bias"), a) for n, a in zip(self.names[4:], acts)]
        return enc, dec

    def linear_tensors(self):
        """(weights, biases) float64 ndarrays in layer order - what bb_trainer_create takes"""
        return [self._np(n + ".weight") for n in self.names], [self._np(n + ".bias") for n in self.names]

    def set_linear_tensors(self, weights, biases):
        for n, w, b in zip(self.names, weights, biases):
            self._sd[n + ".weight"] = torch.from_numpy(np.asarray(w)).to(self.dtype).clone()
            self._sd[n + ".bias"] = torch.from_numpy(np.asarray(b)).to(self.dtype).clone()
        self._codec = None

    # activation extraction (models.py:160-183): filled by training.train from the last forward
    def get_layers(self):
        return [_Layer(self._sd, n) for n in ("en1", "en2", "en3", "de1", "de2", "de3")]

    def store_hooks(self):
        self._hooks = True
        return ["hook%d" % i for i in range(6)]

    def get_activations(self):
        return self.activations

    def detach_hooks(self, hooks):
        self._hooks = False


class CFD_dense_AE(AE):
    """reference models.py:186-253: the float32 twin of AE."""

    dtype = torch.float32


class AE_Dropout_BN(_DenseBase):
    """reference models.py:256-313.  Eval mode: Dropout is the identity and BatchNorm1d is a per-feature
    affine map, folded here (float64) into the neighbouring Linear; the encoder keeps LeakyReLU on the
    latent, the decoder ends in BN -> ReLU."""

    enc_names = ("enc_nn.0", "enc_nn.3", "enc_nn.6", "enc_nn.9")
    dec_names = ("dec_nn.0", "dec_nn.3", "dec_nn.6", "dec_nn.9")
    bn_names = ("dec_nn.2", "dec_nn.5", "dec_nn.8", "dec_nn.10")
    dropout_p = (0.5, 0.4, 0.3, 0.2)

    def _build(self):
        dims = (self.n_features,) + self.hidden + (self.z_dim,)
        for i, name in enumerate(self.enc_names):
            self._linear(name, dims[i], dims[i + 1])
        ddims = dims[::-1]
        for i, name in enumerate(self.dec_names):
            self._linear(name, ddims[i], ddims[i + 1])
            n = ddims[i + 1]
            bn = self.bn_names[i]
            self._sd[bn + ".weight"] = torch.ones(n, dtype=self.dtype)
            self._sd[bn + ".bias"] = torch.zeros(n, dtype=self.dtype)
            self._sd[bn + ".running_mean"] = torch.zeros(n, dtype=self.dtype)
            self._sd[bn + ".running_var"] = torch.ones(n, dtype=self.dtype)
            self._sd[bn + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)

    def children(self):
        return ["enc_nn", "dec_nn"]

    def parameters(self):
        return [v for k, v in self._sd.items() if k.endswith((".weight", ".bias"))]

    def _chains(self):
        enc = [(self._np(n + ".weight"), self._np(n + ".bias"), "leaky") for n in self.enc_names]
        s, t = [], []
        for bn in self.bn_names:
            sc = self._np(bn + ".weight") / np.sqrt(self._np(bn + ".running_var") + BN_EPS)
            s.append(sc)
            t.append(self._np(bn + ".bias") - sc * self._np(bn + ".running_mean"))
        dec = []
        for i, n in enumerate(self.dec_names):
            w, b = self._np(n + ".weight"), self._np(n + ".bias")
            if i > 0:  # BN_{i-1} sits between LeakyReLU_{i-1} and this Linear
                b = b + w @ t[i - 1]
                w = w * s[i - 1][None, :]
            if i == 3:  # Linear -> BN -> ReLU
                w = w * s[3][:, None]
                b = b * s[3] + t[3]
            dec.append((w, b, "relu" if i == 3 else "leaky"))
        return enc, dec

    # what bb_trainer_create_dbn takes / returns
    def linear_tensors(self):
        names = self.enc_names + self.dec_names
        return [self._np(n + ".weight") for n in names], [self._np(n + ".bias") for n in names]

    def bn_tensors(self):
        out = {k: [self._np(bn + "." + k) for bn in self.bn_names] for k in ("weight", "bias", "running_mean", "running_var")}
        out["num_batches_tracked"] = [int(self._sd[bn + ".num_batches_tracked"]) for bn in self.bn_names]
        return out

    def set_linear_tensors(self, weights, biases):
        for n, w, b in zip(self.enc_names + self.dec_names, weights, biases):
            self._sd[n + ".weight"] = torch.from_numpy(np.asarray(w)).to(self.dtype).clone()
            self._sd[n + ".bias"] = torch.from_numpy(np.asarray(b)).to(self.dtype).clone()
        self._codec = None

    def set_bn_tensors(self, bn):
        for i, name in enumerate(self.bn_names):
            for k in ("weight", "bias", "running_mean", "running_var"):
                self._sd[name + "." + k] = torch.from_numpy(np.asarray(bn[k][i])).to(self.dtype).clone()
            self._sd[name + ".num_batches_tracked"] = torch.tensor(int(bn["num_batches_tracked"][i]), dtype=torch.long)
        self._codec = None

    def forward(self, x):
        if self.training:
            raise NotImplementedError("train-mode forward of AE_Dropout_BN runs inside training.train")
        return super().forward(x)

    def encode(self, x, precision="auto"):
        if self.training:
            raise NotImplementedError("train-mode forward of AE_Dropout_BN runs inside training.train")
        return super().encode(x, precision)

    def decode(self, z, precision="auto"):
        if self.training:
            raise NotImplementedError("train-mode forward of AE_Dropout_BN runs inside training.train")
        return super().decode(z, precision)


class Conv_AE:
    """reference models.py:316-407 (float32).  Only inputs whose conv stack flattens to 128 values are valid
    upstream (5x5, 3x6, 2x8 blocks: the Linear(128, 2000) is hard-coded, SURVEY F7b); `convert_to_blocks=[1,5,5]`
    is the working configuration.

    Inference here: on a fixed block shape every (transposed) convolution is a linear map of the flattened tensor,
    so the whole network is a dense chain
        encode  HW -> 8x(H+1)x(W-2) -> 16x.. (BN2d folded) -> 128 -> 2000 -> z        (ReLU after every layer)
        decode  z -> 2000 -> 128 -> 16x.. (BN folded) -> 8x.. (BN folded) -> HW      (ReLU except the output)
    whose matrices are built once on the host (float64, by pushing an identity basis through torch's own conv on
    the CPU - weight preprocessing, not the data path) and run by the CUDA GEMM chain (96 % of the FLOPs are the
    two 2000-wide Linears either way).

    Training (training.train -> engine.LayeredTrainer, bb_ltrainer_create_ex): the same chain with the convolutions
    as weight-sharing dense layers (`training_spec`: entry -> kernel-weight index maps) and BatchNorm2d on batch
    statistics; only the kernels, channel biases, Linears and BatchNorm affine parameters are trained."""

    dtype = torch.float32

    def __init__(self, n_features, z_dim, *args, **kwargs):
        nn = torch.nn
        self.n_features, self.z_dim = n_features, z_dim
        self.q_z_mid_dim, self.q_z_output_dim = 2000, 128
        self.conv_op_shape = None
        self.training = True
        # same construction order as the reference so that the RNG stream (initial weights) is identical
        mods = OrderedDict()
        mods["q_z_conv.0"] = nn.Conv2d(1, 8, kernel_size=(2, 5), stride=1, padding=1)
        mods["q_z_conv.2"] = nn.Conv2d(8, 16, kernel_size=3, stride=1, padding=1)
        mods["q_z_conv.3"] = nn.BatchNorm2d(16)
        mods["q_z_conv.5"] = nn.Conv2d(16, 32, kernel_size=3, stride=1, padding=0)
        mods["q_z_lin.0"] = nn.Linear(self.q_z_output_dim, self.q_z_mid_dim)
        mods["q_z_lin.2"] = nn.Linear(self.q_z_mid_dim, z_dim)
        mods["p_x_lin.0"] = nn.Linear(z_dim, self.q_z_mid_dim)
        mods["p_x_lin.2"] = nn.Linear(self.q_z_mid_dim, self.q_z_output_dim)
        mods["p_x_conv.0"] = nn.ConvTranspose2d(32, 16, kernel_size=3, stride=1, padding=0)
        mods["p_x_conv.1"] = nn.BatchNorm2d(16)
        mods["p_x_conv.3"] = nn.ConvTranspose2d(16, 8, kernel_size=3, stride=1, padding=1)
        mods["p_x_conv.4"] = nn.BatchNorm2d(8)
        mods["p_x_conv.6"] = nn.ConvTranspose2d(8, 1, kernel_size=(2, 5), stride=1, padding=1)
        self._sd = OrderedDict()
        for name, m in mods.items():
            for k, v in m.state_dict().items():
                self._sd[name + "." + k] = v.detach().clone()
        self._codec, self._codec_hw = None, None

    # -- nn.Module-like protocol (same as the dense models)
    state_dict = _DenseBase.state_dict
    load_state_dict = _DenseBase.load_state_dict
    train = _DenseBase.train
    eval = _DenseBase.eval
    to = _DenseBase.to
    __call__ = _DenseBase.__call__

    def parameters(self):
        return [v for k, v in self._sd.items() if k.endswith((".weight", ".bias"))]

    def children(self):
        return ["q_z_conv", "flatten", "q_z_lin", "p_x_lin", "p_x_conv"]

    def get_final_layer_dims(self):
        return self.conv_op_shape

    def set_final_layer_dims(self, conv_op_shape):
        self.conv_op_shape = conv_op_shape

    # -- dense-equivalent chains for a block shape (h, w)
    def _t(self, key):
        return self._sd[key].detach().to(torch.float64)

    def _bn(self, name):
        s = self._t(name + ".weight") / torch.sqrt(self._t(name + ".running_var") + BN_EPS)
        return s, self._t(name + ".bias") - s * self._t(name + ".running_mean")

    @staticmethod
    def _as_matrix(fn, in_shape):
        """dense (out, in) matrix and bias of the affine map `fn` on tensors of shape in_shape"""
        n_in = int(np.prod(in_shape))
        with torch.no_grad():
            b = fn(torch.zeros((1,) + in_shape, dtype=torch.float64))
            out_shape = tuple(b.shape[1:])
            m = fn(torch.eye(n_in, dtype=torch.float64).reshape((n_in,) + in_shape)) - b
        return m.reshape(n_in, -1).T.contiguous().numpy(), b.reshape(-1).numpy(), out_shape

    def _chains(self, h, w):
        F = torch.nn.functional

        def chan_affine(mat, bias, shape, s, t):  # per-channel y * s + t on a flattened (C, H, W) output
            rep = shape[1] * shape[2]
            sv, tv = s.repeat_interleave(rep).numpy(), t.repeat_interleave(rep).numpy()
            return mat * sv[:, None], bias * sv + tv

        # the conv stack's output shape, before any matrix is built (a 50x50 snapshot would ask for a 100 GB identity basis):
        # (2,5) kernel pad 1 -> (h + 1, w - 2); 3x3 pad 1 keeps it; 3x3 pad 0 -> (h - 1, w - 4), 32 channels
        flat = 32 * max(h - 1, 0) * max(w - 4, 0)
        if flat != self.q_z_output_dim:
            raise RuntimeError("Conv_AE: a %dx%d block flattens to %d values, the model's Linear expects %d "
                               "(reference models.py:320-343)" % (h, w, flat, self.q_z_output_dim))
        enc, shape = [], (1, h, w)
        m, b, shape = self._as_matrix(lambda x: F.conv2d(x, self._t("q_z_conv.0.weight"), self._t("q_z_conv.0.bias"), padding=1), shape)
        enc.append((m, b, "relu"))
        m, b, shape = self._as_matrix(lambda x: F.conv2d(x, self._t("q_z_conv.2.weight"), self._t("q_z_conv.2.bias"), padding=1), shape)
        m, b = chan_affine(m, b, shape, *self._bn("q_z_conv.3"))
        enc.append((m, b, "relu"))
        m, b, shape = self._as_matrix(lambda x: F.conv2d(x, self._t("q_z_conv.5.weight"), self._t("q_z_conv.5.bias"), padding=0), shape)
        enc.append((m, b, "relu"))
        conv_out = shape
        assert int(np.prod(shape)) == flat
        enc.append((self._t("q_z_lin.0.weight").numpy(), self._t("q_z_lin.0.bias").numpy(), "relu"))
        enc.append((self._t("q_z_lin.2.weight").numpy(), self._t("q_z_lin.2.bias").numpy(), "relu"))
        dec = [(self._t("p_x_lin.0.weight").numpy(), self._t("p_x_lin.0.bias").numpy(), "relu"),
               (self._t("p_x_lin.2.weight").numpy(), self._t("p_x_lin.2.bias").numpy(), "relu")]
        shape = conv_out
        m, b, shape = self._as_matrix(lambda x: F.conv_transpose2d(x, self._t("p_x_conv.0.weight"), self._t("p_x_conv.0.bias"), padding=0), shape)
        m, b = chan_affine(m, b, shape, *self._bn("p_x_conv.1"))
        dec.append((m, b, "relu"))
        m, b, shape = self._as_matrix(lambda x: F.conv_transpose2d(x, self._t("p_x_conv.3.weight"), self._t("p_x_conv.3.bias"), padding=1), shape)
        m, b = chan_affine(m, b, shape, *self._bn("p_x_conv.4"))
        dec.append((m, b, "relu"))
        m, b, shape = self._as_matrix(lambda x: F.conv_transpose2d(x, self._t("p_x_conv.6.weight"), self._t("p_x_conv.6.bias"), padding=1), shape)
        dec.append((m, b, "none"))
        return enc, dec, conv_out

    # -- training: the chain as weight-sharing dense layers
    _CONV = [("q_z_conv.0", "conv", 1, None), ("q_z_conv.2", "conv", 1, "q_z_conv.3"), ("q_z_conv.5", "conv", 0, None),
             ("q_z_lin.0", "lin", 0, None), ("q_z_lin.2", "lin", 0, None), ("p_x_lin.0", "lin", 0, None),
             ("p_x_lin.2", "lin", 0, None), ("p_x_conv.0", "convT", 0, "p_x_conv.1"), ("p_x_conv.3", "convT", 1, "p_x_conv.4"),
             ("p_x_conv.6", "convT", 1, None)]
    latent_layer = [c[0] for c in _CONV].index("q_z_lin.2")  # training_spec layer whose output model.encode returns

    def training_spec(self, h=5, w=5):
        """dict(dims, acts, weights, biases, w_maps, bn) for engine.LayeredTrainer.  w_maps[l][i] is the flat index of the
        kernel weight that dense entry i of layer l repeats (-1: structural zero), found by pushing an identity basis
        through torch's own (transposed) convolution with the kernel entries replaced by their 1-based flat indices: at
        stride 1 every (output, input) pair meets at most one kernel entry."""
        F = torch.nn.functional
        flat = 32 * max(h - 1, 0) * max(w - 4, 0)  # as in _chains: refuse before any identity basis is built
        if flat != self.q_z_output_dim:
            raise RuntimeError("Conv_AE: a %dx%d block flattens to %d values, the model's Linear expects %d "
                               "(reference models.py:320-343)" % (h, w, flat, self.q_z_output_dim))
        dims, acts, weights, biases, maps, bn = [h * w], [], [], [], [], []
        shape = (1, h, w)
        for i, (name, kind, pad, bn_name) in enumerate(self._CONV):
            wt, bs = self._t(name + ".weight"), self._t(name + ".bias")
            if kind == "lin":
                if dims[-1] != wt.shape[1]:
                    raise RuntimeError("Conv_AE: a %dx%d block flattens to %d values, the model's Linear expects %d "
                                       "(reference models.py:320-343)" % (h, w, dims[-1], wt.shape[1]))
                weights.append(wt.numpy()); biases.append(bs.numpy()); maps.append(None)
                dims.append(wt.shape[0])
                if name == "q_z_lin.0":
                    conv_out = shape
                if name == "p_x_lin.2":
                    shape = conv_out
            else:
                op = F.conv2d if kind == "conv" else F.conv_transpose2d
                codes = torch.arange(1, wt.numel() + 1, dtype=torch.float64).reshape(wt.shape)
                m, _, shape = self._as_matrix(lambda x: op(x, codes, None, padding=pad), shape)
                maps.append(np.rint(m).astype(np.int32).reshape(-1) - 1)
                weights.append(wt.reshape(-1).numpy()); biases.append(bs.numpy())
                dims.append(int(np.prod(shape)))
            acts.append("none" if i == len(self._CONV) - 1 else "relu")
            bn.append(None if bn_name is None else np.stack([self._t(bn_name + "." + k).numpy()
                                                             for k in ("weight", "bias", "running_mean", "running_var")]))
        self._conv_out = conv_out
        return dict(dims=dims, acts=acts, weights=weights, biases=biases, w_maps=maps, bn=bn)

    def load_trained(self, weights, biases, bn, steps):
        """write the trainer's parameters (training_spec order) back into the state_dict; `steps` batches were counted
        (num_batches_tracked): one count for every BatchNorm, or one per training_spec layer"""
        steps = np.broadcast_to(np.asarray(steps, dtype=np.int64), (len(self._CONV),))
        for (name, kind, pad, bn_name), wt, bs, b4, n in zip(self._CONV, weights, biases, bn, steps):
            dt = self._sd[name + ".weight"].dtype
            self._sd[name + ".weight"] = torch.from_numpy(np.asarray(wt)).reshape(self._sd[name + ".weight"].shape).to(dt)
            self._sd[name + ".bias"] = torch.from_numpy(np.asarray(bs)).reshape(-1).to(dt)
            if bn_name is not None:
                for k, row in zip(("weight", "bias", "running_mean", "running_var"), b4):
                    self._sd[bn_name + "." + k] = torch.from_numpy(np.asarray(row)).to(dt)
                self._sd[bn_name + ".num_batches_tracked"] = self._sd[bn_name + ".num_batches_tracked"] + int(n)
        self._codec = None

    def codec(self, h=5, w=5):
        if self._codec is None or self._codec_hw != (h, w):
            enc, dec, conv_out = self._chains(h, w)
            self._codec, self._codec_hw, self._conv_out = engine.DenseCodec(enc, dec), (h, w), conv_out
        return self._codec

    def encode(self, x, precision="auto"):
        if self.training:
            raise NotImplementedError("the train-mode forward of Conv_AE (batch statistics) runs inside training.train")
        x = _as_cuda_f32(x)
        h, w = x.shape[-2], x.shape[-1]
        z = self.codec(h, w).encode(x.reshape(-1, h * w), precision=precision)
        self.conv_op_shape = torch.Size((z.shape[0],) + self._conv_out)
        return z

    def decode(self, z, precision="auto"):
        if self.training:
            raise NotImplementedError("the train-mode forward of Conv_AE (batch statistics) runs inside training.train")
        h, w = self._codec_hw if self._codec_hw else (5, 5)
        y = self.codec(h, w).decode(_as_cuda_f32(z).reshape(-1, self.z_dim), precision=precision)
        return y.reshape(-1, 1, h, w)  # any batch size: the reference's view() to the LAST TRAINING batch (F7c) is not reproduced

    def forward(self, x):
        return self.decode(self.encode(x))
