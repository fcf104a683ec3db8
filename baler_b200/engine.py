"""Thin Python host side over the C ABI: device memory and streams come from torch, every FLOP of the
path runs in libbaler_b200.so.  Nothing here falls back to torch math."""
import ctypes as C

import numpy as np
import torch

from . import _lib, latent_q8
from ._lib import BB_ACT_LEAKY, BB_ACT_NONE, BB_ACT_RELU, BB_F16, BB_F32, BB_F64, BB_PREC_FP64, PRECISIONS, check

_NP2BB = {np.dtype(np.float32): BB_F32, np.dtype(np.float16): BB_F16, np.dtype(np.float64): BB_F64}
_T2BB = {torch.float32: BB_F32, torch.float16: BB_F16, torch.float64: BB_F64}
# shapes the float64 chain takes (precision "fp64"; include/baler_b200.h, BB_PREC_FP64)
FP64_MAX_LAYERS, FP64_MAX_WIDTH = 8, 256
_contexts = {}


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("baler_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


class Context:
    """bb_ctx for one CUDA device (replaces helper.get_device, reference helper.py:425-439)."""

    def __init__(self, index):
        require_cuda()
        self.index = index
        self.handle = C.c_void_p()
        check(_lib.lib().bb_ctx_create(index, C.byref(self.handle)), "bb_ctx_create")
        self.sm_count = _lib.lib().bb_ctx_sm_count(self.handle)
        self.device = torch.device("cuda", index)


def get_context(device=None):
    require_cuda()
    if device is None:
        index = torch.cuda.current_device()
    else:
        device = torch.device(device)
        index = device.index if device.index is not None else torch.cuda.current_device()
    if index not in _contexts:
        _contexts[index] = Context(index)
    return _contexts[index]


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(ctx):
    return C.c_void_p(torch.cuda.current_stream(ctx.device).cuda_stream)


def _host_ptrs(arrays):
    """ctypes array of pointers to contiguous float64 host arrays (kept alive by the caller)"""
    arr = (C.c_void_p * len(arrays))()
    for i, a in enumerate(arrays):
        arr[i] = a.ctypes.data
    return arr


def _prec(precision):
    if isinstance(precision, str):
        return PRECISIONS[precision]
    return int(precision)


def host_convert(a, dtype):
    """C-contiguous array `a` as float32 / float64 - ndarray.astype with the conversion done on the library's worker threads
    (bb_host_convert: float32 -> float64 exact, float64 -> float32 round-to-nearest-even, the bits astype gives; numpy does
    it on one thread, ~7 s for a 100M x 24 float64 file).  Other dtype pairs, small or strided arrays go through numpy."""
    a = np.asarray(a)
    dtype = np.dtype(dtype)
    pair = {(np.dtype(np.float32), np.dtype(np.float64)): (BB_F32, BB_F64),
            (np.dtype(np.float64), np.dtype(np.float32)): (BB_F64, BB_F32)}.get((a.dtype, dtype))
    if a.dtype == dtype:
        return np.ascontiguousarray(a)
    if pair is None or not a.flags.c_contiguous or a.size < (1 << 16):
        return np.ascontiguousarray(a, dtype=dtype)
    out = np.empty(a.shape, dtype=dtype)
    check(_lib.lib().bb_host_convert(a.ctypes.data, pair[0], out.ctypes.data, pair[1], a.size), "bb_host_convert")
    return out


def colminmax(x, ctx=None):
    """per-column (min, max) of a row-major CUDA float32 or float64 table -> two CUDA vectors of the table's dtype"""
    ctx = ctx or get_context(x.device)
    assert x.is_cuda and x.dtype in (torch.float32, torch.float64) and x.dim() == 2 and x.is_contiguous()
    mn = torch.empty(x.shape[1], dtype=x.dtype, device=x.device)
    mx = torch.empty_like(mn)
    name = "bb_colminmax_f64" if x.dtype == torch.float64 else "bb_colminmax_f32"
    check(getattr(_lib.lib(), name)(ctx.handle, _ptr(x), x.shape[0], x.shape[1], _ptr(mn), _ptr(mx), _stream(ctx)), name)
    return mn, mx


def _host_table(x, window_rows, batch):
    """(pointer, BB dtype) of a C-contiguous 2-D float32 / float64 numpy table streamed through device windows of
    `window_rows` rows (bb_*_epoch_host: a positive multiple of the batch)"""
    if not (isinstance(x, np.ndarray) and x.ndim == 2 and x.flags.c_contiguous and x.dtype in (np.float32, np.float64)):
        raise ValueError("a host table is a C-contiguous 2-D float32 / float64 numpy array")
    if window_rows is None or window_rows < batch or window_rows % batch:
        raise ValueError("window_rows must be a positive multiple of the batch (%d), not %r" % (batch, window_rows))
    return x.ctypes.data, _NP2BB[x.dtype]


def fp64_refusal(chains):
    """None when the float64 kernel takes every chain in `chains` ({name: [width of each layer boundary]}), else the
    message of the NotImplementedError precision "fp64" raises for it"""
    for name, dims in chains.items():
        if len(dims) - 1 > FP64_MAX_LAYERS or max(dims) > FP64_MAX_WIDTH:
            return ("precision='fp64' takes dense chains of at most %d layers with every width <= %d; the %s is %s"
                    % (FP64_MAX_LAYERS, FP64_MAX_WIDTH, name, "-".join(str(d) for d in dims)))
    return None


def normalize_table(x, mn, rg, inverse=False, out=None, ctx=None):
    """(x - min) / range, or x * range + min when inverse, on a CUDA float32 table"""
    ctx = ctx or get_context(x.device)
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
    out = torch.empty_like(x) if out is None else out
    c = x.shape[-1]
    fn = _lib.lib().bb_renormalize_f32 if inverse else _lib.lib().bb_normalize_f32
    check(fn(ctx.handle, _ptr(x), x.numel() // c, c, _ptr(mn), _ptr(rg), _ptr(out), _stream(ctx)), "bb_(re)normalize_f32")
    return out


def normalize_table_f64(x, mn, rg, out=None, ctx=None):
    """(x - min) / range on a CUDA float64 table, one IEEE subtract and divide per element (bit-equal to numpy)"""
    ctx = ctx or get_context(x.device)
    assert x.is_cuda and x.dtype == torch.float64 and x.is_contiguous()
    assert mn.dtype == rg.dtype == torch.float64 and mn.is_contiguous() and rg.is_contiguous()
    out = torch.empty_like(x) if out is None else out
    c = x.shape[-1]
    check(_lib.lib().bb_normalize_f64(ctx.handle, _ptr(x), x.numel() // c, c, _ptr(mn), _ptr(rg), _ptr(out), _stream(ctx)),
          "bb_normalize_f64")
    return out


def mse_sum(a, b, ctx=None):
    """sum((a - b)^2) of two CUDA float32 tensors -> python float (one device->host read)"""
    ctx = ctx or get_context(a.device)
    out = torch.zeros(1, dtype=torch.float64, device=a.device)
    check(_lib.lib().bb_mse_sum_f32(ctx.handle, _ptr(a), _ptr(b), a.numel(), _ptr(out), _stream(ctx)), "bb_mse_sum_f32")
    return float(out.item())


class DenseCodec:
    """Packed encoder + decoder of one dense autoencoder (bb_model).

    enc_layers / dec_layers: lists of (weight (out, in) float64, bias (out,) float64, act) with
    act in {"none", "leaky", "relu"}; eval-mode BatchNorm already folded by the caller."""

    _ACT = {"none": BB_ACT_NONE, "leaky": BB_ACT_LEAKY, "relu": BB_ACT_RELU}

    def __init__(self, enc_layers, dec_layers, device=None):
        self.ctx = get_context(device)
        self.handle = C.c_void_p()
        keep, widths = [], []

        def pack(layers):
            w = [np.ascontiguousarray(l[0], dtype=np.float64) for l in layers]
            b = [np.ascontiguousarray(l[1], dtype=np.float64) for l in layers]
            widths.append([w[0].shape[1]] + [x.shape[0] for x in w])
            dims = (C.c_int * (len(layers) + 1))(*widths[-1])
            acts = (C.c_int * len(layers))(*[self._ACT[l[2]] for l in layers])
            keep.extend(w + b)
            return len(layers), dims, acts, _host_ptrs(w), _host_ptrs(b)

        ne, ed, ea, ew, eb = pack(enc_layers)
        nd, dd, da, dw, db = pack(dec_layers)
        with torch.cuda.device(self.ctx.device):
            check(_lib.lib().bb_model_create_dense(self.ctx.handle, ne, ed, ea, ew, eb, nd, dd, da, dw, db,
                                                   C.byref(self.handle)), "bb_model_create_dense")
        self.n_features = _lib.lib().bb_model_n_features(self.handle)
        self.z_dim = _lib.lib().bb_model_z_dim(self.handle)
        self.widths = {"encoder": widths[0], "decoder": widths[1]}

    def require_fp64(self, precision="fp64"):
        """True for precision "fp64" (raises NotImplementedError when the float64 kernel does not take this model's
        chains), False for the other precisions"""
        if _prec(precision) != _lib.BB_PREC_FP64:
            return False
        msg = fp64_refusal(self.widths)
        if msg:
            raise NotImplementedError(msg)
        return True

    def _fp64_input(self, precision):
        """float64 inputs run the float64 chain: precision "auto" or "fp64" """
        if _prec(precision) not in (_lib.BB_PREC_AUTO, _lib.BB_PREC_FP64):
            raise ValueError("float64 tensors run on precision 'fp64' only")
        self.require_fp64()

    def __del__(self):
        try:
            if getattr(self, "handle", None) and self.handle.value:
                _lib.lib().bb_model_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    def trim(self):
        """release the scratch the host pipelines keep between calls (resident table copy, pinned bounce buffers)"""
        check(_lib.lib().bb_model_trim(self.handle), "bb_model_trim")

    @property
    def auto_precision(self):
        return {v: k for k, v in PRECISIONS.items() if k in ("fp32", "split16")}[
            _lib.lib().bb_model_auto_precision(self.handle)]

    def range_flag(self, reset=True):
        """sticky fp16-range flag of the split16 path (synchronises the device)"""
        flag = C.c_int(0)
        check(_lib.lib().bb_model_range_flag(self.handle, int(reset), C.byref(flag)), "bb_model_range_flag")
        return bool(flag.value)

    def _guarded(self, launch, precision, check_range, direction):
        """run `launch(precision)`; with precision "auto" on a chain (direction 0 encoder, 1 decoder) that resolves to the
        tensor-core path, re-run on the fp32 kernel if a value left the fp16 range (costs one 4-byte device->host read;
        pass check_range=False to stay async)"""
        launch(_prec(precision))
        if (check_range and _prec(precision) == _lib.BB_PREC_AUTO
                and _lib.lib().bb_model_chain_precision(self.handle, direction) == _lib.BB_PREC_SPLIT16 and self.range_flag()):
            launch(_lib.BB_PREC_FP32)

    # ---- device-resident tensors
    def encode(self, x, fmin=None, frange=None, out_dtype=torch.float32, precision="auto", out=None, check_range=True):
        """z = encode((x - fmin) / frange).  A float64 `x` (with float64 fmin / frange) runs the float64 chain and gives a
        float64 latent; precision "fp64" runs it on a float32 `x`, normalised in float32 first (out_dtype may be float64)."""
        assert x.is_cuda and x.dtype in (torch.float32, torch.float64) and x.is_contiguous() and x.shape[-1] == self.n_features
        n = x.numel() // self.n_features
        if x.dtype == torch.float64:
            self._fp64_input(precision)
            assert fmin is None or (fmin.dtype == frange.dtype == torch.float64)
            z = out if out is not None else torch.empty((n, self.z_dim), dtype=torch.float64, device=x.device)
            assert z.dtype == torch.float64
            check(_lib.lib().bb_encode_f64(self.handle, _ptr(x), n, _ptr(fmin), _ptr(frange), _ptr(z), _stream(self.ctx)),
                  "bb_encode_f64")
            return z
        self.require_fp64(precision)
        z = out if out is not None else torch.empty((n, self.z_dim), dtype=out_dtype, device=x.device)
        self._guarded(lambda p: check(_lib.lib().bb_encode_f32(
            self.handle, _ptr(x), n, _ptr(fmin), _ptr(frange), _ptr(z), _T2BB[z.dtype], p, _stream(self.ctx)),
            "bb_encode_f32"), precision, check_range, 0)
        return z

    def decode(self, z, fmin=None, frange=None, precision="auto", out=None, check_range=True):
        """y = decode(z) * frange + fmin.  A float64 `z` runs the float64 chain and gives float64 rows (float32 features
        are widened exactly); precision "fp64" runs it on a float32 / float16 `z` with float32 rows out."""
        assert z.is_cuda and z.dtype in _T2BB and z.is_contiguous() and z.shape[-1] == self.z_dim
        n = z.numel() // self.z_dim
        if z.dtype == torch.float64:
            self._fp64_input(precision)
            if fmin is not None:
                fmin, frange = fmin.to(torch.float64).contiguous(), frange.to(torch.float64).contiguous()
            y = out if out is not None else torch.empty((n, self.n_features), dtype=torch.float64, device=z.device)
            assert y.dtype == torch.float64
            check(_lib.lib().bb_decode_f64(self.handle, _ptr(z), n, _ptr(fmin), _ptr(frange), _ptr(y), _stream(self.ctx)),
                  "bb_decode_f64")
            return y
        self.require_fp64(precision)
        y = out if out is not None else torch.empty((n, self.n_features), dtype=torch.float32, device=z.device)
        self._guarded(lambda p: check(_lib.lib().bb_decode_f32(
            self.handle, _ptr(z), _T2BB[z.dtype], n, _ptr(fmin), _ptr(frange), _ptr(y), p, _stream(self.ctx)),
            "bb_decode_f32"), precision, check_range, 1)
        return y

    # ---- host buffers (numpy), chunked copy/compute pipeline inside the library
    def compress_host(self, x, features=None, recompute_minmax=False, z_dtype=np.float32, precision="auto", out=None):
        """x: (n, F) float32 ndarray.  features: None (no normalisation) or (2, F) float32 [min; range]
        (overwritten when recompute_minmax).  Returns (z, features).
        precision "fp64": the float64 chain; a float32 table is normalised in float32 as above, any other table in
        float64 with (2, F) float64 features (bb_compress_host_f64, float64 latent)."""
        if self.require_fp64(precision) and np.asarray(x).dtype != np.float32:
            return self._compress_host_f64(x, features, recompute_minmax, z_dtype, out)
        x = host_convert(x, np.float32)  # (float64 tables: narrowed on the worker threads)
        n = x.shape[0]
        z = out if out is not None else np.empty((n, self.z_dim), dtype=z_dtype)
        feats = None
        if features is not None or recompute_minmax:
            feats = np.zeros((2, self.n_features), dtype=np.float32) if features is None else \
                np.ascontiguousarray(features, dtype=np.float32).copy()
        check(_lib.lib().bb_compress_host(self.handle, x.ctypes.data, n,
                                          None if feats is None else feats.ctypes.data, int(bool(recompute_minmax)),
                                          z.ctypes.data, _NP2BB[z.dtype], _prec(precision)), "bb_compress_host")
        return z, feats

    def _compress_host_f64(self, x, features, recompute_minmax, z_dtype, out):
        """float64 table: float64 features and latent (narrowed on the host when z_dtype asks for less)"""
        x = host_convert(x, np.float64)
        n = x.shape[0]
        z = out if out is not None else np.empty((n, self.z_dim), dtype=np.float64)
        assert z.dtype == np.float64 and z.flags.c_contiguous
        feats = None
        if features is not None or recompute_minmax:
            feats = np.zeros((2, self.n_features), dtype=np.float64) if features is None else \
                np.ascontiguousarray(features, dtype=np.float64).copy()
        check(_lib.lib().bb_compress_host_f64(self.handle, x.ctypes.data, n, None if feats is None else feats.ctypes.data,
                                              int(bool(recompute_minmax)), z.ctypes.data), "bb_compress_host_f64")
        return (z if out is not None else host_convert(z, z_dtype)), feats

    def decompress_host(self, z, features=None, y_dtype=np.float64, precision="auto", out=None):
        """z: (n, z_dim) ndarray, features None or (2, F) [min; range] of the table (float32).  Returns y of y_dtype.
        precision "fp64": the float64 chain; float64 features (a float64 table's) run bb_decompress_host_f64."""
        if (self.require_fp64(precision) and features is not None and np.asarray(features).dtype == np.float64):
            z = host_convert(z, np.float64)
            n = z.shape[0]
            y = out if out is not None else np.empty((n, self.n_features), dtype=np.float64)
            assert y.dtype == np.float64 and y.flags.c_contiguous
            feats = np.ascontiguousarray(features, dtype=np.float64)
            check(_lib.lib().bb_decompress_host_f64(self.handle, z.ctypes.data, n, feats.ctypes.data, y.ctypes.data),
                  "bb_decompress_host_f64")
            return y if out is not None else host_convert(y, y_dtype)
        z = np.ascontiguousarray(z)
        n = z.shape[0]
        y = out if out is not None else np.empty((n, self.n_features), dtype=y_dtype)
        feats = None if features is None else np.ascontiguousarray(features, dtype=np.float32)
        check(_lib.lib().bb_decompress_host(self.handle, z.ctypes.data, _NP2BB[z.dtype], n,
                                            None if feats is None else feats.ctypes.data, y.ctypes.data,
                                            _NP2BB[y.dtype], _prec(precision)), "bb_decompress_host")
        return y

    # ---- quantised latent (latent_q8: b-bit codes in packed rows, float32 lo / step per 128-row block and column); the
    # *_q8 methods are the b = 8 calls, with Q8Latent in place of PackedLatent
    def quantize_packed(self, z, bits):
        """PackedLatent of CUDA tensors for a CUDA float32 latent [n, z_dim]; blocks start at its row 0"""
        assert z.is_cuda and z.dtype == torch.float32 and z.is_contiguous() and z.shape[-1] == self.z_dim
        n = z.numel() // self.z_dim
        nb = latent_q8.n_blocks(n)
        q = latent_q8.PackedLatent(torch.empty((n, latent_q8.row_bytes(self.z_dim, bits)), dtype=torch.uint8, device=z.device),
                                   torch.empty((nb, self.z_dim), dtype=torch.float32, device=z.device),
                                   torch.empty((nb, self.z_dim), dtype=torch.float32, device=z.device), int(bits))
        check(_lib.lib().bb_latent_quantize_packed(self.ctx.handle, _ptr(z), n, self.z_dim, q.bits, _ptr(q.codes), _ptr(q.lo),
                                                   _ptr(q.step), _stream(self.ctx)), "bb_latent_quantize_packed")
        return q

    def dequantize_packed(self, q):
        """the CUDA float32 latent [n, z_dim] of a PackedLatent of CUDA tensors"""
        codes, lo, step = (t.contiguous() for t in q[:3])
        n = codes.shape[0]
        assert codes.is_cuda and codes.dtype == torch.uint8 and codes.shape == (n, latent_q8.row_bytes(self.z_dim, q.bits))
        assert lo.dtype == step.dtype == torch.float32 and lo.shape == step.shape == (latent_q8.n_blocks(n), self.z_dim)
        z = torch.empty((n, self.z_dim), dtype=torch.float32, device=codes.device)
        check(_lib.lib().bb_latent_dequantize_packed(self.ctx.handle, q.bits, _ptr(codes), _ptr(lo), _ptr(step), n, self.z_dim,
                                                     _ptr(z), _stream(self.ctx)), "bb_latent_dequantize_packed")
        return z

    def compress_host_packed(self, x, bits, features=None, recompute_minmax=False, precision="auto", out=None):
        """compress_host with the `bits`-bit latent (bb_compress_host_packed): returns (PackedLatent of numpy arrays,
        features).  `out`: a PackedLatent of host buffers to fill (latent_q8.empty_packed).  precision "fp64" is refused."""
        if _prec(precision) == BB_PREC_FP64:
            raise NotImplementedError("precision='fp64' does not write a quantised latent (latent_dtype='q%d'): the %d-bit "
                                      "codes discard far more than float64 arithmetic gains" % (bits, bits))
        x = host_convert(x, np.float32)
        n = x.shape[0]
        q = out if out is not None else latent_q8.empty_packed(n, self.z_dim, bits)
        feats = None
        if features is not None or recompute_minmax:
            feats = np.zeros((2, self.n_features), dtype=np.float32) if features is None else \
                np.ascontiguousarray(features, dtype=np.float32).copy()
        check(_lib.lib().bb_compress_host_packed(self.handle, x.ctypes.data, n, None if feats is None else feats.ctypes.data,
                                                 int(bool(recompute_minmax)), int(bits), q.codes.ctypes.data, q.lo.ctypes.data,
                                                 q.step.ctypes.data, _prec(precision)), "bb_compress_host_packed")
        return q, feats

    def decompress_host_packed(self, q, features=None, y_dtype=np.float64, precision="auto", out=None):
        """decompress_host of a PackedLatent of numpy arrays (bb_decompress_host_packed): dequantised and decoded on the
        device"""
        if _prec(precision) == BB_PREC_FP64:
            raise NotImplementedError("precision='fp64' does not read a quantised latent (latent_dtype='q%d')" % q.bits)
        codes, lo, step = (np.ascontiguousarray(a) for a in q[:3])
        n, width = codes.shape[0], latent_q8.row_bytes(self.z_dim, q.bits)
        if codes.dtype != np.uint8 or codes.shape[1:] != (width,) or lo.dtype != np.float32 or step.dtype != np.float32 \
                or lo.shape != (latent_q8.n_blocks(n), self.z_dim) or step.shape != lo.shape:
            raise ValueError("a q%d latent of %d rows is uint8 codes (%d, %d) and float32 lo / step (%d, %d)"
                             % (q.bits, n, n, width, latent_q8.n_blocks(n), self.z_dim))
        y = out if out is not None else np.empty((n, self.n_features), dtype=y_dtype)
        feats = None if features is None else np.ascontiguousarray(features, dtype=np.float32)
        check(_lib.lib().bb_decompress_host_packed(self.handle, int(q.bits), codes.ctypes.data, lo.ctypes.data,
                                                   step.ctypes.data, n, None if feats is None else feats.ctypes.data,
                                                   y.ctypes.data, _NP2BB[y.dtype], _prec(precision)),
              "bb_decompress_host_packed")
        return y

    def quantize_q8(self, z):
        """Q8Latent of CUDA tensors for a CUDA float32 latent [n, z_dim]; blocks start at its row 0"""
        return latent_q8.Q8Latent(*self.quantize_packed(z, 8)[:3])

    def dequantize_q8(self, q):
        """the CUDA float32 latent [n, z_dim] of a Q8Latent of CUDA tensors"""
        return self.dequantize_packed(latent_q8.PackedLatent(*q, 8))

    def compress_host_q8(self, x, features=None, recompute_minmax=False, precision="auto", out=None):
        """compress_host with the 8-bit latent (bb_compress_host_q8): returns (Q8Latent of numpy arrays, features).
        `out`: a Q8Latent of host buffers to fill (latent_q8.empty).  precision "fp64" is refused."""
        q, feats = self.compress_host_packed(x, 8, features, recompute_minmax, precision,
                                             None if out is None else latent_q8.PackedLatent(*out, 8))
        return latent_q8.Q8Latent(*q[:3]), feats

    def decompress_host_q8(self, q, features=None, y_dtype=np.float64, precision="auto", out=None):
        """decompress_host of a Q8Latent of numpy arrays (bb_decompress_host_q8): dequantised and decoded on the device"""
        return self.decompress_host_packed(latent_q8.PackedLatent(*q, 8), features, y_dtype, precision, out)


# torch's CPU generator state (torch.Generator.get_state(), 5056 bytes): the MT19937 engine as
# {uint64 seed, int32 left, int32 seeded, uint64 next, uint64 state[624]} followed by the cached normal samples.
# The next word is state[next] unless left == 1, when the engine twists first: numpy's position 624 - (left - 1).
_MT_LEFT, _MT_NEXT, _MT_KEY = 8, 16, 24
_MT_STATE_BYTES = 5056


def mt19937_from_torch_state(blob):
    """(key uint32[624], position 0..624) of a torch CPU generator state"""
    b = blob.numpy().tobytes()
    if len(b) != _MT_STATE_BYTES:
        raise ValueError("not a torch CPU generator state (%d bytes, expected %d)" % (len(b), _MT_STATE_BYTES))
    left = int(np.frombuffer(b, np.int32, 1, _MT_LEFT)[0])
    key = np.frombuffer(b, np.uint64, 624, _MT_KEY).astype(np.uint32)
    return key, 624 - (left - 1)


def mt19937_to_torch_state(blob, key, pos):
    """`blob` with its MT19937 key and position replaced (everything else, e.g. the seed and the normal cache, kept)"""
    b = bytearray(blob.numpy().tobytes())
    if len(b) != _MT_STATE_BYTES or not 0 <= pos <= 624:
        raise ValueError("bad torch CPU generator state or position")
    b[_MT_LEFT:_MT_LEFT + 4] = np.int32(625 - pos).tobytes()
    b[_MT_NEXT:_MT_NEXT + 8] = np.uint64(pos % 624).tobytes()
    b[_MT_KEY:_MT_KEY + 8 * 624] = np.asarray(key, dtype=np.uint32).astype(np.uint64).tobytes()
    return torch.frombuffer(b, dtype=torch.uint8).clone()


class Trainer:
    """bb_trainer: parameters, Adam state and scratch of one dense-AE training run on one GPU."""

    def __init__(self, weights, biases, n_features, z_dim, max_batch, device=None, bn=None):
        """bn: None for AE / CFD_dense_AE; for AE_Dropout_BN a dict with lists of 4 arrays `weight`, `bias`,
        `running_mean`, `running_var` and `num_batches_tracked` (4 ints)"""
        self.ctx = get_context(device)
        self.handle = C.c_void_p()
        self._w = [np.ascontiguousarray(w, dtype=np.float64) for w in weights]
        self._b = [np.ascontiguousarray(b, dtype=np.float64) for b in biases]
        self._bn = None
        self._masks = None
        with torch.cuda.device(self.ctx.device):
            if bn is None:
                check(_lib.lib().bb_trainer_create(self.ctx.handle, n_features, z_dim, _host_ptrs(self._w),
                                                   _host_ptrs(self._b), max_batch, C.byref(self.handle)), "bb_trainer_create")
            else:
                self._bn = {k: [np.ascontiguousarray(a, dtype=np.float64) for a in bn[k]]
                            for k in ("weight", "bias", "running_mean", "running_var")}
                nbt = (C.c_longlong * 4)(*[int(v) for v in bn["num_batches_tracked"]])
                check(_lib.lib().bb_trainer_create_dbn(
                    self.ctx.handle, n_features, z_dim, _host_ptrs(self._w), _host_ptrs(self._b),
                    _host_ptrs(self._bn["weight"]), _host_ptrs(self._bn["bias"]), _host_ptrs(self._bn["running_mean"]),
                    _host_ptrs(self._bn["running_var"]), nbt, max_batch, C.byref(self.handle)), "bb_trainer_create_dbn")
        self.n_params = _lib.lib().bb_trainer_param_count(self.handle)
        self.loss_accum = torch.zeros(1, dtype=torch.float64, device=self.ctx.device)

    def __del__(self):
        try:
            if getattr(self, "handle", None) and self.handle.value:
                _lib.lib().bb_trainer_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    def _flat(self, ptr, n=None, typestr="<f4"):
        # zero-copy torch view of library-owned device memory
        from torch.utils import dlpack  # noqa: F401  (documented route; below uses __cuda_array_interface__)

        class _Arr:
            pass

        a = _Arr()
        a.__cuda_array_interface__ = {"shape": (n or self.n_params,), "typestr": typestr, "data": (int(ptr), False), "version": 2}
        return torch.as_tensor(a, device=self.ctx.device)

    def set_precision(self, precision):
        """"auto" / "split16": tensor-core step (AE family, MSE loss); "fp32": the fp32 FFMA kernels; "fp64": the float64
        kernels with float64 master parameters (before the first step; params_view / grads_view / bn_running_views are
        float64 from then on, step / epoch / validate take float32 or float64 tables).  AE_Dropout_BN under "fp64": batches
        up to 4 rows x resident CTAs (592 on a B200), dropout from Philox, injected masks or set_dropout_torch"""
        check(_lib.lib().bb_trainer_set_precision(self.handle, _prec(precision)), "bb_trainer_set_precision")

    @property
    def precision(self):
        return {_lib.BB_PREC_FP32: "fp32", _lib.BB_PREC_SPLIT16: "split16", _lib.BB_PREC_FP64: "fp64"}[
            _lib.lib().bb_trainer_precision(self.handle)]

    @property
    def _fp64(self):
        return _lib.lib().bb_trainer_precision(self.handle) == _lib.BB_PREC_FP64

    def _x(self, x, name):
        """(pointer, C entry point) of a float32 or float64 CUDA table"""
        assert x.is_cuda and x.is_contiguous() and x.dtype in (torch.float32, torch.float64)
        if x.dtype == torch.float64:
            name += "_f64"  # BB_PREC_FP64 trainers only: the library refuses the others
        return _ptr(x), getattr(_lib.lib(), name), name

    def range_flag(self, reset=True):
        """sticky flag of the split16 step: a batch loss was not finite (values beyond the fp16 range); synchronises"""
        flag = C.c_int(0)
        check(_lib.lib().bb_trainer_range_flag(self.handle, int(reset), C.byref(flag)), "bb_trainer_range_flag")
        return bool(flag.value)

    def dp_connect(self, group=None):
        """data parallel inside the library: exchange the CUDA IPC handles of every rank's exchange block over
        torch.distributed (host plumbing) and map the peers' blocks; afterwards `epoch(full_table, global_batch, hyper)`
        with hyper.world_size == world runs the fused gradient exchange (include/baler_b200.h, bb_trainer_dp_connect)"""
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        mine = (C.c_ubyte * 64)()
        check(_lib.lib().bb_trainer_dp_export(self.handle, world, mine), "bb_trainer_dp_export")
        handles = [None] * world
        dist.all_gather_object(handles, bytes(mine), group=group)
        blob = (C.c_ubyte * (64 * world)).from_buffer_copy(b"".join(handles))
        check(_lib.lib().bb_trainer_dp_connect(self.handle, rank, world, blob), "bb_trainer_dp_connect")
        dist.barrier(group)
        self.dp_world = world
        return world

    def debug_layer(self, which, layer, rows):
        """split16 step diagnostics: (features, rows) float32 of the input (which=0, last feature = bias ones) or the
        pre-activation gradient (which=1) of `layer` as the last step left them"""
        out = np.empty(256 * rows, dtype=np.float32)
        n = _lib.lib().bb_trainer_debug_layer(self.handle, which, layer, rows, out.ctypes.data, out.size)
        if n <= 0:
            check(n if n < 0 else -1, "bb_trainer_debug_layer")
        return out[:n * rows].reshape(n, rows)

    def params_view(self):
        """flat parameters (float32; float64 under precision "fp64")"""
        if self._fp64:
            return self._flat(_lib.lib().bb_trainer_params_dev_f64(self.handle), typestr="<f8")
        return self._flat(_lib.lib().bb_trainer_params_dev(self.handle))

    def grads_view(self):
        """n_params gradient entries followed by the batch loss (one flat buffer = one all-reduce); float64 under "fp64" """
        if self._fp64:
            return self._flat(_lib.lib().bb_trainer_grads_dev_f64(self.handle), self.n_params + 1, "<f8")
        return self._flat(_lib.lib().bb_trainer_grads_dev(self.handle), self.n_params + 1)

    def step(self, x, hyper, phase=0):
        ptr, fn, name = self._x(x, "bb_trainer_step")
        check(fn(self.handle, ptr, x.shape[0], C.byref(hyper), phase, _ptr(self.loss_accum), _stream(self.ctx)), name)

    def epoch(self, x, batch, hyper, window_rows=None):
        """one epoch over a CUDA table, or over a C-contiguous numpy table streamed through two device windows of
        `window_rows` rows (a multiple of `batch`; bb_trainer_epoch_host): the same steps, bit for bit"""
        out = C.c_double()
        if isinstance(x, np.ndarray):
            ptr, dt = _host_table(x, window_rows, batch)
            check(_lib.lib().bb_trainer_epoch_host(self.handle, ptr, dt, x.shape[0], batch, C.byref(hyper), int(window_rows),
                                                   C.byref(out), _stream(self.ctx)), "bb_trainer_epoch_host")
            return out.value
        ptr, fn, name = self._x(x, "bb_trainer_epoch")
        check(fn(self.handle, ptr, x.shape[0], batch, C.byref(hyper), C.byref(out), _stream(self.ctx)), name)
        return out.value

    def validate(self, x, batch, window_rows=None):
        """validate over a CUDA table, or a numpy table streamed as in epoch()"""
        out = C.c_double()
        if isinstance(x, np.ndarray):
            ptr, dt = _host_table(x, window_rows, batch)
            check(_lib.lib().bb_trainer_validate_host(self.handle, ptr, dt, x.shape[0], batch, int(window_rows), C.byref(out),
                                                      _stream(self.ctx)), "bb_trainer_validate_host")
            return out.value
        ptr, fn, name = self._x(x, "bb_trainer_validate")
        check(fn(self.handle, ptr, x.shape[0], batch, C.byref(out), _stream(self.ctx)), name)
        return out.value

    def set_dropout(self, seed=0, masks=None):
        """AE_Dropout_BN: Philox seed, or 4 CUDA uint8 keep-masks [batch, width] injected for parity tests"""
        self._masks = None if masks is None else [m.contiguous() for m in masks]
        ptrs = None
        if self._masks is not None:
            ptrs = (C.c_void_p * 4)(*[m.data_ptr() for m in self._masks])
        check(_lib.lib().bb_trainer_set_dropout(self.handle, int(seed), ptrs), "bb_trainer_set_dropout")

    def bn_running_views(self):
        """AE_Dropout_BN: zero-copy views (running_mean, running_var) of the concatenated BatchNorm buffers"""
        rm, rv, n = C.c_void_p(), C.c_void_p(), C.c_int()
        name, typestr = ("bb_trainer_bn_running_dev_f64", "<f8") if self._fp64 else ("bb_trainer_bn_running_dev", "<f4")
        check(getattr(_lib.lib(), name)(self.handle, C.byref(rm), C.byref(rv), C.byref(n)), name)
        return self._flat(rm.value, n.value, typestr), self._flat(rv.value, n.value, typestr)

    def set_dropout_torch(self, generator=None):
        """AE_Dropout_BN under "fp64": the following steps draw their dropout masks on the device from `generator`'s
        Mersenne Twister (torch's default CPU generator when None) exactly as the reference's bernoulli_ calls would;
        write_back_dropout_torch() then leaves the generator where the reference's would be"""
        self._torch_gen = torch.default_generator if generator is None else generator
        key, pos = mt19937_from_torch_state(self._torch_gen.get_state())
        check(_lib.lib().bb_trainer_set_dropout_mt19937(self.handle, key.ctypes.data, pos), "bb_trainer_set_dropout_mt19937")

    def write_back_dropout_torch(self):
        """set the generator of set_dropout_torch to the device's state after the last drawn word (synchronises)"""
        key = np.empty(624, dtype=np.uint32)
        pos = C.c_int()
        check(_lib.lib().bb_trainer_get_dropout_mt19937(self.handle, key.ctypes.data, C.byref(pos)),
              "bb_trainer_get_dropout_mt19937")
        self._torch_gen.set_state(mt19937_to_torch_state(self._torch_gen.get_state(), key, pos.value))

    def get_bn(self):
        out = {k: [np.empty_like(a) for a in self._bn[k]] for k in ("weight", "bias", "running_mean", "running_var")}
        nbt = (C.c_longlong * 4)()
        check(_lib.lib().bb_trainer_get_bn(self.handle, _host_ptrs(out["weight"]), _host_ptrs(out["bias"]),
                                           _host_ptrs(out["running_mean"]), _host_ptrs(out["running_var"]), nbt),
              "bb_trainer_get_bn")
        out["num_batches_tracked"] = [int(v) for v in nbt]
        return out

    def activation_means(self):
        out = np.empty((6, 200), dtype=np.float64)
        check(_lib.lib().bb_trainer_activation_means(self.handle, out.ctypes.data), "bb_trainer_activation_means")
        return out

    def get_params(self):
        w = [np.empty_like(a) for a in self._w]
        b = [np.empty_like(a) for a in self._b]
        check(_lib.lib().bb_trainer_get_params(self.handle, _host_ptrs(w), _host_ptrs(b)), "bb_trainer_get_params")
        return w, b


def error_bounded_deltas(x, y, mn, rg, bound_percent, row0=0):
    """helper.save_error_bounded_requirement on device tensors: x raw rows, y decoded normalised rows (float32 CUDA),
    mn / rg the normalisation features (or None).  Returns (rows int64, cols int64, deltas float16) sorted row-major."""
    ctx = get_context()
    assert x.is_cuda and y.is_cuda and x.dtype == torch.float32 and y.dtype == torch.float32 and x.shape == y.shape
    n, c = x.shape
    cap = n * c
    count = torch.zeros(1, dtype=torch.int64, device=x.device)
    rows = torch.empty(cap, dtype=torch.int64, device=x.device)
    cols = torch.empty(cap, dtype=torch.int32, device=x.device)
    deltas = torch.empty(cap, dtype=torch.float16, device=x.device)
    check(_lib.lib().bb_error_bounded_deltas_f32(ctx.handle, _ptr(x.contiguous()), _ptr(y.contiguous()), n, c, _ptr(mn), _ptr(rg),
                                                 float(bound_percent), int(row0), cap, _ptr(count), _ptr(rows), _ptr(cols),
                                                 _ptr(deltas), _stream(ctx)), "bb_error_bounded_deltas_f32")
    k = int(count.item())
    r, cc, d = rows[:k].cpu().numpy(), cols[:k].cpu().numpy().astype(np.int64), deltas[:k].cpu().numpy()
    order = np.lexsort((cc, r))
    return r[order], cc[order], d[order]


class LayeredTrainer:
    """bb_ltrainer: the layer-by-layer trainer for dense autoencoders too wide for the fused training kernels
    (CFD_dense_AE on 2500-feature snapshots), and for AE_Dropout_BN batches beyond the fused step's (LayeredTrainer.dbn).
    Same surface as Trainer for what training.train uses."""

    _ACT = {"none": 0, "leaky": 1, "relu": 2}
    dbn_kind = False

    def __init__(self, weights, biases, acts, max_batch, device=None, dims=None, w_maps=None, bn=None, loss_columns=0):
        """plain Linears: weights[l] is the (out, in) matrix.  Conv_AE (weight sharing, BatchNorm2d; see
        bb_ltrainer_create_ex): `dims` gives the layer widths, w_maps[l] (int32 (out * in,), or None) maps dense entries to
        the flat kernel weights[l], biases[l] is per channel; bn[l] = None or a (4, channels) array gamma / beta /
        running_mean / running_var."""
        self.ctx = get_context(device)
        self.handle = C.c_void_p()
        n = len(weights)
        self._w = [np.ascontiguousarray(w, dtype=np.float64) for w in weights]
        self._b = [np.ascontiguousarray(b, dtype=np.float64) for b in biases]
        self._maps = [None if m is None else np.ascontiguousarray(m, dtype=np.int32) for m in (w_maps or [None] * n)]
        self._bn = None if bn is None or all(b is None for b in bn) else \
            [None if b is None else np.ascontiguousarray(b, dtype=np.float64) for b in bn]
        if dims is None:
            dims = [self._w[0].shape[1]] + [w.shape[0] for w in self._w]
        self.dims = list(dims)
        dims_c = (C.c_int * (n + 1))(*self.dims)
        acts_c = (C.c_int * n)(*[self._ACT[a] for a in acts])
        shared = (C.c_int * n)(*[0 if m is None else self._w[l].size for l, m in enumerate(self._maps)])
        n_bias = (C.c_int * n)(*[0 if m is None else self._b[l].size for l, m in enumerate(self._maps)])
        bn_ch = (C.c_int * n)(*[0 if self._bn is None or self._bn[l] is None else self._bn[l].shape[1] for l in range(n)])
        maps_c, bn_c = (C.c_void_p * n)(), (C.c_void_p * n)()
        for l in range(n):
            if self._maps[l] is not None:
                assert self._maps[l].size == self.dims[l] * self.dims[l + 1]
                maps_c[l] = self._maps[l].ctypes.data
            if bn_ch[l]:
                bn_c[l] = self._bn[l].ctypes.data
        with torch.cuda.device(self.ctx.device):
            check(_lib.lib().bb_ltrainer_create_ex(self.ctx.handle, n, dims_c, acts_c, shared, maps_c, n_bias, bn_ch,
                                                   _host_ptrs(self._w), _host_ptrs(self._b), bn_c, loss_columns, max_batch,
                                                   C.byref(self.handle)), "bb_ltrainer_create_ex")
        self.n_params = _lib.lib().bb_ltrainer_param_count(self.handle)
        self.loss_accum = torch.zeros(1, dtype=torch.float64, device=self.ctx.device)

    @classmethod
    def dbn(cls, weights, biases, n_features, z_dim, max_batch, bn, device=None):
        """AE_Dropout_BN (bb_ltrainer_create_dbn): the arguments of Trainer(..., bn=bn) - the 8 Linears (out, in), and bn
        = {weight, bias, running_mean, running_var: 4 arrays each, num_batches_tracked: 4 ints}.  No batch limit beyond
        memory.  get_bn() then returns that dict."""
        self = cls.__new__(cls)
        self.ctx = get_context(device)
        self.handle = C.c_void_p()
        self.dbn_kind = True
        self._w = [np.ascontiguousarray(w, dtype=np.float64) for w in weights]
        self._b = [np.ascontiguousarray(b, dtype=np.float64) for b in biases]
        self._bn = {k: [np.ascontiguousarray(a, dtype=np.float64) for a in bn[k]]
                    for k in ("weight", "bias", "running_mean", "running_var")}
        self.dims = [n_features, 200, 100, 50, z_dim, 50, 100, 200, n_features]
        nbt = (C.c_longlong * 4)(*[int(v) for v in bn.get("num_batches_tracked", [0] * 4)])
        with torch.cuda.device(self.ctx.device):
            check(_lib.lib().bb_ltrainer_create_dbn(self.ctx.handle, n_features, z_dim, _host_ptrs(self._w), _host_ptrs(self._b),
                                                    _host_ptrs(self._bn["weight"]), _host_ptrs(self._bn["bias"]),
                                                    _host_ptrs(self._bn["running_mean"]), _host_ptrs(self._bn["running_var"]),
                                                    nbt, max_batch, C.byref(self.handle)), "bb_ltrainer_create_dbn")
        self.n_params = _lib.lib().bb_ltrainer_param_count(self.handle)
        self.loss_accum = torch.zeros(1, dtype=torch.float64, device=self.ctx.device)
        return self

    def set_dropout(self, seed=0, masks=None):
        """AE_Dropout_BN: Philox seed (the fused trainer's stream), or 4 CUDA uint8 keep-masks [batch, width]"""
        self._masks = None if masks is None else [m.contiguous() for m in masks]
        ptrs = None
        if self._masks is not None:
            ptrs = (C.c_void_p * 4)(*[m.data_ptr() for m in self._masks])
        check(_lib.lib().bb_ltrainer_set_dropout(self.handle, int(seed), ptrs), "bb_ltrainer_set_dropout")

    def __del__(self):
        try:
            if getattr(self, "handle", None) and self.handle.value:
                _lib.lib().bb_ltrainer_destroy(self.handle)
                self.handle = C.c_void_p()
        except Exception:
            pass

    _flat = Trainer._flat

    def params_view(self):
        return self._flat(_lib.lib().bb_ltrainer_params_dev(self.handle))

    def grads_view(self):
        return self._flat(_lib.lib().bb_ltrainer_grads_dev(self.handle), self.n_params + 1)

    def step(self, x, hyper, phase=0):
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
        check(_lib.lib().bb_ltrainer_step(self.handle, _ptr(x), x.shape[0], C.byref(hyper), phase, _ptr(self.loss_accum),
                                          _stream(self.ctx)), "bb_ltrainer_step")

    def step_swae(self, x, hyper, prior, proj, latent_layer, reg_weight=100.0, phase=0):
        """one step with utils.loss_function_swae: `prior` [rows, z_dim] standard-normal draws, `proj` [S, z_dim] unit
        projection directions (float32, device), the latent = output of layer `latent_layer`"""
        for t in (x, prior, proj):
            assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
        assert prior.shape[0] == x.shape[0] and prior.shape[1] == proj.shape[1] == self.dims[latent_layer + 1]
        check(_lib.lib().bb_ltrainer_step_swae(self.handle, _ptr(x), x.shape[0], C.byref(hyper), phase, _ptr(prior), _ptr(proj),
                                               proj.shape[0], latent_layer, float(reg_weight), _ptr(self.loss_accum),
                                               _stream(self.ctx)), "bb_ltrainer_step_swae")

    def epoch(self, x, batch, hyper, window_rows=None):
        """Trainer.epoch: a CUDA table, or a float32 numpy table streamed in windows (bb_ltrainer_epoch_host)"""
        out = C.c_double()
        if isinstance(x, np.ndarray):
            ptr, dt = _host_table(x, window_rows, batch)
            check(_lib.lib().bb_ltrainer_epoch_host(self.handle, ptr, dt, x.shape[0], batch, C.byref(hyper), int(window_rows),
                                                    C.byref(out), _stream(self.ctx)), "bb_ltrainer_epoch_host")
            return out.value
        check(_lib.lib().bb_ltrainer_epoch(self.handle, _ptr(x), x.shape[0], batch, C.byref(hyper), C.byref(out),
                                           _stream(self.ctx)), "bb_ltrainer_epoch")
        return out.value

    def validate(self, x, batch, window_rows=None):
        out = C.c_double()
        if isinstance(x, np.ndarray):
            ptr, dt = _host_table(x, window_rows, batch)
            check(_lib.lib().bb_ltrainer_validate_host(self.handle, ptr, dt, x.shape[0], batch, int(window_rows),
                                                       C.byref(out), _stream(self.ctx)), "bb_ltrainer_validate_host")
            return out.value
        check(_lib.lib().bb_ltrainer_validate(self.handle, _ptr(x), x.shape[0], batch, C.byref(out), _stream(self.ctx)),
              "bb_ltrainer_validate")
        return out.value

    def get_params(self):
        w = [np.empty_like(a) for a in self._w]
        b = [np.empty_like(a) for a in self._b]
        check(_lib.lib().bb_ltrainer_get_params(self.handle, _host_ptrs(w), _host_ptrs(b)), "bb_ltrainer_get_params")
        return w, b

    def get_bn(self):
        """per layer None or (4, channels): gamma / beta / running_mean / running_var.  AE_Dropout_BN (dbn): Trainer.get_bn's
        dict, num_batches_tracked included"""
        if not self.dbn_kind:
            out = [None if b is None else np.empty_like(b) for b in self._bn]
        else:
            out = [None] * 4 + [np.empty((4, n)) for n in self.dims[5:]]
        ptrs = (C.c_void_p * len(out))()
        for l, a in enumerate(out):
            if a is not None:
                ptrs[l] = a.ctypes.data
        check(_lib.lib().bb_ltrainer_get_bn(self.handle, ptrs), "bb_ltrainer_get_bn")
        if not self.dbn_kind:
            return out
        nbt = (C.c_longlong * 8)()
        check(_lib.lib().bb_ltrainer_bn_batches_tracked(self.handle, nbt), "bb_ltrainer_bn_batches_tracked")
        keys = ("weight", "bias", "running_mean", "running_var")
        res = {k: [out[4 + i][j].copy() for i in range(4)] for j, k in enumerate(keys)}
        res["num_batches_tracked"] = [int(v) for v in nbt[4:]]
        return res

    def bn_running_views(self):
        """zero-copy view of the running statistics of all BatchNorm layers (one tensor; DataParallelTrainer averages it)"""
        n = C.c_int()
        ptr = _lib.lib().bb_ltrainer_bn_running_dev(self.handle, C.byref(n))
        return (self._flat(ptr, n.value),)

    def activation_means(self):
        """bb_ltrainer_activation_means: the (6, 200) NaN-padded matrix of Trainer.activation_means, from the last forward
        pass; the 8-Linear autoencoders only"""
        if len(self.dims) != 9:
            raise NotImplementedError("activation extraction is implemented for the dense autoencoders (8 Linears), not "
                                      "for a %d-layer chain" % (len(self.dims) - 1))
        out = np.empty((6, 200), dtype=np.float64)
        check(_lib.lib().bb_ltrainer_activation_means(self.handle, out.ctypes.data), "bb_ltrainer_activation_means")
        return out


def make_hyper(lr=1e-3, reg_param=0.0, l1=False, world_size=1, beta1=0.9, beta2=0.999, eps=1e-8):
    return _lib.TrainHyper(lr, beta1, beta2, eps, reg_param, int(bool(l1)), world_size)
