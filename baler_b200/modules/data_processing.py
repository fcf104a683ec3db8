"""Host-side mirror of the reference's baler/modules/data_processing.py for the hot path: same
function names and argument meaning; min/max and (re)normalisation run in CUDA kernels."""
import numpy as np
import torch

from .. import engine
from . import models


def convert_to_blocks_util(blocks, data):
    """reference data_processing.py:26-34: plain reshape into (n_blocks, blocks[1], blocks[2])"""
    print("Converted Dataset to Blocks of Size - ", blocks, " from original ", data.shape)
    b1, b2 = int(blocks[1]), int(blocks[2])
    return data.reshape(int(np.prod(data.shape)) // (b1 * b2), b1, b2)


def save_model(model, model_path):
    """reference data_processing.py:37-47: torch zip-pickle of the state_dict (same keys / dtypes)"""
    torch.save(model.state_dict(), model_path)


def initialise_model(model_name):
    """reference data_processing.py:76-86"""
    return getattr(models, model_name)


def load_model(model_object, model_path, n_features, z_dim):
    """reference data_processing.py:89-110"""
    model = model_object(n_features, z_dim)
    model.load_state_dict(torch.load(str(model_path), map_location="cpu"), strict=False)
    return model


def _table(data):
    """(n, c) float32 view of 1-D / 2-D / 3-D input: statistics are per position over axis 0"""
    arr = np.asarray(data)
    flat = arr.reshape(arr.shape[0], -1) if arr.ndim > 1 else arr.reshape(-1, 1)
    return arr, engine.host_convert(flat, np.float32)


# float64 tables whose offset dwarfs their spread (IDs, timestamps ~1e9 with a range of a few units): in float32, x alone
# is rounded to |x| * 2^-24, i.e. max(|min|, |max|) / range * 6e-8 of the normalised range.  Up to this ratio that stays
# below 4e-6 and the kernels' float32 normalisation is used; beyond it the (re)normalisation is done on the host in
# float64, the arithmetic the reference's numpy code performs on such a table (data_processing.py:133-153, 188-203).
F32_OFFSET_LIMIT = 64.0


def _ill_conditioned(mn, mx, probe=False):
    mn, mx = np.asarray(mn, dtype=np.float64), np.asarray(mx, dtype=np.float64)
    a, r = np.maximum(np.abs(mn), np.abs(mx)), mx - mn
    limit = F32_OFFSET_LIMIT - 1.0 if probe else F32_OFFSET_LIMIT  # a row sample's ratio is at most 1 below the table's
    bad = a > limit * r
    if not probe:
        bad &= r > 0  # a constant column is 0 / 0 whatever the arithmetic
    return bool(np.any(bad & np.isfinite(a)))


def float64_stats(flat, minmax=None):
    """exact float64 (min, range) per column of a float64 table that float32 normalisation would damage, else None.
    A strided sample of ~4096 rows decides first: every value lies between the table's min and max, so a sample whose
    ratio is <= F32_OFFSET_LIMIT - 1 proves the table's is <= F32_OFFSET_LIMIT and the two full reductions are skipped.
    `minmax(flat) -> (min, max)` replaces the local reductions (torchrun: global statistics from row shards)."""
    flat = np.asarray(flat)
    if flat.dtype != np.float64 or flat.ndim != 2 or len(flat) == 0:
        return None
    probe = flat[:: max(1, len(flat) // 4096)]
    if not _ill_conditioned(probe.min(axis=0), probe.max(axis=0), probe=True):
        return None
    mn, mx = minmax(flat) if minmax is not None else (flat.min(axis=0), flat.max(axis=0))
    return (mn, mx - mn) if _ill_conditioned(mn, mx) else None


def normalize_float64_host(flat, mn, rg, out_dtype=np.float64):
    """(x - min) / range in float64 on the host (0 / 0 -> nan as numpy gives the reference), narrowed to out_dtype"""
    with np.errstate(divide="ignore", invalid="ignore"):
        return ((np.asarray(flat, dtype=np.float64) - mn) / rg).astype(out_dtype, copy=False)


# Device buffer of the row-chunked preprocessing passes: find_minmax / normalize / minmax_normalize_f64 / renormalize_func
# upload the table in chunks of at most this many bytes, so a table larger than device memory is preprocessed too
PREPROCESS_CHUNK_BYTES = 1 << 28


def _row_chunks(flat):
    """(r0, rows) of the row chunks of a C-contiguous 2-D host table (one empty chunk for an empty table)"""
    rows = max(1, PREPROCESS_CHUNK_BYTES // max(1, flat.shape[1] * flat.itemsize))
    return [(r0, flat[r0:r0 + rows]) for r0 in range(0, len(flat), rows)] or [(0, flat)]


def _minmax_dev(flat):
    """(device table or None, column min, column max) of a C-contiguous host table.  Per-chunk min / max, combined by the
    same kernel over the stacked chunk results (min of mins, max of maxes: exact, -0 < +0 and NaN kept as in one pass).
    A table of one chunk stays on the device for the caller's second pass."""
    chunks = _row_chunks(flat)
    mins, maxs, x = [], [], None
    for _, c in chunks:
        x = torch.from_numpy(c).cuda()
        mn, mx = engine.colminmax(x)
        mins.append(mn)
        maxs.append(mx)
    if len(chunks) == 1:
        return x, mins[0], maxs[0]
    return None, engine.colminmax(torch.stack(mins))[0], engine.colminmax(torch.stack(maxs))[1]


def _map_chunks(flat, x, fn, out_dtype):
    """host array of fn(device chunk) over the row chunks of `flat` (x: the device copy of a one-chunk table, or None)"""
    if x is not None:
        return fn(x).cpu().numpy()
    out = np.empty(flat.shape, dtype=out_dtype)
    for r0, c in _row_chunks(flat):
        out[r0:r0 + len(c)] = fn(torch.from_numpy(c).cuda()).cpu().numpy()
    return out


def find_minmax(data):
    """[min; max - min] per column (reference data_processing.py:113-130), computed on the GPU in row chunks of at most
    PREPROCESS_CHUNK_BYTES.
    float32 arithmetic: exact for float32 / small-integer tables (what the CMS path feeds); float64 tables whose offset
    dwarfs their spread get exact float64 statistics from the host (float64_stats)."""
    arr = np.asarray(data)
    if arr.dtype == np.float64 and arr.ndim >= 1 and arr.size:
        st = float64_stats(arr.reshape(arr.shape[0], -1))
        if st is not None:  # offset >> spread: exact float64 statistics (see F32_OFFSET_LIMIT)
            feats = np.array([st[0], st[1]])
            return feats.reshape((2,) + arr.shape[1:]) if arr.ndim > 1 else feats.reshape(2)
    arr, flat = _table(data)
    _, mn, mx = _minmax_dev(flat)
    mn, mx = mn.cpu().numpy(), mx.cpu().numpy()
    out_dtype = arr.dtype if arr.dtype.kind in "iuf" else np.float32
    feats = np.array([mn, mx - mn]).astype(out_dtype)
    return feats.reshape((2,) + arr.shape[1:]) if arr.ndim > 1 else feats.reshape(2)


def normalize(data, custom_norm):
    """(x - min) / (max - min) over axis 0 (reference data_processing.py:133-153 applied per column by
    helper.normalize); identity when custom_norm."""
    arr = np.asarray(data)
    if custom_norm:
        return arr
    if arr.dtype == np.float64 and arr.size:
        flat64 = arr.reshape(arr.shape[0], -1) if arr.ndim > 1 else arr.reshape(-1, 1)
        st = float64_stats(flat64)
        if st is not None:
            return normalize_float64_host(flat64, st[0], st[1]).reshape(arr.shape)
    arr, flat = _table(data)
    x, mn, mx = _minmax_dev(flat)
    rg = mx - mn  # one float32 subtraction per column
    out = _map_chunks(flat, x, lambda c: engine.normalize_table(c, mn, rg, out=c), np.float32).reshape(arr.shape)
    return out if arr.dtype == np.float32 else engine.host_convert(out, np.float64)


def minmax_normalize_f64(data, normalise=True):
    """precision "fp64" on a float64 table: ([min; max - min] exact in float64, the table normalised in float64 on the
    device when `normalise`, else as it is) - what the reference's float64 numpy computes (data_processing.py:113-153),
    bit for bit, with no float32 step and no host pass over the table; row chunks as find_minmax"""
    engine.require_cuda()
    arr = np.asarray(data)
    assert arr.dtype == np.float64
    flat = np.ascontiguousarray(arr.reshape(arr.shape[0], -1) if arr.ndim > 1 else arr.reshape(-1, 1))
    x, mn, mx = _minmax_dev(flat)
    mn_h, mx_h = mn.cpu().numpy(), mx.cpu().numpy()
    rg_h = mx_h - mn_h  # one float64 subtraction per column, as numpy
    feats = np.array([mn_h, rg_h])
    feats = feats.reshape((2,) + arr.shape[1:]) if arr.ndim > 1 else feats.reshape(2)
    if not normalise:
        return feats, arr
    rg = torch.from_numpy(rg_h).cuda()
    out = _map_chunks(flat, x, lambda c: engine.normalize_table_f64(c, mn, rg, out=c), np.float64)
    return feats, out.reshape(arr.shape)


def renormalize_std(input_data, true_min, feature_range):
    """reference data_processing.py:171-185 (one column)"""
    return renormalize_func(np.asarray(input_data).reshape(-1, 1), [true_min], [feature_range]).reshape(-1)


def renormalize_func(norm_data, min_list, range_list):
    """y * range + min (reference data_processing.py:188-203); float32 on the GPU, returned as float64 (in float64 on the
    host when the features say float32 could not hold the result)"""
    mn64, rg64 = np.asarray(min_list, dtype=np.float64).reshape(-1), np.asarray(range_list, dtype=np.float64).reshape(-1)
    if _ill_conditioned(mn64, mn64 + rg64):  # float32 would round the result to |min| * 2^-24 (see F32_OFFSET_LIMIT)
        arr = np.asarray(norm_data)
        flat64 = (arr.reshape(arr.shape[0], -1) if arr.ndim > 1 else arr.reshape(-1, 1)).astype(np.float64)
        return (flat64 * rg64 + mn64).reshape(arr.shape)
    arr, flat = _table(norm_data)
    mn = torch.as_tensor(np.asarray(min_list, dtype=np.float32).reshape(-1)).cuda()
    rg = torch.as_tensor(np.asarray(range_list, dtype=np.float32).reshape(-1)).cuda()
    out = _map_chunks(flat, None, lambda c: engine.normalize_table(c, mn, rg, inverse=True, out=c), np.float32)
    return engine.host_convert(out, np.float64).reshape(arr.shape)
