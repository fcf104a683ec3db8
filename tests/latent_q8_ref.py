"""numpy mirror of the 8-bit latent (baler_b200/latent_q8.py, csrc/bb_latent_q8.cu): quantise, dequantise, the error bound
and the compressed.npz writer.  The device results are compared with it bit for bit."""
import numpy as np

BLOCK = 128


def _keys(v):
    """order-preserving int32 keys of float32 values (-0 < +0)"""
    u = np.ascontiguousarray(v, dtype=np.float32).view(np.int32)
    return u ^ ((u >> 31) & np.int32(0x7fffffff))


def _unkey(k):
    k = np.asarray(k, dtype=np.int32)
    return np.where(k >= 0, k, k ^ np.int32(0x7fffffff)).astype(np.int32).view(np.float32)


def quantize(z):
    """float32 latent [N, Z] -> (codes uint8 [N, Z], lo float32 [B, Z], step float32 [B, Z])"""
    z = np.ascontiguousarray(z, dtype=np.float32)
    n, zd = z.shape
    nb = (n + BLOCK - 1) // BLOCK
    v = np.full((nb * BLOCK, zd), np.nan, np.float32)  # the short last block is padded with non-finite rows
    v[:n] = z
    v = v.reshape(nb, BLOCK, zd)
    fin = np.isfinite(v)
    k = _keys(v)
    kmn = np.where(fin, k, np.int32(np.iinfo(np.int32).max)).min(axis=1)
    kmx = np.where(fin, k, np.int32(np.iinfo(np.int32).min)).max(axis=1)
    anyf = fin.any(axis=1)
    lo = np.where(anyf, _unkey(kmn), np.float32(0)).astype(np.float32)
    hi = np.where(anyf, _unkey(kmx), np.float32(0)).astype(np.float32)
    step = ((hi.astype(np.float64) - lo.astype(np.float64)) / 254.0).astype(np.float32)
    flat = step == 0
    inv = np.where(flat, 0.0, 1.0 / np.where(flat, 1.0, step.astype(np.float64)))
    with np.errstate(invalid="ignore", over="ignore"):
        t = np.rint((v.astype(np.float64) - lo.astype(np.float64)[:, None]) * inv[:, None])
    q = np.clip(np.where(fin, t, 0.0), 0.0, 254.0).astype(np.uint8)
    q = np.where(flat[:, None], np.uint8(0), q)
    codes = np.where(fin, q, np.uint8(255)).reshape(nb * BLOCK, zd)[:n]
    return np.ascontiguousarray(codes), lo, step


def dequantize(codes, lo, step):
    """float32 latent of (codes, lo, step)"""
    n = codes.shape[0]
    rows = np.arange(n) // BLOCK
    lo64, st64 = lo.astype(np.float64)[rows], step.astype(np.float64)[rows]
    v = (lo64 + codes.astype(np.float64) * st64).astype(np.float32)
    return np.where(codes == 255, np.float32(np.nan), v)


def error_bound(z, step):
    """per element: step / 2 (widened by the float32 rounding of step, at most 2^-16 of it) plus the float32 rounding of
    the decoded value"""
    st = step.astype(np.float64)[np.arange(len(z)) // BLOCK]
    return 0.5 * st * (1 + 2.0 ** -16) + np.spacing(np.abs(z).astype(np.float32)).astype(np.float64)


def write_npz(path, codes, lo, step, names, normalization_features):
    """a compressed.npz holding an 8-bit latent, written without the package"""
    np.savez(path, data=codes, latent_min=lo, latent_step=step, latent_block_rows=np.int64(BLOCK), names=names,
             normalization_features=normalization_features)
