"""numpy mirror of the b-bit latent (baler_b200/latent_q8.py, csrc/bb_latent_q8.cu) for b = 2..8: quantise, pack, unpack,
dequantise, the error bound and the compressed.npz writer.  The device results are compared with it bit for bit; at
b = 8 it is the 8-bit mirror (tests/latent_q8_ref.py) byte for byte."""
import numpy as np

from latent_q8_ref import BLOCK, _keys, _unkey


def row_bytes(z_dim, bits):
    return (z_dim * bits + 7) // 8


def quantize(z, bits):
    """float32 latent [N, Z] -> (codes uint8 [N, Z], one code per byte, lo float32 [B, Z], step float32 [B, Z])"""
    levels = float(2 ** bits - 2)
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
    step = ((hi.astype(np.float64) - lo.astype(np.float64)) / levels).astype(np.float32)
    flat = step == 0
    inv = np.where(flat, 0.0, 1.0 / np.where(flat, 1.0, step.astype(np.float64)))
    with np.errstate(invalid="ignore", over="ignore"):
        t = np.rint((v.astype(np.float64) - lo.astype(np.float64)[:, None]) * inv[:, None])
    q = np.clip(np.where(fin, t, 0.0), 0.0, levels).astype(np.uint8)
    q = np.where(flat[:, None], np.uint8(0), q)
    codes = np.where(fin, q, np.uint8(2 ** bits - 1)).reshape(nb * BLOCK, zd)[:n]
    return np.ascontiguousarray(codes), lo, step


def pack(codes, bits):
    """codes [N, Z] (one per byte) -> packed rows [N, ceil(Z * bits / 8)]: column j is bits [j b, j b + b) of its row, bit k
    being bit k % 8 of byte k // 8"""
    n, zd = codes.shape
    bitplanes = ((codes[:, :, None] >> np.arange(bits, dtype=np.uint8)) & 1).reshape(n, zd * bits)
    padded = np.zeros((n, row_bytes(zd, bits) * 8), np.uint8)
    padded[:, :zd * bits] = bitplanes
    return np.ascontiguousarray(np.packbits(padded, axis=1, bitorder="little"))


def unpack(packed, z_dim, bits):
    """packed rows -> codes [N, z_dim], one per byte"""
    n = packed.shape[0]
    planes = np.unpackbits(packed, axis=1, bitorder="little")[:, :z_dim * bits].reshape(n, z_dim, bits)
    return np.ascontiguousarray((planes << np.arange(bits, dtype=np.uint8)).sum(axis=2, dtype=np.uint32).astype(np.uint8))


def dequantize(codes, lo, step, bits):
    """float32 latent of (codes [N, Z] one per byte, lo, step)"""
    n = codes.shape[0]
    rows = np.arange(n) // BLOCK
    lo64, st64 = lo.astype(np.float64)[rows], step.astype(np.float64)[rows]
    v = (lo64 + codes.astype(np.float64) * st64).astype(np.float32)
    return np.where(codes == 2 ** bits - 1, np.float32(np.nan), v)


def error_bound(z, step, bits):
    """per element: step / 2, widened by the float32 rounding of step (L steps of it, L = 2^b - 2, at most L 2^-24 of a
    step), plus the float32 rounding of the decoded value"""
    st = step.astype(np.float64)[np.arange(len(z)) // BLOCK]
    return (0.5 + (2 ** bits - 2) * 2.0 ** -24) * st + np.spacing(np.abs(z).astype(np.float32)).astype(np.float64)


def write_npz(path, packed, lo, step, bits, names, normalization_features):
    """a compressed.npz holding a b-bit latent, written without the package (no latent_bits key at b = 8)"""
    extra = {} if bits == 8 else {"latent_bits": np.int64(bits)}
    np.savez(path, data=packed, latent_min=lo, latent_step=step, latent_block_rows=np.int64(BLOCK), names=names,
             normalization_features=normalization_features, **extra)
