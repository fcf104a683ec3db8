"""The quantised latent of `latent_dtype = "q2"` ... `"q8"`: its one definition in Python.

The latent [N, z] is stored as b-bit codes (b = 2..8) plus a float32 pair (lo, step) per latent column and block of
BLOCK_ROWS consecutive rows, counted from row 0 of the file (the last block may be short).  With L = 2^b - 2:

    lo, hi   min / max of the block column's finite values (-0 < +0; 0 when it has none)
    step     float32((float64(hi) - float64(lo)) / L)
    code     2^b - 1 for a non-finite value (decodes to NaN); 0 when step == 0;
             else clamp(rint((float64(v) - lo) * (1.0 / float64(step))), 0, L), every float64 operation IEEE
    value    float32(float64(lo) + float64(code) * float64(step)), within step / 2 of v plus float32 rounding
    packing  row r of `data` is row_bytes(z, b) = ceil(z b / 8) bytes; column j's code is bits [j b, j b + b) of the row,
             bit k being bit k % 8 of byte k // 8; the unused high bits of the last byte are 0

b = 8 is the 8-bit latent of `"q8"`: one byte per code, `data` [N, z].  The kernels are in csrc/bb_latent_q8.cu
(include/baler_b200.h: bb_latent_quantize_packed and the *_host_packed pipelines; the *_q8 entry points are b = 8).
compressed.npz then holds `data` (the packed codes), `latent_min`, `latent_step`, `latent_block_rows` and, for b < 8,
`latent_bits` (a q8 file has no such key and is read as b = 8); decompress recognises the format by `latent_step` in the
file and takes z from `latent_min`.  The arrays are plain numpy, so the file stays readable without this package.
"""
from typing import NamedTuple

import numpy as np

BLOCK_ROWS = 128
NAME = "q8"  # the latent_dtype value of the 8-bit latent
MIN_BITS, MAX_BITS = 2, 8


class Q8Latent(NamedTuple):
    """codes uint8 [N, z], lo / step float32 [ceil(N / BLOCK_ROWS), z]: numpy arrays, or CUDA tensors on the device"""
    codes: object
    lo: object
    step: object


class PackedLatent(NamedTuple):
    """codes uint8 [N, row_bytes(z, bits)] (packed rows), lo / step float32 [ceil(N / BLOCK_ROWS), z], bits 2..8"""
    codes: object
    lo: object
    step: object
    bits: int


def bits_of(latent_dtype):
    """the code width of a latent_dtype value "q2" ... "q8", None for any value not starting with "q" (a float type);
    ValueError for another "q..." value"""
    if not (isinstance(latent_dtype, str) and latent_dtype.startswith("q")):
        return None
    names = {"q%d" % b: b for b in range(MIN_BITS, MAX_BITS + 1)}
    if latent_dtype not in names:
        raise ValueError("latent_dtype %r: a quantised latent is one of %s" % (latent_dtype, ", ".join(names)))
    return names[latent_dtype]


def row_bytes(z_dim, bits):
    """bytes per packed row"""
    return (int(z_dim) * int(bits) + 7) // 8


def n_blocks(n_rows):
    return (int(n_rows) + BLOCK_ROWS - 1) // BLOCK_ROWS


def empty(n_rows, z_dim):
    """host buffers for the 8-bit latent of n_rows rows"""
    nb = n_blocks(n_rows)
    return Q8Latent(np.empty((n_rows, z_dim), np.uint8), np.empty((nb, z_dim), np.float32),
                    np.empty((nb, z_dim), np.float32))


def empty_packed(n_rows, z_dim, bits):
    """host buffers for the `bits`-bit latent of n_rows rows"""
    nb = n_blocks(n_rows)
    return PackedLatent(np.empty((n_rows, row_bytes(z_dim, bits)), np.uint8), np.empty((nb, z_dim), np.float32),
                        np.empty((nb, z_dim), np.float32), int(bits))


def rows(q, lo, hi):
    """rows [lo, hi) of a host latent (Q8Latent or PackedLatent); lo must start a block"""
    if lo % BLOCK_ROWS:
        raise ValueError("a slice of a q8 latent starts on a %d-row block boundary, not at row %d" % (BLOCK_ROWS, lo))
    b0, b1 = lo // BLOCK_ROWS, (hi + BLOCK_ROWS - 1) // BLOCK_ROWS
    return q._replace(codes=np.ascontiguousarray(q.codes[lo:hi]), lo=np.ascontiguousarray(q.lo[b0:b1]),
                      step=np.ascontiguousarray(q.step[b0:b1]))


def npz_arrays(q):
    """the compressed.npz entries of a host latent (with `names` and `normalization_features` added by the caller)"""
    out = {"data": q.codes, "latent_min": q.lo, "latent_step": q.step, "latent_block_rows": np.int64(BLOCK_ROWS)}
    bits = getattr(q, "bits", 8)
    if bits != 8:
        out["latent_bits"] = np.int64(bits)
    return out


def in_file(loaded):
    """a loaded compressed.npz holds a quantised latent"""
    return "latent_step" in getattr(loaded, "files", loaded)


def read(loaded):
    """PackedLatent of a loaded compressed.npz (np.load result or dict); ValueError when the arrays do not describe one"""
    files = getattr(loaded, "files", loaded)
    for key in ("data", "latent_min", "latent_step", "latent_block_rows"):
        if key not in files:
            raise ValueError("compressed file has latent_step but no %r: not a q8 latent" % key)
    codes, lo, step = loaded["data"], loaded["latent_min"], loaded["latent_step"]
    block = np.asarray(loaded["latent_block_rows"])
    if block.size != 1 or int(block.reshape(-1)[0]) != BLOCK_ROWS:
        raise ValueError("q8 latent with blocks of %s rows; this version reads blocks of %d rows"
                         % (block.reshape(-1).tolist(), BLOCK_ROWS))
    bits = 8
    if "latent_bits" in files:
        b = np.asarray(loaded["latent_bits"])
        if b.size != 1 or b.dtype.kind not in "iu" or not MIN_BITS <= int(b.reshape(-1)[0]) <= MAX_BITS:
            raise ValueError("latent_bits must be one integer from %d to %d, not %s" % (MIN_BITS, MAX_BITS, b.tolist()))
        bits = int(b.reshape(-1)[0])
    if codes.dtype != np.uint8 or codes.ndim != 2:
        raise ValueError("q8 latent: data must be a 2-D uint8 array, not %s %s" % (codes.dtype, codes.shape))
    if lo.dtype != np.float32 or lo.ndim != 2 or lo.shape[0] != n_blocks(codes.shape[0]):
        raise ValueError("q8 latent: latent_min must be float32 of shape (%d, z) for data of shape %s, not %s %s"
                         % (n_blocks(codes.shape[0]), codes.shape, lo.dtype, lo.shape))
    want = (n_blocks(codes.shape[0]), lo.shape[1])
    if step.dtype != np.float32 or step.shape != want:
        raise ValueError("q8 latent: latent_step must be float32 of shape %s for data of shape %s, not %s %s"
                         % (want, codes.shape, step.dtype, step.shape))
    if codes.shape[1] != row_bytes(lo.shape[1], bits):
        raise ValueError("%d-bit latent of %d columns: data must be %d bytes wide (ceil(z * b / 8)), not %d"
                         % (bits, lo.shape[1], row_bytes(lo.shape[1], bits), codes.shape[1]))
    return PackedLatent(np.ascontiguousarray(codes), np.ascontiguousarray(lo), np.ascontiguousarray(step), bits)


def from_npz(loaded):
    """Q8Latent of a loaded compressed.npz holding an 8-bit latent (np.load result or dict); ValueError when the arrays do
    not describe one (a file of fewer bits is read with `read`)"""
    q = read(loaded)
    if q.bits != 8:
        raise ValueError("compressed file holds a %d-bit latent, not a q8 one" % q.bits)
    return Q8Latent(q.codes, q.lo, q.step)
