"""The 8-bit latent of `latent_dtype = "q8"`: its one definition in Python.

The latent [N, z] is stored as uint8 codes plus a float32 pair (lo, step) per latent column and block of BLOCK_ROWS
consecutive rows, counted from row 0 of the file (the last block may be short):

    lo, hi   min / max of the block column's finite values (-0 < +0; 0 when it has none)
    step     float32((float64(hi) - float64(lo)) / 254)
    code     255 for a non-finite value (decodes to NaN); 0 when step == 0;
             else clamp(rint((float64(v) - lo) * (1.0 / float64(step))), 0, 254), every float64 operation IEEE
    value    float32(float64(lo) + float64(code) * float64(step)), within step / 2 of v plus float32 rounding

The kernels are in csrc/bb_latent_q8.cu (include/baler_b200.h: bb_latent_quantize_q8 and the *_host_q8 pipelines).
compressed.npz then holds `data` (the codes), `latent_min`, `latent_step` and `latent_block_rows`; decompress recognises the
format by `latent_step` in the file.  The arrays are plain numpy, so the file stays readable without this package.
"""
from typing import NamedTuple

import numpy as np

BLOCK_ROWS = 128
NAME = "q8"  # the latent_dtype value


class Q8Latent(NamedTuple):
    """codes uint8 [N, z], lo / step float32 [ceil(N / BLOCK_ROWS), z]: numpy arrays, or CUDA tensors on the device"""
    codes: object
    lo: object
    step: object


def n_blocks(n_rows):
    return (int(n_rows) + BLOCK_ROWS - 1) // BLOCK_ROWS


def empty(n_rows, z_dim):
    """host buffers for the 8-bit latent of n_rows rows"""
    nb = n_blocks(n_rows)
    return Q8Latent(np.empty((n_rows, z_dim), np.uint8), np.empty((nb, z_dim), np.float32),
                    np.empty((nb, z_dim), np.float32))


def rows(q, lo, hi):
    """rows [lo, hi) of a host latent; lo must start a block"""
    if lo % BLOCK_ROWS:
        raise ValueError("a slice of a q8 latent starts on a %d-row block boundary, not at row %d" % (BLOCK_ROWS, lo))
    b0, b1 = lo // BLOCK_ROWS, (hi + BLOCK_ROWS - 1) // BLOCK_ROWS
    return Q8Latent(np.ascontiguousarray(q.codes[lo:hi]), np.ascontiguousarray(q.lo[b0:b1]),
                    np.ascontiguousarray(q.step[b0:b1]))


def npz_arrays(q):
    """the compressed.npz entries of a host latent (with `names` and `normalization_features` added by the caller)"""
    return {"data": q.codes, "latent_min": q.lo, "latent_step": q.step, "latent_block_rows": np.int64(BLOCK_ROWS)}


def in_file(loaded):
    """a loaded compressed.npz holds an 8-bit latent"""
    return "latent_step" in getattr(loaded, "files", loaded)


def from_npz(loaded):
    """Q8Latent of a loaded compressed.npz (np.load result or dict); ValueError when the arrays do not describe one"""
    for key in ("data", "latent_min", "latent_step", "latent_block_rows"):
        if key not in getattr(loaded, "files", loaded):
            raise ValueError("compressed file has latent_step but no %r: not a q8 latent" % key)
    codes, lo, step = loaded["data"], loaded["latent_min"], loaded["latent_step"]
    block = np.asarray(loaded["latent_block_rows"])
    if block.size != 1 or int(block.reshape(-1)[0]) != BLOCK_ROWS:
        raise ValueError("q8 latent with blocks of %s rows; this version reads blocks of %d rows"
                         % (block.reshape(-1).tolist(), BLOCK_ROWS))
    if codes.dtype != np.uint8 or codes.ndim != 2:
        raise ValueError("q8 latent: data must be a 2-D uint8 array, not %s %s" % (codes.dtype, codes.shape))
    want = (n_blocks(codes.shape[0]), codes.shape[1])
    for name, a in (("latent_min", lo), ("latent_step", step)):
        if a.dtype != np.float32 or a.shape != want:
            raise ValueError("q8 latent: %s must be float32 of shape %s for data of shape %s, not %s %s"
                             % (name, want, codes.shape, a.dtype, a.shape))
    return Q8Latent(np.ascontiguousarray(codes), np.ascontiguousarray(lo), np.ascontiguousarray(step))

