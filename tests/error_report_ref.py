"""numpy mirror of the error report (baler_b200/error_report.py is the definition): the error_report.Record of rows y against
raw rows x, in float64, row by row as the definition states it."""
import numpy as np

from baler_b200 import error_report


def record(x, y, row0=0, post=None, scale_range=None, int_mask=None):
    """x, y: [n, C] float32 / float64.  post: (min, range) float64 applied to y as y * range + min; scale_range: float64 [C]
    (None = 1); int_mask: [C] (non-zero = truncate y toward zero)"""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).copy()
    n, c = x.shape
    if post is not None:
        mn, rg = (np.asarray(a, dtype=np.float64) for a in post)
        y = y * rg
        y = y + mn  # (two roundings, as numpy's decompressed * range + min)
    is_int = np.zeros(c, bool) if int_mask is None else np.asarray(int_mask).astype(bool)
    y[:, is_int] = np.trunc(y[:, is_int])
    rng = np.ones(c) if scale_range is None else np.asarray(scale_range, dtype=np.float64).copy()
    rng[~(np.isfinite(rng) & (rng > 0))] = 1.0
    thr = error_report.HIST_EDGES[None, :] * rng[:, None]  # [C, 10]
    rec = error_report.Record.empty(c)
    fx, fy = np.isfinite(x), np.isfinite(y)
    rec.nonfinite_x = (~fx).sum(axis=0).astype(np.int64)
    rec.nonfinite_y = (~fy).sum(axis=0).astype(np.int64)
    for j in range(c):
        xf = x[fx[:, j], j]
        if len(xf):
            rec.x_min[j], rec.x_max[j] = xf.min(), xf.max()
        both = fx[:, j] & fy[:, j]
        rows = np.nonzero(both)[0]
        e = y[rows, j] - x[rows, j]
        a = np.abs(e)
        rec.count[j] = len(rows)
        rec.sum_e[j], rec.sum_e2[j] = e.sum(), (e * e).sum()
        if len(rows):
            k = int(np.argmax(a))  # (the first, i.e. smallest, row among equal maxima)
            rec.err_max_abs[j], rec.err_max_row[j] = a[k], row0 + rows[k]
        nz = x[rows, j] != 0
        r = (100.0 * e[nz]) / x[rows, j][nz]
        rec.response_count[j] = int(nz.sum())
        rec.sum_r[j], rec.sum_r2[j] = r.sum(), (r * r).sum()
        rec.hist[j] = np.bincount((a[:, None] > thr[j][None, :]).sum(axis=1), minlength=error_report.N_BINS)
        if is_int[j]:
            rec.int_mismatch[j] = int((y[rows, j] != x[rows, j]).sum())
    return rec


def from_files(x, y, post=None, features=None, int_mask=None):
    """the record of a whole table from the input rows and decompressed.npz rows ([N, ...] each, flattened per row): the
    training `features` ([min; range]) give the histogram's range"""
    x = np.asarray(x).reshape(len(x), -1)
    y = np.asarray(y).reshape(len(y), -1)
    scale = None if features is None else np.asarray(features, dtype=np.float64).reshape(2, -1)[1]
    return record(x, y, post=post, scale_range=scale, int_mask=int_mask)
