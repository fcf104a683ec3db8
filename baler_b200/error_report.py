"""error_report = True: the per-column error of what --mode decompress will write, measured on the GPU during --mode compress.

This module is the one definition of the report (tests/error_report_ref.py is its numpy mirror; csrc/bb_error_stats.cu the
kernel that computes a chunk's record).  All arithmetic is float64.  The columns are those of the [N, C] rows the codec sees:
the table's columns for 1-D data, block or snapshot positions for 2-D data.  x is a raw input row, y the row decompress
writes for it: the latent as stored (float16 rounding, q-codes dequantised), decoded at the configured precision,
un-normalised with the training features as helper.decompress does, integer type_list columns truncated toward zero, and
before error-bounded deltas are applied.  For each column j, over the rows where x and y are both finite, e = y - x:

  count, nonfinite_x, nonfinite_y     int64; nonfinite_* count the rows where x (resp. y) is not finite
  x_min, x_max                        over the finite x (NaN when there is none)
  err_mean, err_rms                   sum(e) / count, sqrt(sum(e^2) / count)
  err_max_abs, err_max_row            max |e| and the smallest global row attaining it (NaN and -1 when count is 0)
  response_count / _mean / _rms       Baler's response r = 100 * e / x, over the rows with x != 0
  hist [C, 11]                        |e| against edge_k * range_j for the edges 1e-9, 1e-8, ..., 0.1, 1: the bins
                                      [0, 1e-9 range], (1e-9 range, 1e-8 range], ..., (0.1 range, range], (range, inf)
  int_mismatch                        integer type_list columns: the rows where trunc(y) != x; 0 elsewhere

range_j is the training-feature range decompress un-normalises with (scale_range in the file); it is 1 when
apply_normalization is off or the range is not a positive finite number.  The histogram compares |e| with the float64
product edge_k * range_j rather than dividing, so the kernel needs no division for it.

A Record holds the mergeable sums of one chunk; merge() folds records in chunk order, then rank order; finalize() gives the
arrays of output/compressed_output/error_report.npz.
"""
import numpy as np

HIST_EDGES = np.array([1e-9, 1e-8, 1e-7, 1e-6, 1e-5, 1e-4, 1e-3, 1e-2, 1e-1, 1.0])
N_BINS = len(HIST_EDGES) + 1
# the 8-byte words per column of a device record (BB_ERROR_STATS_FIELDS, include/baler_b200.h), field-major
_INT_FIELDS = ("count", "nonfinite_x", "nonfinite_y", "response_count", "int_mismatch", "err_max_row")
_FLOAT_FIELDS = ("x_min", "x_max", "sum_e", "sum_e2", "err_max_abs", "sum_r", "sum_r2")
N_FIELDS = len(_INT_FIELDS) + N_BINS + len(_FLOAT_FIELDS)
SCOPE = "the rows decompress writes, before error-bounded deltas are applied, against the raw input rows"


class Record:
    """mergeable per-column statistics of a set of rows (int64 / float64 arrays of length C; hist is [C, 11])"""

    def __init__(self, **arrays):
        for k in _INT_FIELDS + _FLOAT_FIELDS + ("hist",):
            setattr(self, k, arrays[k])

    @property
    def n_cols(self):
        return len(self.count)

    @classmethod
    def empty(cls, n_cols):
        """the record of no rows"""
        z = np.zeros(n_cols, dtype=np.int64)
        return cls(count=z, nonfinite_x=z.copy(), nonfinite_y=z.copy(), response_count=z.copy(), int_mismatch=z.copy(),
                   err_max_row=np.full(n_cols, -1, np.int64), hist=np.zeros((n_cols, N_BINS), np.int64),
                   x_min=np.full(n_cols, np.inf), x_max=np.full(n_cols, -np.inf), sum_e=np.zeros(n_cols),
                   sum_e2=np.zeros(n_cols), err_max_abs=np.zeros(n_cols), sum_r=np.zeros(n_cols), sum_r2=np.zeros(n_cols))

    @classmethod
    def from_words(cls, words, n_cols):
        """a device record (N_FIELDS x n_cols 8-byte words, field-major) as a Record"""
        w = np.ascontiguousarray(words).view(np.int64).reshape(N_FIELDS, n_cols)
        ni = len(_INT_FIELDS)
        arrays = {k: w[i].copy() for i, k in enumerate(_INT_FIELDS)}
        arrays["hist"] = np.ascontiguousarray(w[ni:ni + N_BINS].T)
        f = w[ni + N_BINS:].copy().view(np.float64)
        arrays.update({k: f[i].copy() for i, k in enumerate(_FLOAT_FIELDS)})
        return cls(**arrays)

    def __eq__(self, other):
        return all(np.array_equal(getattr(self, k), getattr(other, k), equal_nan=k in _FLOAT_FIELDS)
                   for k in _INT_FIELDS + _FLOAT_FIELDS + ("hist",))


def merge(records):
    """one Record of the rows of `records`, folded in list order (chunk order, then rank order): counts and sums add,
    minima / maxima keep the extreme, the maximum error keeps the smallest row among equal values.  Attributes beyond the
    statistics (rows, latent_dtype, precision: set by helper.compress on a whole table's record) come from the first."""
    records = list(records)
    out = Record.empty(records[0].n_cols)
    out.__dict__.update({k: v for k, v in records[0].__dict__.items() if not hasattr(out, k)})
    for r in records:
        for k in ("count", "nonfinite_x", "nonfinite_y", "response_count", "int_mismatch", "hist", "sum_e", "sum_e2", "sum_r",
                  "sum_r2"):
            setattr(out, k, getattr(out, k) + getattr(r, k))
        out.x_min = np.where(r.x_min < out.x_min, r.x_min, out.x_min)
        out.x_max = np.where(r.x_max > out.x_max, r.x_max, out.x_max)
        take = (r.err_max_row >= 0) & ((r.err_max_abs > out.err_max_abs) | (out.err_max_row < 0) |
                                       ((r.err_max_abs == out.err_max_abs) & (r.err_max_row < out.err_max_row)))
        out.err_max_abs = np.where(take, r.err_max_abs, out.err_max_abs)
        out.err_max_row = np.where(take, r.err_max_row, out.err_max_row)
    return out


def enabled(config):
    """config.error_report as a bool (absent = False); ValueError for anything but a bool"""
    value = getattr(config, "error_report", False)
    if not isinstance(value, (bool, np.bool_)):
        raise ValueError("error_report must be True or False, not %r" % (value,))
    return bool(value)


def scale_range(features, n_cols):
    """float64 range_j of the histogram: the [min; range] features' range, 1 where it is not a positive finite number (and
    everywhere without features)"""
    if features is None:
        return np.ones(n_cols)
    rg = np.asarray(features, dtype=np.float64).reshape(2, -1)[1].copy()
    rg[~(np.isfinite(rg) & (rg > 0))] = 1.0
    return rg


def int_columns(config, row_shape):
    """uint8 mask over the flattened rows of shape `row_shape` (what perform_decompression writes per row, before any
    block reshape) of the integer type_list entries, which decompress truncates toward zero (baler.py:426-435), or None"""
    types = getattr(config, "type_list", None)
    if types is None:
        return None
    mask = np.zeros(row_shape, dtype=np.uint8)
    for index, t in enumerate(types):
        if np.dtype(t).kind in "iu":
            mask[index] = 1
    return mask.reshape(-1) if mask.any() else None


def finalize(rec, names, scale, rows, latent_dtype, precision):
    """the arrays of error_report.npz for a merged Record"""
    with np.errstate(divide="ignore", invalid="ignore"):
        cnt, rc = rec.count.astype(np.float64), rec.response_count.astype(np.float64)
        out = dict(
            names=np.asarray(names), count=rec.count, nonfinite_x=rec.nonfinite_x, nonfinite_y=rec.nonfinite_y,
            x_min=np.where(np.isfinite(rec.x_min), rec.x_min, np.nan), x_max=np.where(np.isfinite(rec.x_max), rec.x_max, np.nan),
            err_mean=np.where(rec.count > 0, rec.sum_e / cnt, np.nan), err_rms=np.where(rec.count > 0, np.sqrt(rec.sum_e2 / cnt), np.nan),
            err_max_abs=np.where(rec.count > 0, rec.err_max_abs, np.nan), err_max_row=rec.err_max_row,
            response_count=rec.response_count, response_mean=np.where(rec.response_count > 0, rec.sum_r / rc, np.nan),
            response_rms=np.where(rec.response_count > 0, np.sqrt(rec.sum_r2 / rc), np.nan),
            hist=rec.hist, hist_edges=HIST_EDGES, scale_range=np.asarray(scale, dtype=np.float64), int_mismatch=rec.int_mismatch,
            sum_e=rec.sum_e, sum_e2=rec.sum_e2, rows=np.int64(rows), latent_dtype=np.str_(latent_dtype),
            precision=np.str_(precision), scope=np.str_(SCOPE))
    return out


def summary(report, worst=10):
    """the lines compress prints: mean and worst err_rms / range over the columns, the largest err_max_abs / range, and the
    `worst` columns by err_rms / range"""
    rel = report["err_rms"] / report["scale_range"]
    peak = report["err_max_abs"] / report["scale_range"]
    ok = np.isfinite(rel)
    lines = ["Error report (%s; %d rows, latent %s, precision %s):" % (SCOPE, int(report["rows"]), report["latent_dtype"],
                                                                      report["precision"])]
    if not ok.any():
        return "\n".join(lines + ["  no column has a finite input and output row"])
    lines.append("  err_rms / range: mean %.6g, worst %.6g; largest err_max_abs / range %.6g"
                 % (rel[ok].mean(), rel[ok].max(), np.nanmax(peak)))
    lines.append("  worst columns (err_rms / range, err_max_abs / range at row):")
    for j in np.argsort(-np.where(ok, rel, -np.inf), kind="stable")[:min(worst, int(ok.sum()))]:
        lines.append("    %-24s %.6g  %.6g at %d" % (report["names"][j], rel[j], peak[j], report["err_max_row"][j]))
    return "\n".join(lines)
