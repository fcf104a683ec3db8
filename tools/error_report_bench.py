"""error_report = True on the device, one JSON document (printed, and written to --out):

  card      name, power limit and max SM clock, read in this call (before and after)
  kernel    bb_error_stats on resident [rows, 24] CMS tables (x and y, 2 x 9.6 GB float32 or 2 x 19 GB float64 at 100M rows,
            far beyond L2): ms per call (CUDA events around --reps calls, after a warm-up call), the bytes it must read
            (2 x 24 x itemsize per row) over that time, against 7.7 TB/s; float32 and float64
  compress  helper.compress of a pageable [rows, 24] CMS table with error_report off and on, alternated over --rounds rounds
            (median, min, max seconds): latent "auto" / float64, "q4", and precision "fp64" on the float64 table
  mirror    tests/error_report_ref.record (numpy, one host thread) on --mirror-rows rows, seconds

The model is the CMS AE of tests/golden/ae_cms.npz; the tables are synth.cms_table with y = x plus noise for the kernel.

    python tools/error_report_bench.py [--rows 100000000] [--compress-rows 100000000] [--mirror-rows 600000] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(ROOT, "tests"))
from baler_b200 import engine, synth  # noqa: E402
from baler_b200.modules import helper  # noqa: E402

HBM_BYTES_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def kernel(rows, dtype, reps):
    x = synth.cms_table_device(rows).to(dtype)
    y = x + 1e-3 * torch.randn(x.shape, device="cuda", dtype=dtype)
    scale = torch.ones(24, dtype=torch.float64, device="cuda")
    engine.error_stats(x, y, scale_range=scale)  # warm-up (scratch, module load)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    from baler_b200 import _lib
    ctx = engine.get_context()
    rec = torch.empty(24 * 24, dtype=torch.int64, device="cuda")
    bb = _lib.BB_F64 if dtype == torch.float64 else _lib.BB_F32
    stream = engine._stream(ctx)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(reps):
        _lib.check(_lib.lib().bb_error_stats(ctx.handle, x.data_ptr(), bb, y.data_ptr(), bb, rows, 24, 0, None, None,
                                             scale.data_ptr(), None, rec.data_ptr(), stream), "bb_error_stats")
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / reps
    nbytes = 2 * rows * 24 * x.element_size()
    del x, y
    torch.cuda.empty_cache()
    return {"dtype": str(dtype).replace("torch.", ""), "rows": rows, "ms": ms, "ms_per_100M_rows": ms * 1e8 / rows,
            "bytes": nbytes, "TB_s": nbytes / (ms * 1e-3) / 1e12, "share_of_7.7TB_s": nbytes / (ms * 1e-3) / HBM_BYTES_S}


def compress(rows, rounds, tmp):
    from baler_b200.modules import models
    g = np.load(os.path.join(ROOT, "tests", "golden", "ae_cms.npz"))
    model_path = os.path.join(tmp, "model.pt")
    m = models.AE(24, 15)
    m.load_state_dict({k[3:]: torch.from_numpy(np.asarray(g[k])) for k in g.files if k.startswith("sd/")})
    torch.save(m.state_dict(), model_path)
    table = synth.cms_table(rows, seed=5)
    feats = np.stack([table.min(axis=0), table.max(axis=0) - table.min(axis=0)])
    out = {}
    for name, latent, precision, f64 in (("auto_float64", None, "auto", False), ("q4", "q4", "auto", False),
                                         ("fp64", None, "fp64", True)):
        path = os.path.join(tmp, "t%s.npz" % name)
        np.savez(path, data=table.astype(np.float64) if f64 else table, names=synth.CMS_NAMES)
        times = {False: [], True: []}
        for _ in range(rounds):
            for rep in (False, True):
                cfg = SimpleNamespace(input_path=path, data_dimension=1, compression_ratio=1.6, apply_normalization=True,
                                      custom_norm=False, model_name="AE", latent_dtype=latent, precision=precision,
                                      save_error_bounded_deltas=False, batch_size=512, error_report=rep)
                torch.cuda.synchronize()
                t = time.perf_counter()
                helper.compress(model_path, cfg, renormalize_features=feats if rep else None)
                torch.cuda.synchronize()
                times[rep].append(time.perf_counter() - t)
        os.remove(path)
        out[name] = {("report_on" if k else "report_off"): {"median_s": statistics.median(v), "min_s": min(v), "max_s": max(v)}
                     for k, v in times.items()}
        out[name]["rows"] = rows
    return out


def mirror(rows):
    import error_report_ref as ref
    x = synth.cms_table(rows, seed=6).astype(np.float64)
    y = x + 1e-3 * np.random.default_rng(0).standard_normal(x.shape)
    t = time.perf_counter()
    ref.record(x, y, scale_range=np.ones(24))
    return {"rows": rows, "s": time.perf_counter() - t}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--compress-rows", type=int, default=100_000_000)
    ap.add_argument("--mirror-rows", type=int, default=600_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args()
    doc = {"card_before": card()}
    doc["kernel"] = [kernel(a.rows, torch.float32, a.reps), kernel(a.rows, torch.float64, a.reps)]
    with tempfile.TemporaryDirectory() as tmp:
        doc["compress"] = compress(a.compress_rows, a.rounds, tmp) if a.compress_rows else None
    doc["mirror"] = mirror(a.mirror_rows)
    doc["card_after"] = card()
    text = json.dumps(doc)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
