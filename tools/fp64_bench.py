"""precision "fp64" on the CMS workload, one JSON line on stdout:

  resident   bb_encode_f32 / bb_decode_f32 with BB_PREC_FP64 on the whole synthetic CMS table generated in HBM (float32,
             normalised in the kernel; float64 latent and rows): G rows/s and the useful FP64 TFLOP/s (61,100 FLOP per
             row and direction), CUDA events around `--reps` launches after a warm-up;
  e2e        bb_compress_host + bb_decompress_host with the reference's file dtypes (float32 table in pinned memory,
             float64 latent and reconstruction in pageable arrays), BB_PREC_FP64 against BB_PREC_AUTO, alternated in
             this process, wall clock per round trip;
  errors     whole-table error of auto / fp32 / split16 / fast against the fp64 output: max|d| / max|ref| and
             ||d||2 / ||ref||2 of the latent and of the un-normalised reconstruction;
  card       name and power limit, read in this call.

    python tools/fp64_bench.py [--rows 100000000] [--e2e-rows 20000000] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from baler_b200 import engine, synth  # noqa: E402
from baler_b200.modules import models  # noqa: E402

FLOP_PER_ROW = 61_100  # 2 x (24*200 + 200*100 + 100*50 + 50*15) multiply-adds, one direction


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def err(a, ref):
    d = a.double() - ref
    return {"max_rel": float(d.abs().max() / ref.abs().max()), "l2_rel": float(d.norm() / ref.norm())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--e2e-rows", type=int, default=20_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--e2e-rounds", type=int, default=4)
    args = ap.parse_args()
    engine.require_cuda()
    g = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "ae_cms.npz"))
    m = models.AE(24, 15)
    m.load_state_dict({k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd/")})
    codec = m.eval().codec()
    res = {"card": card(), "rows": args.rows, "flop_per_row_and_direction": FLOP_PER_ROW}

    # ---- resident: whole table in HBM
    n = args.rows
    x = synth.cms_table_device(n)
    mn, mx = engine.colminmax(x)
    rg = mx - mn
    z64 = torch.empty((n, 15), dtype=torch.float64, device="cuda")
    y64 = torch.empty((n, 24), dtype=torch.float64, device="cuda")
    t_enc = timed(lambda: codec.encode(x, mn, rg, precision="fp64", out=z64), args.reps)
    t_dec = timed(lambda: codec.decode(z64, mn, rg, out=y64), args.reps)
    res["resident"] = {
        "encode_grows_s": n / t_enc / 1e9, "decode_grows_s": n / t_dec / 1e9,
        "encode_fp64_tflops": n * FLOP_PER_ROW / t_enc / 1e12, "decode_fp64_tflops": n * FLOP_PER_ROW / t_dec / 1e12,
        "encode_s": t_enc, "decode_s": t_dec}

    # ---- whole-table errors of the other precisions against fp64
    errors = {}
    for p in ("auto", "fp32", "split16", "fast"):
        if p in ("split16", "fast") and codec.auto_precision != "split16":
            continue
        z = codec.encode(x, mn, rg, precision=p)
        y = codec.decode(z, mn, rg, precision=p)
        errors[p] = {"latent": err(z, z64), "reconstruction": err(y, y64)}
        del z, y
    res["errors_vs_fp64"] = errors
    del x, z64, y64
    torch.cuda.empty_cache()

    # ---- end to end through host buffers, fp64 against auto, alternated
    ne = args.e2e_rows
    xd = synth.cms_table_device(ne)
    xh = torch.empty((ne, 24), dtype=torch.float32, pin_memory=True)
    xh.copy_(xd)
    torch.cuda.synchronize()
    del xd
    xn = xh.numpy()
    zh = np.empty((ne, 15), dtype=np.float64)
    yh = np.empty((ne, 24), dtype=np.float64)
    rates = {"fp64": [], "auto": []}
    for r in range(args.e2e_rounds + 1):  # round 0 warms both up
        for p in ("fp64", "auto"):
            t0 = time.perf_counter()
            _, feats = codec.compress_host(xn, recompute_minmax=True, z_dtype=np.float64, precision=p, out=zh)
            codec.decompress_host(zh, features=feats, y_dtype=np.float64, precision=p, out=yh)
            dt = time.perf_counter() - t0
            if r:
                rates[p].append(ne / dt / 1e6)
    res["e2e_f64_file_dtypes"] = {"rows": ne, "unit": "M rows/s (compress + decompress)",
                                   **{p: {"median": float(np.median(v)), "all": [round(a, 1) for a in v]} for p, v in rates.items()}}
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
