"""The 8-bit latent (latent_dtype "q8") on the device, one JSON document (printed, and written to --out):

  kernels     latent_q8_quantize_kernel / latent_q8_dequantize_kernel on a resident [rows, 15] float32 latent: ms per call
              (CUDA events around --reps calls), bytes the format needs per call (quantise: 4z read, z + 8z / 128
              written per row; dequantise the reverse) and those bytes over the time, against 7.7 TB/s
  encode      resident AE 24 -> 15 encode (split16, chain_tc4) alone and encode + quantise, alternated over --rounds rounds
  host        bb_compress_host / bb_decompress_host rows/s with float16 and float64 latents and the *_q8 pipelines on
              pageable host tables, alternated over --rounds rounds: median, min, max
  file_bytes  compressed.npz sizes (np.savez) at --file-rows rows for each latent, and the input file
  error       reconstruction error against the original table at --file-rows rows for float64, float16 and q8 latents:
              per-column RMS / range (mean and max over columns) and the latent's own max error / step
  card        name, power limit and max SM clock, read in this call

The model is the CMS AE of tests/golden/ae_cms.npz (the reference's AE 24 -> 15 after its training run on the synthetic
CMS table); the tables are synth.cms_table.

    python tools/latent_q8_bench.py [--rows 100000000] [--file-rows 600000] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baler_b200 import engine, latent_q8, synth  # noqa: E402
from baler_b200.modules import models  # noqa: E402

HBM_BYTES_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def model():
    g = np.load(os.path.join(ROOT, "tests", "golden", "ae_cms.npz"))
    sd = {k[3:]: torch.from_numpy(np.asarray(g[k])) for k in g.files if k.startswith("sd/")}
    m = models.AE(24, 15)
    m.load_state_dict(sd)
    return m.eval()


def timed(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def host_table(rows):
    out = np.empty((rows, 24), dtype=np.float32)
    step = 20_000_000
    for r0 in range(0, rows, step):
        out[r0:r0 + step] = synth.cms_table_device(min(step, rows - r0), seed=1 + r0 // step).cpu().numpy()
    return out


def spread(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}


def kernels(codec, rows, reps):
    z_dim = codec.z_dim
    z = torch.randn((rows, z_dim), device="cuda")
    q = codec.quantize_q8(z)  # warm-up (and the buffers the caching allocator then reuses)
    codec.dequantize_q8(q)
    tq = timed(lambda: codec.quantize_q8(z), reps)
    td = timed(lambda: codec.dequantize_q8(q), reps)
    small = rows * z_dim + 2 * 4 * z_dim * latent_q8.n_blocks(rows)
    big = 4 * rows * z_dim
    out = {}
    for name, ms in (("quantize", tq), ("dequantize", td)):
        byt = big + small
        out[name] = {"ms": ms, "bytes": byt, "bytes_per_s": byt / (ms * 1e-3), "of_hbm": byt / (ms * 1e-3) / HBM_BYTES_S}
    del z, q
    torch.cuda.empty_cache()
    return out


def encode(codec, rows, rounds):
    x = synth.cms_table_device(rows, seed=5)
    mn, mx = engine.colminmax(x)
    rg = mx - mn
    zbuf = torch.empty((rows, codec.z_dim), device="cuda")
    codec.encode(x, mn, rg, out=zbuf)
    codec.quantize_q8(zbuf)
    alone, both = [], []
    for _ in range(rounds):
        alone.append(timed(lambda: codec.encode(x, mn, rg, out=zbuf)))
        both.append(timed(lambda: codec.quantize_q8(codec.encode(x, mn, rg, out=zbuf))))
    del x, zbuf
    torch.cuda.empty_cache()
    return {"rows": rows, "encode_ms": spread(alone), "encode_quantize_ms": spread(both),
            "overhead": float(np.median(both) / np.median(alone) - 1)}


def host(codec, rows, rounds):
    x = host_table(rows)
    feats = np.zeros((2, 24), np.float32)
    codec.compress_host(x[:1 << 20], features=feats, recompute_minmax=True)  # features of the table, warm-up
    _, feats = codec.compress_host(x, features=feats, recompute_minmax=True)
    z16 = np.empty((rows, codec.z_dim), np.float16)
    z64 = np.empty((rows, codec.z_dim), np.float64)
    q = latent_q8.empty(rows, codec.z_dim)
    y = np.empty((rows, 24), np.float64)
    ops = {
        "compress_float16": lambda: codec.compress_host(x, features=feats, out=z16),
        "compress_float64": lambda: codec.compress_host(x, features=feats, out=z64),
        "compress_q8": lambda: codec.compress_host_q8(x, features=feats, out=q),
        "decompress_float16": lambda: codec.decompress_host(z16, features=feats, out=y),
        "decompress_float64": lambda: codec.decompress_host(z64, features=feats, out=y),
        "decompress_q8": lambda: codec.decompress_host_q8(q, features=feats, out=y),
    }
    for fn in ops.values():  # warm-up: staging, pinned buffers, page faults of the outputs
        fn()
    res = {k: [] for k in ops}
    for _ in range(rounds):
        for k, fn in ops.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            res[k].append(rows / (time.perf_counter() - t0))
    return {"rows": rows, "rows_per_s": {k: spread(v) for k, v in res.items()}}


def files_and_error(codec, rows):
    x = synth.cms_table(rows, seed=17)
    mn, mx = x.min(axis=0), x.max(axis=0)
    feats = np.stack([mn, mx - mn]).astype(np.float32)
    names = np.array(synth.CMS_NAMES)
    z32, _ = codec.compress_host(x, features=feats)
    lat = {"float64": codec.compress_host(x, features=feats, z_dtype=np.float64)[0],
           "float16": codec.compress_host(x, features=feats, z_dtype=np.float16)[0],
           "q8": codec.compress_host_q8(x, features=feats)[0]}
    sizes, err = {}, {}
    with tempfile.TemporaryDirectory() as d:
        np.savez(os.path.join(d, "input.npz"), data=x, names=names)
        sizes["input"] = os.path.getsize(os.path.join(d, "input.npz"))
        for k, z in lat.items():
            arrays = latent_q8.npz_arrays(z) if k == "q8" else {"data": z}
            p = os.path.join(d, k + ".npz")
            np.savez(p, **arrays, names=names, normalization_features=feats)
            sizes[k] = os.path.getsize(p)
    rng = (mx - mn).astype(np.float64)
    for k, z in lat.items():
        y = (codec.decompress_host_q8(z, features=feats) if k == "q8" else codec.decompress_host(z, features=feats))
        rms = np.sqrt(np.mean((y - x.astype(np.float64)) ** 2, axis=0)) / np.where(rng > 0, rng, 1)
        e = {"rms_over_range_mean": float(rms.mean()), "rms_over_range_max": float(rms.max())}
        if k == "q8":
            back = codec.dequantize_q8(tuple(torch.from_numpy(a).cuda() for a in z)).cpu().numpy()
            st = z.step.astype(np.float64)[np.arange(rows) // latent_q8.BLOCK_ROWS]
            e["latent_max_err_over_step"] = float(np.max(np.abs(back.astype(np.float64) - z32) / np.where(st > 0, st, 1)))
        err[k] = e
    return {"rows": rows, "bytes": sizes, "bytes_per_row": {k: v / rows for k, v in sizes.items()}}, err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--file-rows", type=int, default=600_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.require_cuda()
    with open("/proc/meminfo") as f:  # the host pipelines hold ~450 bytes per row (table, three latents, float64 rows)
        avail = int([l.split()[1] for l in f if l.startswith("MemAvailable")][0]) * 1024
    a.rows = min(a.rows, int(avail * 0.6) // 450 // (1 << 20) * (1 << 20))
    codec = model().codec()
    res = {"card": card(), "model": "AE 24 -> 15 (tests/golden/ae_cms.npz)"}
    res["file_bytes"], res["error"] = files_and_error(codec, a.file_rows)
    res["kernels"] = kernels(codec, a.rows, a.reps)
    res["kernels"]["rows"] = a.rows
    res["encode"] = encode(codec, a.rows, a.rounds)
    res["host"] = host(codec, a.rows, a.rounds)
    res["card_after"] = card()
    text = json.dumps(res)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
