"""Resident vs streamed training epochs (a table in device memory vs the same table streamed from host memory through two
device windows, bb_trainer_epoch_host), one JSON line on stdout:

  epoch_s    seconds per epoch: CUDA events around one epoch call, resident and streamed alternated over `--rounds`
             rounds, each round from a fresh trainer with the same initial weights
  bit_equal  the epoch losses of the two placements are the same bits in every round
  window     rows per device window (training.stream_window_rows under the device's real budget)
  mem_high   device memory the run holds at its high-water mark (total - free from cudaMemGetInfo, sampled around every
             epoch, less what was in use before): trainer scratch plus the table (resident) or the two windows (streamed)
  card       name, power limit and max SM clock, read in this call

Cases (the CMS shape, 24 columns, latent 15): AE split16 at batch 512, AE_Dropout_BN fused at batch 2368, AE fp64 at batch
512 (float64 table); each at `--rows` rows (default 600k and 100M).  A size whose host tables would take more than half of
the host's memory is skipped and reported as such.

    python tools/stream_train_bench.py [--rows 600000 100000000] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baler_b200 import engine, synth  # noqa: E402
from baler_b200.modules import models, training  # noqa: E402

CASES = (("ae_split16", 512), ("dbn_fused", 2368), ("ae_fp64", 512))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def host_table(rows, dtype):
    """normalised synthetic CMS table in host memory, generated on the device in slices"""
    out = np.empty((rows, 24), dtype=dtype)
    step = 20_000_000
    mn = mx = None
    for r0 in range(0, rows, step):  # column min / max of the whole table first, then the normalised slices
        x = synth.cms_table_device(min(step, rows - r0), seed=1 + r0 // step)
        a, b = engine.colminmax(x)
        mn, mx = (a, b) if mn is None else (torch.minimum(mn, a), torch.maximum(mx, b))
    for r0 in range(0, rows, step):
        x = synth.cms_table_device(min(step, rows - r0), seed=1 + r0 // step)
        out[r0:r0 + len(x)] = engine.normalize_table(x, mn, mx - mn).to(torch.float64 if dtype == np.float64 else torch.float32).cpu().numpy()
    return out


def make(case, bs):
    torch.manual_seed(0)
    if case == "dbn_fused":
        m = models.AE_Dropout_BN(24, 15)
        w, b = m.linear_tensors()
        tr = engine.Trainer(w, b, 24, 15, bs, bn=m.bn_tensors())
        tr.set_dropout(seed=3)
        return tr
    w, b = models.AE(24, 15).linear_tensors()
    tr = engine.Trainer(w, b, 24, 15, bs)
    if case == "ae_fp64":
        tr.set_precision("fp64")
    return tr


def in_use():
    free, total = torch.cuda.mem_get_info()
    return total - free


def timed_epoch(tr, x, bs, h, window):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    loss = tr.epoch(x, bs, h, window) if window else tr.epoch(x, bs, h)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3, loss


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[600_000, 100_000_000])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    engine.require_cuda()
    host_mem = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    res = {"card": card(), "rounds": args.rounds, "host_mem": host_mem, "cases": {}}
    h = engine.make_hyper(lr=1e-3)
    for rows in args.rows:
        for case, bs in CASES:
            name = "%s_b%d_%d" % (case, bs, rows)
            dtype = np.float64 if case == "ae_fp64" else np.float32
            if rows * 24 * np.dtype(dtype).itemsize > host_mem // 2:
                res["cases"][name] = {"skipped": "host table above half of host memory"}
                continue
            table = host_table(rows, dtype)
            dev = torch.from_numpy(table).cuda()
            warm = make(case, bs)  # module load and first launches of both paths
            warm.epoch(dev[:bs * 8], bs, h)
            warm.epoch(table[:bs * 8], bs, h, 4 * bs)
            del warm
            window = training.stream_window_rows(table.strides[0], bs, training.device_table_budget())
            times = {"resident": [], "streamed": []}
            losses = {"resident": [], "streamed": []}
            base = in_use()  # (the resident copy of the table is already allocated: counted for the resident runs below)
            high = {"resident": 0, "streamed": 0}
            for _ in range(args.rounds):
                for kind in ("resident", "streamed"):
                    tr = make(case, bs)
                    high[kind] = max(high[kind], in_use())
                    t, loss = timed_epoch(tr, dev if kind == "resident" else table, bs, h,
                                          None if kind == "resident" else window)
                    high[kind] = max(high[kind], in_use())
                    times[kind].append(t)
                    losses[kind].append(loss)
                    del tr
            r, s = float(np.median(times["resident"])), float(np.median(times["streamed"]))
            res["cases"][name] = {
                "rows": rows, "batch": bs, "window": window, "table_bytes": table.nbytes,
                "epoch_s": {k: {"median": float(np.median(v)), "all": [round(t, 4) for t in v]} for k, v in times.items()},
                "streamed_over_resident": s / r,
                "bit_equal": all(a == b for a, b in zip(losses["resident"], losses["streamed"])),
                "mem_high": {"resident": high["resident"] - base + table.nbytes, "streamed": high["streamed"] - base}}
            print(name, json.dumps(res["cases"][name]), file=sys.stderr)
            del dev, table
            torch.cuda.empty_cache()
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
