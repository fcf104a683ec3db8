"""AE_Dropout_BN training step time on the fused step (tensor cores, batches up to 16 rows x SMs) and on the
layer-by-layer trainer (any batch), one JSON line on stdout:

  step_us   µs per step: CUDA events around `--steps` back-to-back step calls (phase 0, Philox dropout, no host
            synchronisation between them) after a warm-up, alternated over `--rounds` rounds; also M samples/s
  epoch_s   one epoch over a `--rows`-row normalised synthetic CMS table through the trainer's epoch call
  card      name, power limit and max SM clock, read in this call (before and after)

fused: batch 512 and 2368; layered: batch 2369, 4096, 8192 and 16384 (the CMS shape, 24 columns, latent 15).

    python tools/dbn_large_batch_bench.py [--rows 600000] [--steps 200] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baler_b200 import engine, synth  # noqa: E402
from baler_b200.modules import models  # noqa: E402

CASES = (("fused", 512), ("fused", 2368), ("layered", 2369), ("layered", 4096), ("layered", 8192), ("layered", 16384))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def make_trainer(kind, bs):
    torch.manual_seed(0)
    model = models.AE_Dropout_BN(24, 15)
    w, b = model.linear_tensors()
    if kind == "fused":
        tr = engine.Trainer(w, b, 24, 15, bs, bn=model.bn_tensors())
    else:
        tr = engine.LayeredTrainer.dbn(w, b, 24, 15, bs, model.bn_tensors())
    tr.set_dropout(seed=3)
    return tr


def step_us(tr, x, bs, steps, h):
    n_batches = x.shape[0] // bs
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        tr.step(x[(i % n_batches) * bs:(i % n_batches + 1) * bs], h)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / steps


def epoch_s(tr, x, bs, h):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tr.epoch(x, bs, h)  # returns after synchronising its stream
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=600_000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    engine.require_cuda()
    res = {"card": card(), "rows": args.rows, "steps": args.steps, "rounds": args.rounds}
    x = synth.cms_table_device(args.rows, seed=1, device="cuda")
    mn, mx = engine.colminmax(x)
    xt = engine.normalize_table(x, mn, mx - mn)
    h = engine.make_hyper(lr=1e-3)
    names = ["%s_%d" % c for c in CASES]
    trainers = {n: make_trainer(k, bs) for n, (k, bs) in zip(names, CASES)}
    for n, (k, bs) in zip(names, CASES):  # warm-up of every path and shape: module load, first launches
        trainers[n].epoch(xt[:bs * 10], bs, h)
    steps = {n: [] for n in names}
    epochs = {n: [] for n in names}
    for _ in range(args.rounds):
        for n, (k, bs) in zip(names, CASES):
            steps[n].append(step_us(trainers[n], xt, bs, args.steps, h))
        for n, (k, bs) in zip(names, CASES):
            epochs[n].append(epoch_s(trainers[n], xt, bs, h))
    res["step_us"] = {}
    for n, (k, bs) in zip(names, CASES):
        med = float(np.median(steps[n]))
        res["step_us"][n] = {"median": med, "all": [round(t, 2) for t in steps[n]], "msamples_per_s": bs / med}
    res["epoch_s"] = {n: {"median": float(np.median(s)), "all": [round(t, 4) for t in s]} for n, s in epochs.items()}
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
