"""Training step time of precision "fp64" against "fp32" and "split16", one JSON line on stdout:

  step_us    µs per 512-row step: CUDA events around `--steps` back-to-back bb_trainer_step calls (phase 0, no host
             synchronisation between them) after a warm-up, the three precisions alternated over `--rounds` rounds;
  epoch_s    one epoch over a 600,000-row normalised synthetic CMS table (bs 512, 1172 steps) through bb_trainer_epoch,
             alternated the same way (split16: its persistent one-kernel epoch);
  reference  the reference's `fit` per 512-row step on the host CPU: the staged reference (oracle/ref_runner.py, kind
             "reference") when it is there, else torch CPU float64 with the same model, loss and Adam (kind "port");
  card       name, power limit and max SM clock, read in this call.

    python tools/fp64_train_bench.py [--rows 600000] [--steps 200] [--rounds 3] [--ref-steps 20]
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

PRECISIONS = ("fp64", "fp32", "split16")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def make_trainer(prec, bs):
    torch.manual_seed(0)
    w, b = models.AE(24, 15).linear_tensors()
    tr = engine.Trainer(w, b, 24, 15, bs)
    tr.set_precision(prec)
    return tr


def step_us(tr, x, bs, steps, h):
    n_batches = x.shape[0] // bs
    for i in range(10):
        tr.step(x[(i % n_batches) * bs:(i % n_batches + 1) * bs], h)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
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


def reference_step_us(x_norm, bs, steps):
    """the reference's fit on the host CPU, µs per step"""
    sys.path.insert(0, ROOT)
    from oracle import ref_runner
    if ref_runner.available():
        ref_runner.fit_pass("AE", x_norm[:bs * 2], batch_size=bs)
        sec, _ = ref_runner.fit_pass("AE", x_norm[:bs * steps], batch_size=bs)
        return "reference", 1e6 * sec / steps
    # torch CPU float64: nn.Linear chain F-200-100-50-z-50-100-200-F, LeakyReLU, sum-MSE / C, torch.optim.Adam
    import torch.nn.functional as F
    torch.manual_seed(0)
    dims = (24, 200, 100, 50, 15, 50, 100, 200, 24)
    layers = [torch.nn.Linear(dims[i], dims[i + 1], dtype=torch.float64) for i in range(8)]
    params = [p for l in layers for p in l.parameters()]
    opt = torch.optim.Adam(params, lr=1e-3)
    data = torch.tensor(x_norm[:bs * steps], dtype=torch.float64)

    def one(xb):
        opt.zero_grad()
        h = xb
        for i, l in enumerate(layers):
            h = l(h)
            if i not in (3, 7):
                h = F.leaky_relu(h)
        loss = torch.sum((h - xb) ** 2) / xb.shape[1]
        loss.backward()
        opt.step()

    one(data[:bs])
    t0 = time.perf_counter()
    for i in range(steps):
        one(data[i * bs:(i + 1) * bs])
    return "port", 1e6 * (time.perf_counter() - t0) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=600_000)
    ap.add_argument("--bs", type=int, default=512)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ref-steps", type=int, default=20)
    args = ap.parse_args()
    engine.require_cuda()
    res = {"card": card(), "rows": args.rows, "batch": args.bs, "steps_per_epoch": (args.rows + args.bs - 1) // args.bs}
    x = synth.cms_table_device(args.rows, seed=1, device="cuda")
    mn, mx = engine.colminmax(x)
    xt = engine.normalize_table(x, mn, mx - mn)
    h = engine.make_hyper(lr=1e-3)
    trainers = {p: make_trainer(p, args.bs) for p in PRECISIONS}
    for p in PRECISIONS:  # warm-up of every path: module load, first launches
        trainers[p].epoch(xt[:args.bs * 20], args.bs, h)
    steps = {p: [] for p in PRECISIONS}
    epochs = {p: [] for p in PRECISIONS}
    for _ in range(args.rounds):
        for p in PRECISIONS:
            steps[p].append(step_us(trainers[p], xt, args.bs, args.steps, h))
        for p in PRECISIONS:
            epochs[p].append(epoch_s(trainers[p], xt, args.bs, h))
    res["step_us"] = {p: {"median": float(np.median(v)), "all": [round(t, 2) for t in v]} for p, v in steps.items()}
    res["epoch_s"] = {p: {"median": float(np.median(v)), "all": [round(t, 4) for t in v]} for p, v in epochs.items()}
    kind, us = reference_step_us(xt[:args.bs * args.ref_steps].cpu().numpy(), args.bs, args.ref_steps)
    res["reference_fit"] = {"kind": kind, "step_us": us, "cpu_threads": torch.get_num_threads()}
    res["fp64_vs_reference_step"] = us / res["step_us"]["fp64"]["median"]
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
