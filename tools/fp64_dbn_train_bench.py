"""AE_Dropout_BN training step time under precision "fp64" against "fp32" and "split16", one JSON line on stdout:

  step_us     µs per 512-row step: CUDA events around `--steps` back-to-back bb_trainer_step calls (phase 0, no host
              synchronisation between them) after a warm-up, alternated over `--rounds` rounds, for
              fp64_masks (injected keep-masks), fp64_philox, fp64_torch (masks drawn on the device from torch's
              generator, on a side stream one step ahead), fp32 and split16 (Philox);
  mask_kernel torch.profiler in a run of its own: mean device time of the mask kernel and of the float64 step kernel per
              step, and whether the torch stream's step costs more than the Philox one (masks not hidden);
  epoch_s     one epoch over a 600,000-row normalised synthetic CMS table (bs 512) through bb_trainer_epoch;
  host        the host CPU: torch's bernoulli_ for one 512-row step's four masks, and one step of the torch CPU float64
              twin of the reference's loop (tests/dbn_reference.py);
  card        name, power limit and max SM clock, read in this call.

    python tools/fp64_dbn_train_bench.py [--rows 600000] [--steps 200] [--rounds 3]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
from baler_b200 import engine, synth  # noqa: E402
from baler_b200.modules import models  # noqa: E402

VARIANTS = ("fp64_masks", "fp64_philox", "fp64_torch", "fp32", "split16")
WIDTHS, PS = (200, 100, 50, 15), (0.5, 0.4, 0.3, 0.2)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def make_trainer(variant, bs):
    torch.manual_seed(0)
    model = models.AE_Dropout_BN(24, 15)
    w, b = model.linear_tensors()
    tr = engine.Trainer(w, b, 24, 15, bs, bn=model.bn_tensors())
    tr.set_precision("fp64" if variant.startswith("fp64") else variant)
    if variant == "fp64_masks":
        g = torch.Generator().manual_seed(1)
        tr.set_dropout(masks=[(torch.rand(bs, n, generator=g) < 1 - p).to(torch.uint8).cuda() for n, p in zip(WIDTHS, PS)])
    elif variant == "fp64_torch":
        tr.set_dropout_torch(torch.Generator().manual_seed(2))
    else:
        tr.set_dropout(seed=3)
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


def kernel_times(x, bs, h, steps=50):
    """mean device µs per step of the mask kernel and of the float64 AE_Dropout_BN step kernel (torch.profiler)"""
    from torch.profiler import ProfilerActivity, profile
    tr = make_trainer("fp64_torch", bs)
    for i in range(5):
        tr.step(x[i * bs:(i + 1) * bs], h)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            tr.step(x[i * bs:(i + 1) * bs], h)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for key, name in (("mt_dropout_kernel", "mask_us"), ("train_dbn_f64_kernel", "dbn_step_kernel_us")):
            if key in ev.key:
                dt = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                out[name] = dt / ev.count
    return out


def host_costs(x_norm, bs, reps=20):
    t = torch.empty(0)
    t0 = time.perf_counter()
    for _ in range(reps):
        for n, p in zip(WIDTHS, PS):
            t = torch.empty(bs, n, dtype=torch.float64).bernoulli_(1 - p)
    bern = 1e6 * (time.perf_counter() - t0) / reps
    from dbn_reference import DbnTwin, loss_fn
    torch.manual_seed(0)
    twin = DbnTwin(24, 15)
    opt = torch.optim.Adam(twin.parameters(), lr=1e-3)
    xb = torch.from_numpy(x_norm[:bs].astype(np.float64))
    twin.train()

    def one():
        opt.zero_grad()
        loss = loss_fn(twin(xb), xb)
        loss.backward()
        opt.step()
    one()
    t0 = time.perf_counter()
    for _ in range(reps):
        one()
    return {"bernoulli_us_per_step": bern, "twin_step_us": 1e6 * (time.perf_counter() - t0) / reps,
            "cpu_threads": torch.get_num_threads()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=600_000)
    ap.add_argument("--bs", type=int, default=512)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    engine.require_cuda()
    res = {"card": card(), "rows": args.rows, "batch": args.bs, "steps_per_epoch": (args.rows + args.bs - 1) // args.bs}
    x = synth.cms_table_device(args.rows, seed=1, device="cuda")
    mn, mx = engine.colminmax(x)
    xt = engine.normalize_table(x, mn, mx - mn)
    h = engine.make_hyper(lr=1e-3)
    trainers = {v: make_trainer(v, args.bs) for v in VARIANTS}
    for v in VARIANTS:  # warm-up of every path: module load, first launches
        trainers[v].epoch(xt[:args.bs * 20], args.bs, h)
    steps = {v: [] for v in VARIANTS}
    epochs = {v: [] for v in VARIANTS}
    for _ in range(args.rounds):
        for v in VARIANTS:
            steps[v].append(step_us(trainers[v], xt, args.bs, args.steps, h))
        for v in VARIANTS:
            epochs[v].append(epoch_s(trainers[v], xt, args.bs, h))
    res["step_us"] = {v: {"median": float(np.median(s)), "all": [round(t, 2) for t in s]} for v, s in steps.items()}
    res["epoch_s"] = {v: {"median": float(np.median(s)), "all": [round(t, 4) for t in s]} for v, s in epochs.items()}
    kt = kernel_times(xt, args.bs, h)
    kt["torch_stream_overhead_us"] = res["step_us"]["fp64_torch"]["median"] - res["step_us"]["fp64_philox"]["median"]
    res["mask_kernel"] = kt
    res["host"] = host_costs(xt[:args.bs].cpu().numpy(), args.bs)
    res["card_after"] = card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
