"""loss_function_swae step time on the layer-by-layer trainer, one JSON line on stdout:

  step_us   µs per step: CUDA events around `--steps` back-to-back step calls (phase 0, no host synchronisation between
            them) after a warm-up, per round, `--rounds` rounds alternating the cases
  sort_us   device time per call of the projection sort (swd_sort_kernel up to 2048 rows, swd_radix_kernel above), from
            torch.profiler over `--steps` steps in a run of its own
  card      name, power limit and max SM clock, read in this call (before and after)

CFD_dense_AE(64, 10) at 512 / 2048 / 2049 / 4096 / 16384 rows (SWAE only); Conv_AE(25, 10) on 5x5 blocks at 600 / 4096
blocks, SWAE and the MSE step.  2000 projections, as utils.loss_function_swae draws them.

    python tools/swae_bench.py [--steps 100] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baler_b200 import engine  # noqa: E402
from baler_b200.modules import models  # noqa: E402

CASES = [("CFD_dense_AE", r, "swae") for r in (512, 2048, 2049, 4096, 16384)] + \
        [("Conv_AE", r, loss) for r in (600, 4096) for loss in ("swae", "mse")]
SORT_KERNELS = ("swd_sort_kernel", "swd_radix_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def make_case(model, rows, loss):
    """(step callable, description) with the inputs and draws on the device"""
    torch.manual_seed(0)
    if model == "CFD_dense_AE":
        m = models.CFD_dense_AE(64, 10)
        w, b = m.linear_tensors()
        tr = engine.LayeredTrainer(w, b, ["leaky", "leaky", "leaky", "none"] * 2, rows)
        x = torch.rand((rows, 64), device="cuda")
    else:
        m = models.Conv_AE(25, 10)
        sp = m.training_spec(5, 5)
        tr = engine.LayeredTrainer(sp["weights"], sp["biases"], sp["acts"], rows, dims=sp["dims"], w_maps=sp["w_maps"],
                                   bn=sp["bn"], loss_columns=1)
        x = torch.rand((rows, 25), device="cuda")
    prior = torch.randn((rows, 10), device="cuda")
    proj = torch.randn((2000, 10), device="cuda")
    proj = (proj / proj.norm(dim=1, keepdim=True)).contiguous()
    h = engine.make_hyper(lr=1e-4)
    if loss == "mse":
        return lambda: tr.step(x, h)
    return lambda: tr.step_swae(x, h, prior, proj, latent_layer=m.latent_layer)


def step_us(step, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / steps


def sort_us(step, steps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
    total, calls = 0.0, 0
    for ev in prof.key_averages():
        if any(k in ev.key for k in SORT_KERNELS):
            total += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            calls += ev.count
    return total / calls if calls else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    engine.require_cuda()
    res = {"card": card(), "steps": args.steps, "rounds": args.rounds, "projections": 2000}
    steps = {c: make_case(*c) for c in CASES}
    for c in CASES:  # warm-up: modules, first-step allocations
        for _ in range(5):
            steps[c]()
    times = {c: [] for c in CASES}
    for _ in range(args.rounds):
        for c in CASES:
            times[c].append(step_us(steps[c], args.steps))
    res["cases"] = []
    for c in CASES:
        entry = {"model": c[0], "rows": c[1], "loss": c[2], "step_us": [round(t, 1) for t in times[c]]}
        if c[2] == "swae":
            entry["sort_us"] = round(sort_us(steps[c], args.steps), 1)
        res["cases"].append(entry)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
