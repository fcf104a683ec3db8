#!/usr/bin/env python
"""Headline benchmark: CMS AE (24 -> 15) compress + decompress of a synthetic 100M-row x 24-col float32
table per GPU (BASELINE.json configs[1]), plus one training epoch as a secondary line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows R] [--dump-outputs DIR]

One step = one pass of the hot path over the table: column min/max -> normalise+encode -> latent, then
decode+un-normalise -> reconstruction.  `value` = rows / step time with the table resident in HBM.
`--dump-outputs DIR` writes what the last timed step computed (features, and latent and reconstruction at a fixed
sample of rows) as .npy files, so that two builds run with the same arguments can be compared output for output.
`e2e` = the same pass through the C-ABI host entry points (bb_compress_host / bb_decompress_host) with
pinned HOST buffers, H2D / D2H copies inside the timed region.  N > 1: one process per GPU (torchrun), the
table is row-sharded (100M rows per GPU, weak scaling), the only exchange is the 2 x 24 column min / max.
`--impl reference` times the UNMODIFIED reference (oracle/_ref, staged by oracle/stage_ref.py) on the host cores:
helper.compress + helper.decompress as shipped on a bounded sample of the same workload (the restatement on torch CPU,
oracle/torch_port.py, when the staged package is absent; it is always reported as the labelled best case).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_ROW = 61100          # SURVEY 8(d): 2 * (24*200 + 200*100 + 100*50 + 50*15) per direction
BYTES_PER_ROW = 156           # 96 in + 60 out (fp32 latent) per direction
METRIC = "compress+decompress rows/s (CMS AE 24->15, table resident in HBM)"
DUMP_ROWS = 1 << 18           # rows --dump-outputs samples: 41 MB of float32 latent + reconstruction whatever --rows
DUMP_SEED = 0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "tflops_burst": d["bf16_tflops"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1590.0, "src": "fallback"}


def golden_state_dict():
    g = np.load(os.path.join(ROOT, "tests", "golden", "ae_cms.npz"))
    return {k[3:]: g[k] for k in g.files if k.startswith("sd/")}


def dump_rows(n):
    """the sorted row indices --dump-outputs samples from an n-row table: every row when n <= DUMP_ROWS; drawn from a
    fixed seed and n alone, so runs with the same --rows sample the same rows"""
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_ROWS), replace=False))


def dump_outputs(out_dir, z, y, mn, rg):
    """what a caller of the timed path receives, as float32 / float64 .npy files: features.npy (2 x 24: column min and
    range), latent.npy and reconstruction.npy at the rows of dump_rows (float32), rows.npy (those indices, float64)"""
    import torch
    rows = dump_rows(z.shape[0])
    idx = torch.from_numpy(rows).to(z.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("features", torch.stack([mn, rg])), ("latent", z.index_select(0, idx)),
                    ("reconstruction", y.index_select(0, idx))):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s in sm if s > 0.5 * max(sm)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------- reference arm
def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host thread it can"""
    import torch
    torch.set_num_threads(max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)))


def reference_measurements(args, detail):
    """The reference's own CPU implementation of the path on the host cores (BASELINE.md section 3, C1 - C5), from the
    staged unmodified package (oracle/_ref, kind "reference") when it is there, else from the restatement on torch CPU
    (oracle/torch_port.py, kind "port").  CUDA must already be hidden from this process."""
    import torch
    use_all_host_threads()
    from oracle import ref_runner, torch_port
    from oracle import baler_oracle as orc
    from baler_b200 import synth
    sd = golden_state_dict()
    rows = args.ref_rows
    table = synth.cms_table(rows)
    cores = int(torch.get_num_threads())
    out = {"cores": cores, "host_cpus": os.cpu_count(), "rows": rows}
    sd_t = torch_port.to_torch(sd)

    def port_pass(t):
        z, feats = torch_port.compress(sd_t, t)
        return torch_port.decompress(sd_t, z, feats)

    port_pass(table[:50000])
    t0 = time.perf_counter()
    port_pass(table)
    out["port_best_case_rows_per_s"] = rows / (time.perf_counter() - t0)
    if not ref_runner.available():
        out["kind"] = "port"
        out["step"] = lambda: port_pass(table)
        return out
    out["kind"] = "reference"

    def shipped():
        tc, td, dec = ref_runner.compress_decompress_as_shipped(table, synth.CMS_NAMES, sd)
        return tc, td, dec

    out["step"] = shipped
    if detail:
        sec, _ = ref_runner.bare_encode_decode(table, sd, "float64")
        out["bare_model_f64_rows_per_s"] = rows / sec
        sec, _ = ref_runner.bare_encode_decode(table, sd, "float32")
        out["bare_model_f32_rows_per_s"] = rows / sec
        x = orc.normalize(synth.cms_table(512 * 200, seed=7))
        for name in ("AE", "AE_Dropout_BN"):
            ref_runner.fit_pass(name, x[:512 * 10])
            sec, _ = ref_runner.fit_pass(name, x)
            out["fit_%s_samples_per_s" % name] = len(x) / sec
        snaps = synth.cfd_snapshots(60)
        snaps = (snaps - snaps.min()) / (snaps.max() - snaps.min())
        blocks = np.ascontiguousarray(snaps.reshape(-1, 1, 5, 5), dtype=np.float32)
        te, td, nb = ref_runner.conv_encode_decode(blocks)
        out["conv_ae_encode_blocks_per_s"] = nb / te
        out["conv_ae_decode_blocks_per_s"] = nb / td
    return out


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation, all host threads, a bounded sample per step"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if os.environ.get("CUDA_VISIBLE_DEVICES", None) != "":
        # the reference runs on cuda:0 whenever it sees one (helper.py:425-439): re-exec with the GPUs hidden
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS"):
            env.pop(k, None)
        sys.exit(subprocess.call([sys.executable, os.path.abspath(__file__)] + sys.argv[1:], env=env))
    m = reference_measurements(args, args.cpu_detail)
    step = m.pop("step")
    rows = m["rows"]
    for _ in range(args.warmup):
        step()
    parts = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        parts.append(step())
    dt = time.perf_counter() - t0
    value = rows * args.steps / dt
    what = ("helper.compress + helper.decompress + helper.renormalize of the unmodified reference (oracle/_ref, baler 1.4.0) as "
            "shipped: float64, DataLoader batches of 512, np.concatenate per batch") if m["kind"] == "reference" else \
        "reference path restated on torch CPU float64 (oracle/torch_port.py), best case"
    base = dict(m, value=value, unit="rows/s", sample="%d rows of the synthetic CMS table per step; %s" % (rows, what))
    if m["kind"] == "reference" and parts and parts[0] is not None:
        base["compress_rows_per_s"] = rows * len(parts) / sum(p[0] for p in parts)
        base["decompress_rows_per_s"] = rows * len(parts) / sum(p[1] for p in parts)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "CMS AE 24->15 compress+decompress, %d-row bounded sample per step on host CPU cores" % rows},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_baseline_subprocess(args):
    """the cpu_baseline leg of our arm: the reference arm in a child process with the GPUs hidden, C1 - C5 detail"""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--ref-rows", str(args.cpu_rows), "--cpu-detail"]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS"):
        env.pop(k, None)
    r = subprocess.run(cmd, env=env, capture_output=True, text=True)
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)["cpu_baseline"]
    return {"value": None, "unit": "rows/s", "cores": None, "kind": "unavailable", "sample": (r.stderr or r.stdout)[-300:]}


def bind_to_gpu_numa_node(local):
    """one process per GPU: run on (and first-touch pinned host buffers from) the CPUs next to that GPU's PCIe root, so that
    eight ranks' host <-> device streams do not all cross the socket interconnect.  Best effort: silently skipped when the
    topology files are not there."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bdf) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


# --------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from baler_b200 import engine, sharded, synth
    from baler_b200.modules import models

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        bind_to_gpu_numa_node(local)
    if world > 1:
        # stdout carries exactly one JSON line: whatever NCCL logs (NCCL_DEBUG is the launcher's choice) goes to stderr
        if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
            os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    sd = golden_state_dict()
    model = models.AE(24, 15)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    codec = model.eval().codec()
    precision = args.precision
    n = args.rows  # rows PER GPU (weak scaling)
    x = synth.cms_table_device(n, seed=synth.CMS_SEED + rank, device=dev)
    z = torch.empty((n, 15), dtype=torch.float32, device=dev)
    y = torch.empty((n, 24), dtype=torch.float32, device=dev)
    ev_steps = []  # per timed step: (encode start, encode end, decode start, decode end) on the launching stream
    launches = {"n": 0}

    def step(timed_kernels=None):
        # compress: features of THIS table (helper.py:500-502), sharded -> one 2x24 float exchange
        mn, mx = engine.colminmax(x)
        if world > 1:
            sharded.combine_minmax_(mn, mx)
        rg = mx - mn  # torch elementwise on 24 floats: plumbing, not the hot path
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timed_kernels else None
        if ev:
            ev[0].record()
        codec.encode(x, mn, rg, precision=precision, out=z, check_range=False)
        if ev:
            ev[1].record(); ev[2].record()
        codec.decode(z, mn, rg, precision=precision, out=y, check_range=False)
        if ev:
            ev[3].record()
            ev_steps.append(ev)
        launches["n"] += 3
        return mn, rg

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the sampler runs from before the warm-up steps (nvidia-smi takes a moment to produce its first line) to the end
    # of the timed region; idle samples are dropped in stop()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()
    launches["n"] = 0
    enc_ms, dec_ms = [], []
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    t_start.record()
    for _ in range(args.steps):
        features = step(timed_kernels=True)
    t_end.record()
    sync_all()
    total_ms = t_start.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, z, y, *features)  # before the sweep below reuses z and y
    if codec.auto_precision == "split16" and codec.range_flag():
        raise RuntimeError("fp16 range guard tripped on the synthetic table: timed steps are invalid")
    clocks = sampler.stop() if rank == 0 else None
    # per-kernel durations: mean over the timed steps (events on the launching stream)
    enc_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev_steps]))
    dec_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in ev_steps]))
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = t.item()
    ms_per_step = total_ms / args.steps
    value = n * world / (ms_per_step * 1e-3)
    gpu_launches = launches["n"]

    # ---- BASELINE configs[4]: one 1B-row x 24-col table row-sharded over the N GPUs (strong scaling).  It does not fit one
    # GPU next to its latent and reconstruction (252 GB), so every rank walks its contiguous share in chunks regenerated from
    # their seeds, in the two passes the file-level path takes: column min / max of the WHOLE table (chunk results combined,
    # then one 2 x 24 exchange), then encode + decode of every chunk with the global features.  Timed: the kernels
    # (CUDA events around min/max, encode, decode; generating the synthetic chunks is not part of the path).
    sweep = None
    if not args.no_sweep:
        total_rows = 1_000_000_000
        lo, hi = sharded.row_range(total_rows, rank, world)
        rows_r = hi - lo
        chunks = [(c0, min(n, rows_r - c0)) for c0 in range(0, rows_r, n)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_ms = 0.0
        mn_g = torch.full((24,), float("inf"), device=dev)
        mx_g = -mn_g
        del x
        for ci, (c0, rows) in enumerate(chunks):
            xc = synth.cms_table_device(rows, seed=synth.CMS_SEED + 5000 + rank * 64 + ci, device=dev)
            e0.record(); mn, mx = engine.colminmax(xc); e1.record()
            torch.cuda.synchronize()
            t_ms += e0.elapsed_time(e1)
            mn_g, mx_g = torch.minimum(mn_g, mn), torch.maximum(mx_g, mx)
            del xc
        if world > 1:
            sharded.combine_minmax_(mn_g, mx_g)
        rg_g = mx_g - mn_g
        worst = 0.0
        for ci, (c0, rows) in enumerate(chunks):
            xc = synth.cms_table_device(rows, seed=synth.CMS_SEED + 5000 + rank * 64 + ci, device=dev)
            e0.record()
            codec.encode(xc, mn_g, rg_g, precision=precision, out=z[:rows], check_range=False)
            codec.decode(z[:rows], mn_g, rg_g, precision=precision, out=y[:rows], check_range=False)
            e1.record()
            torch.cuda.synchronize()
            t_ms += e0.elapsed_time(e1)
            # size-independent sanity of every chunk: the reconstruction stays inside the table's range envelope
            worst = max(worst, ((y[:rows:1009] - xc[::1009]).abs() / rg_g).max().item())
            del xc
        tt = torch.tensor([t_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        sweep = {"rows": total_rows, "rows_per_rank": rows_r, "chunks_per_rank": len(chunks), "kernel_seconds": tt.item() * 1e-3,
                 "rows_per_s": total_rows / (tt.item() * 1e-3), "scaling": "strong",
                 "max_sampled_recon_error_over_range": worst,
                 "note": "min/max of the whole table (pass 1), then encode + decode of every chunk with the global features (pass 2); "
                         "kernel time, max over ranks; chunks regenerated from their seeds in HBM"}
        x = synth.cms_table_device(n, seed=synth.CMS_SEED + rank, device=dev)  # the table of the lines below

    # ---- the CPU legs first (a child process with the GPUs hidden): the training / CFD lines quote them
    cpu = cpu_baseline_subprocess(args) if (world == 1 and not args.no_cpu) else None

    # ---- other arithmetic / latent modes of the same kernel (BASELINE.md section 4: the exact mode meets 1e-5 and is
    # tensor-bound; the single-product `fast` mode and the float16 latent move towards the HBM roof, outside the tolerance)
    modes = None
    if world == 1 and not args.no_modes:
        modes = {}
        ns = min(n, 2_000_000)
        mn, mx = engine.colminmax(x)
        rg = mx - mn
        # the exact mode's own output on the first ns rows (z / y were reused by the 1B-row sweep above)
        z_ref = torch.empty((ns, 15), dtype=torch.float32, device=dev)
        y_ref = torch.empty((ns, 24), dtype=torch.float32, device=dev)
        codec.encode(x[:ns], mn, rg, precision=precision, out=z_ref, check_range=False)
        codec.decode(z_ref, mn, rg, precision=precision, out=y_ref, check_range=False)
        for name, prec, zdt in (("exact_f16_latent", precision, torch.float16), ("fast", "fast", torch.float32),
                                ("fast_f16_latent", "fast", torch.float16)):
            zz = torch.empty((n, 15), dtype=zdt, device=dev)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            try:
                for it in range(3):
                    if it == 2:
                        ev[0].record()
                    codec.encode(x, mn, rg, precision=prec, out=zz, check_range=False)
                    if it == 2:
                        ev[1].record()
                    codec.decode(zz, mn, rg, precision=prec, out=y, check_range=False)
                    if it == 2:
                        ev[2].record()
                torch.cuda.synchronize()
            except Exception as e:  # a mode the loaded library does not take is reported, not fatal
                modes[name] = {"error": str(e)}
                continue
            em, dm = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
            bytes_row = 96 + (30 if zdt == torch.float16 else 60)
            zerr = ((zz[:ns].float() - z_ref).abs().max() / z_ref.abs().max()).item()
            yerr = ((y[:ns] - y_ref).abs().max() / y_ref.abs().max()).item()
            tf = n * FLOP_PER_ROW / (em * 1e-3) / 1e12
            modes[name] = {"compress_rows_per_s": n / (em * 1e-3), "decompress_rows_per_s": n / (dm * 1e-3),
                           "encode_tflops": tf, "frac_of_bf16_sustained": tf / peaks["tflops"], "frac_of_bf16_burst": tf / peaks["tflops_burst"],
                           "hbm_gbs": n * bytes_row / (em * 1e-3) / 1e9, "hbm_frac": n * bytes_row / (em * 1e-3) / 1e9 / peaks["hbm_gbs"],
                           "bytes_per_row": bytes_row, "latent_err_vs_exact": zerr, "recon_err_vs_exact": yerr,
                           "within_1e-5": bool(zerr <= 1e-5 and yerr <= 1e-5)}
            del zz
        codec.range_flag()  # the fast mode may have tripped it: clear
        codec.decode(z, mn, rg, precision=precision, out=y, check_range=False)  # leave y as the exact reconstruction
        del z_ref, y_ref

    # ---- e2e: host buffers through the C-ABI pipelines
    e2e = None
    if not args.no_e2e:
        ne = min(n, max(args.e2e_rows // world, 1_000_000))  # total pinned host memory stays ~25 GB whatever N
        xh = torch.empty((ne, 24), dtype=torch.float32, pin_memory=True)
        zh = torch.empty((ne, 15), dtype=torch.float32, pin_memory=True)
        yh = torch.empty((ne, 24), dtype=torch.float32, pin_memory=True)
        xh.copy_(x[:ne])
        torch.cuda.synchronize()
        xn, zn, yn = xh.numpy(), zh.numpy(), yh.numpy()

        def e2e_step():
            if world > 1:
                # sharded: local min/max -> exchange -> compress with the global features
                mn, mx = engine.colminmax(x[:ne])
                sharded.combine_minmax_(mn, mx)
                feats = torch.stack([mn, mx - mn]).cpu().numpy()
                codec.compress_host(xn, features=feats, z_dtype=np.float32, precision=precision, out=zn)
            else:
                _, feats = codec.compress_host(xn, recompute_minmax=True, z_dtype=np.float32, precision=precision, out=zn)
            codec.decompress_host(zn, features=feats, y_dtype=np.float32, precision=precision, out=yn)

        for _ in range(min(args.warmup, 2)):
            e2e_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        sync_all()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": ne * world * args.e2e_steps / dt.item(), "unit": "rows/s",
               "h2d_bytes_per_step": int(ne * (96 + 60)), "d2h_bytes_per_step": int(ne * (60 + 96)),
               "rows_per_gpu": ne, "steps": args.e2e_steps,
               "note": "bb_compress_host + bb_decompress_host, pinned host buffers, fp32 latent; timed on the host clock "
                       "around blocking calls (the copies are part of the call)"}
        # the same pass with the reference's on-disk dtypes (helper.py:565: float64 latent in compressed.npz, float64
        # reconstruction): the library widens / narrows on host threads around float32 PCIe copies; smaller sample
        if world == 1:
            nf = min(ne, 20_000_000)
            z64 = np.empty((nf, 15), dtype=np.float64)
            y64 = np.empty((nf, 24), dtype=np.float64)

            def f64_step():
                _, feats = codec.compress_host(xn[:nf], recompute_minmax=True, z_dtype=np.float64, precision=precision, out=z64)
                codec.decompress_host(z64, features=feats, y_dtype=np.float64, precision=precision, out=y64)

            f64_step()
            t0 = time.perf_counter()
            f64_step()
            e2e["reference_file_dtypes"] = {"value": nf / (time.perf_counter() - t0), "unit": "rows/s", "rows": nf,
                                            "note": "float64 latent and float64 reconstruction in pageable host arrays"}
            del z64, y64
        del xh, zh, yh

    # ---- training lines: one epoch over a 600k-row normalised table, batch 512 per GPU (weak scaling: global batch
    # 512 x N, the reference's batch_size = global batch).  AE on the tensor-core step (and on the fp32 step for
    # comparison at N = 1), AE_Dropout_BN (BASELINE configs[2]) on the fp32 cooperative kernel.
    train = train_dbn = None
    if not args.no_train:
        tn = 600_000  # rows per GPU and epoch
        if world == 1:
            xsrc = x[:tn].contiguous()
        else:
            # data parallel = the reference's run at batch_size = 512 x N on ONE table: every rank holds the same
            # (tn x N)-row table and processes its 512-row share of every global batch
            xsrc = synth.cms_table_device(tn * world, seed=synth.CMS_SEED + 77, device=dev)
        mn, mx = engine.colminmax(xsrc)
        xt = engine.normalize_table(xsrc, mn, mx - mn)
        del xsrc
        gb = 512 * world

        def one_epoch(tr, precision_name):
            hyper = engine.make_hyper(lr=1e-3, world_size=world)
            if world == 1:
                tr.epoch(xt[:51200], 512, hyper)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                loss = tr.epoch(xt, 512, hyper)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                fused = None
            else:
                dp = sharded.DataParallelTrainer(tr)
                fused = dp.fused
                dp.epoch_table(xt[:100 * gb], gb, hyper, rank, world)
                dts = []
                for _ in range(2):
                    sync_all()
                    t0 = time.perf_counter()
                    loss = dp.epoch_table(xt, gb, hyper, rank, world)
                    sync_all()
                    dts.append(time.perf_counter() - t0)
                dt = min(dts)
            steps = (xt.shape[0] + gb - 1) // gb
            tdt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
            dt = tdt.item()
            sps = xt.shape[0] / dt
            out = {"samples_per_s": sps, "us_per_step": 1e6 * dt / steps, "steps": steps, "global_batch": gb,
                   "epoch_loss": loss, "precision": precision_name, "flop_per_sample": 357000, "tflops": sps * 357000 / 1e12,
                   "roofline": {"bound": "latency (15 dependent layer passes per 512-row step); tensor peak for reference",
                                "achieved": sps * 357000 / 1e12, "peak": peaks["tflops"] * world, "unit": "TFLOP/s",
                                "frac": sps * 357000 / 1e12 / (peaks["tflops"] * world)}}
            if fused is not None:
                out["gradient_exchange"] = ("fused in the weight-gradient kernel over NVLink peer memory (bb_trainer_dp_connect)"
                                            if fused else "NCCL SUM all-reduce of the flat gradient between two kernel phases")
            return out

        torch.manual_seed(0)
        tm = models.AE(24, 15)
        w, b = tm.linear_tensors()
        tr = engine.Trainer(w, b, 24, 15, 512)
        train = one_epoch(tr, tr.precision)
        train["model"] = "AE 24-200-100-50-15-50-100-200-24"
        if world == 1:
            tr32 = engine.Trainer(w, b, 24, 15, 512)
            tr32.set_precision("fp32")
            train["fp32_step"] = {k: v for k, v in one_epoch(tr32, "fp32").items() if k in ("samples_per_s", "us_per_step", "epoch_loss")}
            del tr32
        if cpu and cpu.get("fit_AE_samples_per_s"):
            train["cpu_baseline"] = {"samples_per_s": cpu["fit_AE_samples_per_s"], "cores": cpu["cores"], "kind": cpu["kind"],
                                     "sample": "training.fit of the unmodified reference, 200 steps of bs 512 (BASELINE.md C4)"}
            train["vs_cpu"] = train["samples_per_s"] / cpu["fit_AE_samples_per_s"]
        del tr
        if world > 1:
            # data-parallel parity, visible to the driver: replicas bit-identical, and equal to ONE GPU running the same
            # 20 global batches at batch_size = 512 x N (<= 1e-5 of max|w|)
            rows_p = 20 * gb
            hyper = engine.make_hyper(lr=1e-3, world_size=world)
            trp = engine.Trainer(w, b, 24, 15, 512)
            dpp = sharded.DataParallelTrainer(trp)
            dpp.epoch_table(xt[:rows_p], gb, hyper, rank, world)
            mine = trp.params_view().clone()
            ref0 = mine.clone()
            dist.broadcast(ref0, src=0)
            same = torch.tensor([1 if torch.equal(mine, ref0) else 0], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            train["dp_parity"] = {"replicas_identical": bool(same.item()), "global_steps": 20, "fused": dpp.fused}
            if rank == 0:
                tr1 = engine.Trainer(w, b, 24, 15, gb)
                tr1.epoch(xt[:rows_p], gb, engine.make_hyper(lr=1e-3))
                one = tr1.params_view()
                train["dp_parity"]["vs_single_gpu_same_global_batch_rel_max"] = ((mine - one).abs().max() / one.abs().max()).item()
                train["dp_parity"]["ok"] = bool(same.item()) and train["dp_parity"]["vs_single_gpu_same_global_batch_rel_max"] <= 1e-5
                del tr1
            del trp, dpp
        torch.manual_seed(0)
        dm = models.AE_Dropout_BN(24, 15)
        w, b = dm.linear_tensors()
        trd = engine.Trainer(w, b, 24, 15, 512, bn=dm.bn_tensors())
        trd.set_dropout(seed=1234)  # one stream keyed by the global batch row, the same on every rank
        train_dbn = one_epoch(trd, trd.precision)
        train_dbn["model"] = "AE_Dropout_BN 24-200-100-50-15-50-100-200-24 (dropout .5/.4/.3/.2, 4 BatchNorm1d)"
        train_dbn["batchnorm"] = ("statistics of the global batch: the 8 reduction points of a step exchanged over NVLink peer "
                                  "memory inside the kernel" if world > 1 else "batch statistics")
        train_dbn["loss"] = "sum-MSE / n_columns as training.fit evaluates it (validate=True: the L1 term never trains, SURVEY F2)"
        if world == 1:
            trd32 = engine.Trainer(w, b, 24, 15, 512, bn=dm.bn_tensors())
            trd32.set_precision("fp32")
            trd32.set_dropout(seed=1234)
            train_dbn["fp32_step"] = {k: v for k, v in one_epoch(trd32, "fp32").items() if k in ("samples_per_s", "us_per_step", "epoch_loss")}
            del trd32
        if cpu and cpu.get("fit_AE_Dropout_BN_samples_per_s"):
            train_dbn["cpu_baseline"] = {"samples_per_s": cpu["fit_AE_Dropout_BN_samples_per_s"], "cores": cpu["cores"],
                                         "kind": cpu["kind"],
                                         "sample": "training.fit of the unmodified reference, 200 steps of bs 512 (BASELINE.md C4)"}
            train_dbn["vs_cpu"] = train_dbn["samples_per_s"] / cpu["fit_AE_Dropout_BN_samples_per_s"]
        if world > 1:
            # BASELINE configs[2] parity, visible to the driver: replicas bit-identical (parameters and BatchNorm running
            # statistics), and equal to ONE GPU training at batch_size = 512 x N with the same dropout seed.  What a step
            # computes - the loss and the statistics of the global batch - is compared at 1e-5 after one global step.
            # Parameters go through Adam, whose first step is lr * sign(g): gradient components below the fp32 noise floor
            # may take either sign in any two correct fp32 implementations (the reference holds float64 noise there), so
            # the fraction of parameters off by more than 1e-5 of max|w| is reported instead of gated to zero, and the
            # 20-step epoch losses are compared.
            hyper = engine.make_hyper(lr=1e-3, world_size=world)
            trp = engine.Trainer(w, b, 24, 15, 512, bn=dm.bn_tensors())
            trp.set_dropout(seed=99)
            dpp = sharded.DataParallelTrainer(trp)
            loss_1 = dpp.epoch_table(xt[:gb], gb, hyper, rank, world)
            after_1 = torch.cat([trp.params_view()] + list(trp.bn_running_views())).clone()
            loss_20 = dpp.epoch_table(xt[:20 * gb], gb, hyper, rank, world)
            mine = torch.cat([trp.params_view()] + list(trp.bn_running_views())).clone()
            ref0 = mine.clone()
            dist.broadcast(ref0, src=0)
            same = torch.tensor([1 if torch.equal(mine, ref0) else 0], device=dev)
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            train_dbn["dp_parity"] = {"replicas_identical": bool(same.item()), "global_steps": 21, "fused": dpp.fused}
            if rank == 0:
                ok = False
                try:
                    tr1 = engine.Trainer(w, b, 24, 15, gb, bn=dm.bn_tensors())
                    if tr1.precision == "split16":  # (one GPU holds at most 148 x 16 rows of a BatchNorm batch)
                        tr1.set_dropout(seed=99)
                        one_loss_1 = tr1.epoch(xt[:gb], gb, engine.make_hyper(lr=1e-3))
                        one_1 = torch.cat([tr1.params_view()] + list(tr1.bn_running_views())).clone()
                        one_loss_20 = tr1.epoch(xt[:20 * gb], gb, engine.make_hyper(lr=1e-3))
                        npar = tr1.n_params
                        pmax = one_1[:npar].abs().max()
                        dpar = (after_1[:npar] - one_1[:npar]).abs()
                        pr = train_dbn["dp_parity"]
                        pr["first_step_loss_rel"] = abs(loss_1 - one_loss_1) / one_loss_1
                        pr["first_step_batch_statistics_rel_max"] = \
                            ((after_1[npar:] - one_1[npar:]).abs().max() / one_1[npar:].abs().max()).item()
                        pr["first_step_params_off_fraction"] = (dpar > 1e-5 * pmax).float().mean().item()
                        pr["first_step_params_max_abs_diff"] = dpar.max().item()
                        pr["epoch_loss_20_steps_rel"] = abs(loss_20 - one_loss_20) / one_loss_20
                        ok = (bool(same.item()) and pr["first_step_loss_rel"] <= 1e-5
                              and pr["first_step_batch_statistics_rel_max"] <= 1e-5 and pr["first_step_params_off_fraction"] <= 0.01
                              and pr["first_step_params_max_abs_diff"] <= 2.002e-3 and pr["epoch_loss_20_steps_rel"] <= 1e-2)
                    else:
                        train_dbn["dp_parity"]["note"] = ("global batch of %d rows exceeds one GPU's tensor-core BatchNorm step "
                                                          "(148 x 16 rows): no single-GPU run to compare with" % gb)
                        ok = bool(same.item())
                    del tr1
                except Exception as e:  # noqa: BLE001
                    train_dbn["dp_parity"]["note"] = "single-GPU comparison unavailable: %s" % e
                train_dbn["dp_parity"]["ok"] = ok
            del trp, dpp
        del trd

    # ---- CFD line (secondary, BASELINE configs[3]): Conv_AE on 5x5 blocks of synthetic 50x50 flow-field snapshots,
    # z = 250 (compression_ratio 10, baler.py:130-135), eval mode; the dense-equivalent chain on the fp32 GEMM path
    cfd = None
    if not args.no_cfd and rank == 0:
        nb = args.cfd_blocks
        torch.manual_seed(0)
        cm = models.Conv_AE(5, 250).eval()
        snaps = synth.cfd_snapshots((nb + 99) // 100)  # 50x50 snapshots -> 100 blocks of 5x5 each (convert_to_blocks=[1,5,5])
        snaps = (snaps - snaps.min()) / (snaps.max() - snaps.min())
        blocks = torch.from_numpy(np.ascontiguousarray(snaps.reshape(-1, 1, 5, 5)[:nb])).cuda()
        flop = 1593216  # per block and direction (SURVEY 8a)

        def cfd_pass(prec):
            zc = cm.encode(blocks, precision=prec); yc = cm.decode(zc, precision=prec)  # warm-up (packs the dense-equivalent matrices)
            del zc, yc  # (the timed pass reuses these blocks of the caching allocator instead of a fresh 600 MB cudaMalloc)
            torch.cuda.synchronize()
            c0, c1, c2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            c0.record(); zc = cm.encode(blocks, precision=prec); c1.record(); yc = cm.decode(zc, precision=prec); c2.record()
            torch.cuda.synchronize()
            return zc, yc, c0.elapsed_time(c1) * 1e-3, c1.elapsed_time(c2) * 1e-3

        zc, yc, te, td = cfd_pass("auto")
        z32, y32, te32, td32 = cfd_pass("fp32")
        cfd_prec = cm.codec(5, 5).auto_precision
        cfd = {"model": "Conv_AE 5x5 -> 250", "blocks": nb, "precision": cfd_prec,
               "encode_blocks_per_s": nb / te, "decode_blocks_per_s": nb / td,
               "encode_tflops": nb * flop / te / 1e12, "decode_tflops": nb * flop / td / 1e12,
               "latent_err_vs_fp32": ((zc - z32).abs().max() / z32.abs().max()).item(),
               "recon_err_vs_fp32": ((yc - y32).abs().max() / y32.abs().max()).item(),
               "roofline": {"bound": "tensor", "achieved": nb * flop / te / 1e12, "peak": peaks["tflops"], "unit": "TFLOP/s",
                            "frac": nb * flop / te / 1e12 / peaks["tflops"],
                            "kernel": "gemm_tc5_kernel (one tcgen05 split16 GEMM launch per layer; useful single-count FLOPs)"},
               "fp32_path": {"encode_blocks_per_s": nb / te32, "decode_blocks_per_s": nb / td32,
                             "encode_tflops": nb * flop / te32 / 1e12,
                             "note": "layered fp32 GEMM path (CUDA cores); nominal FFMA peak 74.5 TFLOP/s"}}
        del z32, y32
        # one training pass over 60k blocks, batch 600 (train-mode BatchNorm2d, sum-MSE, Adam): the layer-by-layer trainer
        # with the convolutions as weight-sharing dense layers
        sp = cm.training_spec(5, 5)
        ctr = engine.LayeredTrainer(sp["weights"], sp["biases"], sp["acts"], 600, dims=sp["dims"], w_maps=sp["w_maps"],
                                    bn=sp["bn"], loss_columns=1)
        tb = blocks[:60_000].reshape(-1, 25).contiguous()
        ctr.epoch(tb[:6000], 600, engine.make_hyper(lr=1e-3))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        closs = ctr.epoch(tb, 600, engine.make_hyper(lr=1e-3))
        torch.cuda.synchronize()
        cdt = time.perf_counter() - t0
        cfd.update(train_blocks_per_s=len(tb) / cdt, train_us_per_step=1e6 * cdt / (len(tb) // 600), train_batch=600,
                   train_epoch_loss=closs)
        del blocks, zc, yc, tb, ctr

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    enc_tflops = n * FLOP_PER_ROW / (enc_ms * 1e-3) / 1e12
    dec_tflops = n * FLOP_PER_ROW / (dec_ms * 1e-3) / 1e12
    traffic = traffic_src = None
    prof = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(prof):
        per_row = json.load(open(prof)).get("encode_dram_bytes_per_row")
        traffic = per_row * n if per_row else None
        traffic_src = "profiles/ncu_traffic.json (dram bytes per row of one ncu --set full capture) x rows of this launch; not measured in this run"
    if cfd is not None and cpu and cpu.get("conv_ae_encode_blocks_per_s"):
        cfd["cpu_baseline"] = {"encode_blocks_per_s": cpu["conv_ae_encode_blocks_per_s"], "decode_blocks_per_s": cpu["conv_ae_decode_blocks_per_s"],
                               "cores": cpu["cores"], "kind": cpu["kind"],
                               "sample": "Conv_AE(5, 250) of the unmodified reference, eval mode, 6000 blocks, batch 600 (BASELINE.md C5)"}
        cfd["encode_vs_cpu"] = cfd["encode_blocks_per_s"] / cpu["conv_ae_encode_blocks_per_s"]
    out = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "CMS AE 24->15 compress+decompress of a %d-row x 24-col float32 table per GPU" % n,
                   "rows_per_gpu": n, "precision": codec.auto_precision if precision == "auto" else precision,
                   "l2": "inputs larger than L2 (%.1f GB table per GPU)" % (n * 96 / 1e9),
                   "weights": "reference AE(24,15) trained 2 epochs (tests/golden/ae_cms.npz)"},
        "gpu_launches": gpu_launches, "clocks": clocks,
        "compress_rows_per_s": n / (enc_ms * 1e-3), "decompress_rows_per_s": n / (dec_ms * 1e-3),
        # useful (un-padded, single-count) FLOPs of the launch over the measured dense bf16 peak.  `frac` uses the
        # SUSTAINED figure (the kernel is timed inside a long step under the power cap); SURVEY 8(d)'s formula uses the
        # burst figure: `frac_burst`.
        "roofline": {"bound": "tensor", "achieved": enc_tflops, "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": enc_tflops / peaks["tflops"], "peak_burst": peaks["tflops_burst"],
                     "frac_burst": enc_tflops / peaks["tflops_burst"], "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": "chain_tc4_kernel (fused encode chain)",
                     "peak_source": peaks["src"] + " (bf16 dense; frac: sustained, frac_burst: burst)", "launch_ms": enc_ms,
                     "algorithmic_flop_per_row": FLOP_PER_ROW,
                     "hbm": {"achieved_gbs": n * BYTES_PER_ROW / (enc_ms * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"],
                             "frac": n * BYTES_PER_ROW / (enc_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                             "algorithmic_bytes_per_row": BYTES_PER_ROW}},
        "roofline_decode": {"bound": "tensor", "achieved": dec_tflops, "peak": peaks["tflops"], "unit": "TFLOP/s",
                            "frac": dec_tflops / peaks["tflops"], "frac_burst": dec_tflops / peaks["tflops_burst"],
                            "kernel": "chain_tc4_kernel (fused decode chain)", "launch_ms": dec_ms,
                            "hbm": {"achieved_gbs": n * BYTES_PER_ROW / (dec_ms * 1e-3) / 1e9,
                                    "frac": n * BYTES_PER_ROW / (dec_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}},
        "modes": modes,
        "sweep_1b": sweep,
        "e2e": e2e, "train": train, "train_dbn": train_dbn, "cfd": cfd,
    }
    if cpu is not None:
        out["cpu_baseline"] = cpu
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="rows per GPU")
    ap.add_argument("--precision", default="auto")
    ap.add_argument("--e2e-rows", type=int, default=100_000_000)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-rows", type=int, default=200_000)
    ap.add_argument("--ref-rows", type=int, default=200_000, help="rows per step of the reference arm (its loop is O(N^2))")
    ap.add_argument("--cpu-detail", action="store_true", help="reference arm: also time C3 - C5 of BASELINE.md")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-cfd", action="store_true")
    ap.add_argument("--no-modes", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the 1B-row strong-scaling sweep (BASELINE configs[4])")
    ap.add_argument("--cfd-blocks", type=int, default=600_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl ours: write the last timed step's outputs as DIR/<name>.npy (rank 0's shard under torchrun)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
