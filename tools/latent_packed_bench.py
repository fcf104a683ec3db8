"""The b-bit latent (latent_dtype "q2" ... "q8") on the device, one JSON document (printed, and written to --out):

  card         name, power limit and max SM clock, read in this call (before and after)
  kernels      latent_quantize_kernel<b> / latent_dequantize_kernel<b> on a resident [rows, 15] float32 latent (6 GB at
               100M rows, larger than L2) for b = 8, 6, 4, 3, 2: ms per call (CUDA events around --reps calls), bytes the
               format needs per call (quantise: 4z read, ceil(z b / 8) + 8z / 128 written per row; dequantise the
               reverse) and those bytes over the time, against 7.7 TB/s
  q8_vs_parent with --parent ROOT (a built checkout of the parent commit): the 8-bit kernels of this tree and of the
               parent's library on the same resident latent, alternated over --rounds rounds (median, min, max), and
               whether their codes, parameters and dequantised values are bit-equal
  host         bb_compress_host_packed / bb_decompress_host_packed rows/s for the same b and bb_compress_host /
               bb_decompress_host with float16 and float64 latents, pageable host tables, alternated over --rounds
               rounds: median, min, max
  files        at --file-rows rows: compressed.npz bytes per row (np.savez) for each latent; reconstruction RMS / range
               per column against the table and against the float32-latent reconstruction (mean and worst column), the
               largest absolute shift; whether the device codes are bit-equal to the numpy mirror (tests/
               latent_packed_ref.py); with --parent, whether the q8 compressed.npz equals the parent's byte for byte

The model is the CMS AE of tests/golden/ae_cms.npz (the reference's AE 24 -> 15 after its training run on the synthetic
CMS table); the tables are synth.cms_table.

    python tools/latent_packed_bench.py [--rows 100000000] [--file-rows 600000] [--rounds 3] [--parent ROOT] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if __name__ == "__main__" and "--write-q8" in sys.argv:  # the parent's package writes its own file (see q8_file)
    ROOT = os.path.abspath(sys.argv[sys.argv.index("--root") + 1])
sys.path.insert(0, ROOT)
sys.path.insert(1, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from baler_b200 import _lib, engine, latent_q8, synth  # noqa: E402
from baler_b200.modules import models  # noqa: E402

HBM_BYTES_S = 7.7e12
BITS = (8, 6, 4, 3, 2)


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


def spread(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": [float(x) for x in v]}


def host_table(rows):
    out = np.empty((rows, 24), dtype=np.float32)
    step = 20_000_000
    for r0 in range(0, rows, step):
        out[r0:r0 + step] = synth.cms_table_device(min(step, rows - r0), seed=1 + r0 // step).cpu().numpy()
    return out


class Q8Lib:
    """bb_latent_quantize_q8 / bb_latent_dequantize_q8 of one libbaler_b200.so, on its own context"""

    def __init__(self, path):
        self.lib = C.CDLL(path)
        self.lib.bb_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        self.lib.bb_latent_quantize_q8.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int] + [C.c_void_p] * 4
        self.lib.bb_latent_dequantize_q8.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_int, C.c_void_p, C.c_void_p]
        self.ctx = C.c_void_p()
        assert self.lib.bb_ctx_create(torch.cuda.current_device(), C.byref(self.ctx)) == 0

    def quantize(self, z, q):
        assert self.lib.bb_latent_quantize_q8(self.ctx, z.data_ptr(), z.shape[0], z.shape[1], q[0].data_ptr(),
                                              q[1].data_ptr(), q[2].data_ptr(), None) == 0

    def dequantize(self, q, z):
        assert self.lib.bb_latent_dequantize_q8(self.ctx, q[0].data_ptr(), q[1].data_ptr(), q[2].data_ptr(), z.shape[0],
                                                z.shape[1], z.data_ptr(), None) == 0


def _buffers(rows, z_dim, bits):
    nb = latent_q8.n_blocks(rows)
    return (torch.empty((rows, latent_q8.row_bytes(z_dim, bits)), dtype=torch.uint8, device="cuda"),
            torch.empty((nb, z_dim), device="cuda"), torch.empty((nb, z_dim), device="cuda"))


def kernels(codec, z, reps):
    rows, z_dim = z.shape
    lib, ctx = _lib.lib(), codec.ctx.handle
    back = torch.empty_like(z)
    out = {"rows": rows, "z_dim": z_dim}
    for bits in BITS:
        q = _buffers(rows, z_dim, bits)

        def quant():
            assert lib.bb_latent_quantize_packed(ctx, z.data_ptr(), rows, z_dim, bits, *(t.data_ptr() for t in q), None) == 0

        def dequant():
            assert lib.bb_latent_dequantize_packed(ctx, bits, *(t.data_ptr() for t in q), rows, z_dim, back.data_ptr(),
                                                   None) == 0
        quant()
        dequant()
        tq, td = timed(quant, reps), timed(dequant, reps)
        byt = 4 * rows * z_dim + rows * latent_q8.row_bytes(z_dim, bits) + 2 * 4 * z_dim * latent_q8.n_blocks(rows)
        out["q%d" % bits] = {name: {"ms": ms, "bytes": byt, "bytes_per_s": byt / (ms * 1e-3),
                                    "of_hbm": byt / (ms * 1e-3) / HBM_BYTES_S}
                             for name, ms in (("quantize", tq), ("dequantize", td))}
        del q
    torch.cuda.empty_cache()
    return out


def q8_vs_parent(z, parent_lib, rounds, reps):
    rows, z_dim = z.shape
    libs = {"this": Q8Lib(_lib.LIB_PATH), "parent": Q8Lib(parent_lib)}
    bufs = {k: _buffers(rows, z_dim, 8) for k in libs}
    backs = {k: torch.empty_like(z) for k in libs}
    for k, L in libs.items():  # warm-up, and the results compared
        L.quantize(z, bufs[k])
        L.dequantize(bufs[k], backs[k])
    torch.cuda.synchronize()
    same = all(torch.equal(a.view(torch.uint8), b.view(torch.uint8)) for a, b in zip(bufs["this"], bufs["parent"]))
    same = same and torch.equal(backs["this"].view(torch.int32), backs["parent"].view(torch.int32))
    t = {"%s_%s" % (k, op): [] for k in libs for op in ("quantize", "dequantize")}
    for r in range(rounds):
        for k in (("this", "parent") if r % 2 == 0 else ("parent", "this")):
            L = libs[k]
            t[k + "_quantize"].append(timed(lambda: L.quantize(z, bufs[k]), reps))
            t[k + "_dequantize"].append(timed(lambda: L.dequantize(bufs[k], backs[k]), reps))
    del bufs, backs
    torch.cuda.empty_cache()
    res = {"rows": rows, "bit_equal": bool(same), "ms": {k: spread(v) for k, v in t.items()}}
    for op in ("quantize", "dequantize"):
        res[op + "_this_over_parent"] = float(np.median(t["this_" + op]) / np.median(t["parent_" + op]))
    return res


def host(codec, rows, rounds):
    x = host_table(rows)
    feats = np.zeros((2, 24), np.float32)
    codec.compress_host(x[:1 << 20], features=feats, recompute_minmax=True)  # warm-up
    _, feats = codec.compress_host(x, features=feats, recompute_minmax=True)
    z16 = np.empty((rows, codec.z_dim), np.float16)
    z64 = np.empty((rows, codec.z_dim), np.float64)
    qs = {b: latent_q8.empty_packed(rows, codec.z_dim, b) for b in BITS}
    y = np.empty((rows, 24), np.float64)
    ops = {"compress_float16": lambda: codec.compress_host(x, features=feats, out=z16),
           "compress_float64": lambda: codec.compress_host(x, features=feats, out=z64),
           "decompress_float16": lambda: codec.decompress_host(z16, features=feats, out=y),
           "decompress_float64": lambda: codec.decompress_host(z64, features=feats, out=y)}
    for b in BITS:
        ops["compress_q%d" % b] = lambda b=b: codec.compress_host_packed(x, b, features=feats, out=qs[b])
        ops["decompress_q%d" % b] = lambda b=b: codec.decompress_host_packed(qs[b], features=feats, out=y)
    for fn in ops.values():  # warm-up: staging, pinned buffers, page faults of the outputs
        fn()
    res = {k: [] for k in ops}
    for _ in range(rounds):
        for k, fn in ops.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            res[k].append(rows / (time.perf_counter() - t0))
    return {"rows": rows, "buffers": "pageable", "rows_per_s": {k: spread(v) for k, v in res.items()}}


def q8_file(codec, x, feats, path):
    """compressed.npz of the 8-bit latent, as baler.perform_compression writes it"""
    q, _ = codec.compress_host_q8(x, features=feats)
    np.savez(path, **latent_q8.npz_arrays(q), names=np.array(synth.CMS_NAMES), normalization_features=feats)


def files(codec, rows, parent):
    import latent_packed_ref as ref
    x = synth.cms_table(rows, seed=17)
    mn, mx = x.min(axis=0), x.max(axis=0)
    feats = np.stack([mn, mx - mn]).astype(np.float32)
    names = np.array(synth.CMS_NAMES)
    z32, _ = codec.compress_host(x, features=feats)
    lat = {"float32": z32, "float64": codec.compress_host(x, features=feats, z_dtype=np.float64)[0],
           "float16": codec.compress_host(x, features=feats, z_dtype=np.float16)[0]}
    mirror_equal = {}
    for b in BITS:
        q = codec.compress_host_packed(x, b, features=feats)[0]
        codes, lo, step = ref.quantize(z32, b)
        mirror_equal["q%d" % b] = bool(np.array_equal(q.codes, ref.pack(codes, b)) and np.array_equal(q.lo, lo)
                                       and np.array_equal(q.step, step))
        lat["q%d" % b] = q
    sizes, err = {}, {}
    rng = (mx - mn).astype(np.float64)
    rng = np.where(rng > 0, rng, 1)
    y32 = codec.decompress_host(z32, features=feats)
    with tempfile.TemporaryDirectory() as d:
        np.savez(os.path.join(d, "input.npz"), data=x, names=names)
        sizes["input"] = os.path.getsize(os.path.join(d, "input.npz"))
        for k, z in lat.items():
            arrays = latent_q8.npz_arrays(z) if isinstance(z, latent_q8.PackedLatent) else {"data": z}
            p = os.path.join(d, k + ".npz")
            np.savez(p, **arrays, names=names, normalization_features=feats)
            sizes[k] = os.path.getsize(p)
        same_as_parent = None
        if parent:
            q8_file(codec, x, feats, os.path.join(d, "this_q8.npz"))
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--root", parent, "--write-q8",
                                os.path.join(d, "parent_q8.npz"), "--file-rows", str(rows)], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr[-2000:]
            same_as_parent = open(os.path.join(d, "this_q8.npz"), "rb").read() == \
                open(os.path.join(d, "parent_q8.npz"), "rb").read()
    for k, z in lat.items():
        y = codec.decompress_host_packed(z, features=feats) if isinstance(z, latent_q8.PackedLatent) else \
            codec.decompress_host(z, features=feats)
        rms = np.sqrt(np.mean((y - x.astype(np.float64)) ** 2, axis=0)) / rng
        shift = np.sqrt(np.mean((y - y32) ** 2, axis=0)) / rng
        err[k] = {"rms_over_range_mean": float(rms.mean()), "rms_over_range_max": float(rms.max()),
                  "shift_vs_float32_rms_over_range_mean": float(shift.mean()),
                  "shift_vs_float32_rms_over_range_max": float(shift.max()),
                  "shift_vs_float32_max_abs_over_range": float((np.abs(y - y32) / rng).max())}
    return {"rows": rows, "bytes": sizes, "bytes_per_row": {k: v / rows for k, v in sizes.items()},
            "codes_bit_equal_to_mirror": mirror_equal, "q8_file_equal_to_parent": same_as_parent, "error": err}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--file-rows", type=int, default=600_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--parent", default=None, help="root of a built checkout of the parent commit")
    ap.add_argument("--root", default=None)
    ap.add_argument("--write-q8", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    engine.require_cuda()
    codec = model().codec()
    if a.write_q8:
        x = synth.cms_table(a.file_rows, seed=17)
        mn, mx = x.min(axis=0), x.max(axis=0)
        q8_file(codec, x, np.stack([mn, mx - mn]).astype(np.float32), a.write_q8)
        return
    with open("/proc/meminfo") as f:  # the host pipelines hold ~500 bytes per row (table, latents, float64 rows)
        avail = int([ln.split()[1] for ln in f if ln.startswith("MemAvailable")][0]) * 1024
    host_rows = min(a.rows, int(avail * 0.6) // 500 // (1 << 20) * (1 << 20))
    res = {"card": card(), "model": "AE 24 -> 15 (tests/golden/ae_cms.npz)"}
    res["files"] = files(codec, a.file_rows, a.parent)
    z = torch.randn((a.rows, codec.z_dim), device="cuda")
    res["kernels"] = kernels(codec, z, a.reps)
    if a.parent:
        res["q8_vs_parent"] = q8_vs_parent(z, os.path.join(a.parent, "baler_b200", "libbaler_b200.so"), 2 * a.rounds + 1,
                                           a.reps)
    del z
    torch.cuda.empty_cache()
    res["host"] = host(codec, host_rows, a.rounds)
    res["card_after"] = card()
    text = json.dumps(res)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
