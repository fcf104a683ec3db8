"""CPU-only checks of the 8-bit latent (latent_dtype "q8"): the numpy mirror keeps its error bound on awkward columns, the
compressed.npz reader refuses malformed parameter arrays, block-aligned row shards (gloo, world size 2), the precision
"fp64" refusal, and the no-CPU-fallback error."""
import os
import socket
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import latent_q8_ref as ref
from baler_b200 import _lib, build, latent_q8, sharded
from baler_b200.modules import helper

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SYMBOLS = ("bb_latent_quantize_q8", "bb_latent_dequantize_q8", "bb_compress_host_q8", "bb_decompress_host_q8")


def _check_bound(z):
    codes, lo, step = ref.quantize(z)
    assert codes.dtype == np.uint8 and lo.dtype == step.dtype == np.float32
    assert codes.shape == z.shape and lo.shape == step.shape == (latent_q8.n_blocks(len(z)), z.shape[1])
    back = ref.dequantize(codes, lo, step)
    fin = np.isfinite(z)
    assert np.array_equal(codes == 255, ~fin) and np.isnan(back[~fin]).all()
    err = np.abs(back.astype(np.float64) - z.astype(np.float64))
    assert (err[fin] <= ref.error_bound(z, step)[fin]).all(), float((err - ref.error_bound(z, step))[fin].max())
    assert codes[fin].max(initial=0) <= 254
    return codes, lo, step


def test_symbols_declared_bound_and_exported():
    build.build()
    hdr = open(os.path.join(ROOT, "include", "baler_b200.h")).read()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in SYMBOLS:
        assert name + "(" in hdr and name in _lib.exported_symbols() and (" T " + name) in out, name
    assert "#define BB_Q8_BLOCK_ROWS 128" in hdr and latent_q8.BLOCK_ROWS == 128


@pytest.mark.parametrize("n", [1, 5, 127, 128, 129, 1000])
def test_mirror_bound_random(n):
    rng = np.random.default_rng(n)
    z = (rng.standard_normal((n, 15)) * rng.uniform(0.01, 100, 15)).astype(np.float32)
    codes, lo, step = _check_bound(z)
    for b in range(len(lo)):  # the extremes of every block column are hit exactly
        v = z[b * 128:(b + 1) * 128]
        assert np.array_equal(lo[b], v.min(axis=0))
        assert (codes[b * 128:(b + 1) * 128].min(axis=0) == 0).all()
        if len(v) > 1:  # (a one-row block has step 0)
            assert (codes[b * 128:(b + 1) * 128].max(axis=0) == 254).all()


def test_mirror_constant_nan_inf_and_huge_offset_columns():
    rng = np.random.default_rng(7)
    n = 300
    z = rng.standard_normal((n, 8)).astype(np.float32)
    z[:, 0] = 3.25                                   # constant: step 0, every code 0, exact
    z[:, 1] = np.nan                                 # all NaN: lo = step = 0, every code 255
    z[::3, 2] = np.inf                               # +-inf among finite values
    z[1::7, 2] = -np.inf
    z[:, 3] = 1e30 + rng.standard_normal(n).astype(np.float32) * 1e24   # huge offset, small spread
    z[:, 4] = np.float32(-3e38)                      # near the float32 limit
    z[5:, 4] = np.float32(3e38)
    z[:, 5] = 0.0                                    # -0 and +0 only
    z[::2, 5] = -0.0
    z[17, 6] = np.nan                                # one NaN in a random column
    codes, lo, step = _check_bound(z)
    assert (codes[:, 0] == 0).all() and (step[:, 0] == 0).all() and np.array_equal(ref.dequantize(codes, lo, step)[:, 0], z[:, 0])
    assert (codes[:, 1] == 255).all() and (lo[:, 1] == 0).all() and (step[:, 1] == 0).all()
    assert np.isfinite(step).all()
    assert np.signbit(lo[:, 5]).all()                # -0 < +0: the minimum keeps its sign bit
    assert codes[17, 6] == 255


def test_mirror_short_blocks():
    rng = np.random.default_rng(3)
    for n in (1, 2, 127, 129, 255, 257):
        z = rng.uniform(-5, 5, (n, 3)).astype(np.float32)
        codes, lo, step = _check_bound(z)
        last = z[(len(lo) - 1) * 128:]
        assert np.array_equal(lo[-1], last.min(axis=0))  # the short last block takes only its own rows
    z = np.array([[1.5, -2.0]], np.float32)  # one row: step 0, exact
    codes, lo, step = ref.quantize(z)
    assert (codes == 0).all() and np.array_equal(ref.dequantize(codes, lo, step), z)


def test_file_round_trip(tmp_path):
    rng = np.random.default_rng(11)
    z = rng.standard_normal((300, 15)).astype(np.float32)
    codes, lo, step = ref.quantize(z)
    names, feats = np.array(["a", "b"]), np.zeros((2, 24), np.float32)
    ref.write_npz(tmp_path / "mirror.npz", codes, lo, step, names, feats)
    q = latent_q8.from_npz(np.load(tmp_path / "mirror.npz"))
    assert all(np.array_equal(a, b) for a, b in zip(q, (codes, lo, step)))
    # the package's writer: the same arrays under the same keys
    np.savez(tmp_path / "pkg.npz", **latent_q8.npz_arrays(latent_q8.Q8Latent(codes, lo, step)), names=names,
             normalization_features=feats)
    a, b = np.load(tmp_path / "mirror.npz"), np.load(tmp_path / "pkg.npz")
    assert sorted(a.files) == sorted(b.files)
    for k in a.files:
        assert a[k].dtype == b[k].dtype and np.array_equal(a[k], b[k]), k
    assert latent_q8.in_file(a) and not latent_q8.in_file({"data": z})
    sub = latent_q8.rows(q, 128, 300)
    assert np.array_equal(sub.codes, codes[128:]) and np.array_equal(sub.lo, lo[1:]) and np.array_equal(sub.step, step[1:])
    with pytest.raises(ValueError, match="block boundary"):
        latent_q8.rows(q, 100, 300)


@pytest.mark.parametrize("bad,match", [
    (dict(latent_block_rows=np.int64(64)), "blocks of"),
    (dict(latent_min=np.zeros((2, 15), np.float32)), "latent_min must be float32 of shape"),
    (dict(latent_step=np.zeros((3, 14), np.float32)), "latent_step must be float32 of shape"),
    (dict(latent_step=np.zeros((3, 15), np.float64)), "latent_step must be float32"),
    (dict(data=np.zeros((300, 15), np.int8)), "uint8"),
    (dict(latent_min=None), "no 'latent_min'"),
])
def test_reader_refuses_malformed_parameters(bad, match):
    codes, lo, step = ref.quantize(np.zeros((300, 15), np.float32))
    arrays = dict(data=codes, latent_min=lo, latent_step=step, latent_block_rows=np.int64(128))
    arrays.update(bad)
    arrays = {k: v for k, v in arrays.items() if v is not None}
    with pytest.raises(ValueError, match=match):
        latent_q8.from_npz(arrays)


@pytest.mark.parametrize("n", [0, 1, 127, 128, 129, 1000, 5_000_001])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_row_range_aligned_covers_every_row_once(n, world):
    cuts = [sharded.row_range(n, r, world, align=128) for r in range(world)]
    assert cuts[0][0] == 0 and cuts[-1][1] == n
    for (lo, hi), (lo2, _) in zip(cuts, cuts[1:]):
        assert hi == lo2
    for lo, hi in cuts:
        assert lo <= hi and (lo % 128 == 0 or lo == n)
    assert sharded.row_range(n, 0, world) == sharded.row_range(n, 0, world, align=1)  # default unchanged


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        n = 1000
        rng = np.random.default_rng(5)
        z = rng.standard_normal((n, 15)).astype(np.float32)
        codes, lo, step = ref.quantize(z)
        r0, r1 = sharded.row_range(n, rank, world, align=128)
        mine = ref.quantize(z[r0:r1])  # a shard quantised alone gives the file's blocks
        got = [sharded.gather_rows_to_rank0(mine[0], n, align=128),
               sharded.gather_rows_to_rank0(mine[1], latent_q8.n_blocks(n)),
               sharded.gather_rows_to_rank0(mine[2], latent_q8.n_blocks(n))]
        if rank == 0:
            np.save(out, np.array([np.array_equal(g, w) for g, w in zip(got, (codes, lo, step))]))
        else:
            assert all(g is None for g in got)
    finally:
        dist.destroy_process_group()


def test_aligned_shards_gather_to_the_single_process_latent_gloo(tmp_path):
    out = str(tmp_path / "ok.npy")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert np.load(out).all()


def test_fp64_with_q8_is_refused_before_any_file(tmp_path):
    cfg = SimpleNamespace(precision="fp64", latent_dtype="q8", input_path=str(tmp_path / "missing.npz"),
                          save_error_bounded_deltas=False)
    with pytest.raises(NotImplementedError, match="precision='fp64'.*latent_dtype='q8'"):
        helper.compress(str(tmp_path / "missing.pt"), cfg)
    with pytest.raises(NotImplementedError, match="latent_dtype='q8'"):
        helper.decompress(str(tmp_path / "missing.pt"), str(tmp_path / "missing.npz"), None, None, "AE", cfg, str(tmp_path),
                          None)
    assert os.listdir(tmp_path) == []


def test_latent_np_dtype_q8():
    cfg = SimpleNamespace(latent_dtype="q8", precision="auto")
    assert helper._latent_np_dtype(SimpleNamespace(dtype=torch.float32), cfg) == latent_q8.NAME


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from baler_b200.modules import models
    m = models.AE(24, 15).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.codec().compress_host_q8(np.zeros((4, 24), np.float32))
    lib = _lib.lib()
    assert lib.bb_latent_quantize_q8(None, None, 0, 15, None, None, None, None) == -1  # BB_ERR_INVALID, no silent work
