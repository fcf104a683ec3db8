"""CPU-only checks of the b-bit latent (latent_dtype "q2" ... "q8"): the bit layout of packed rows, the b = 8 mirror equal
to the 8-bit one byte for byte, the error bound on awkward columns for every b, the compressed.npz reader's refusals,
latent_dtype validation and the precision "fp64" refusal before any file is touched, and the no-CPU-fallback error."""
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import latent_packed_ref as ref
import latent_q8_ref
from baler_b200 import _lib, build, latent_q8
from baler_b200.modules import helper

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BITS = list(range(2, 9))
SYMBOLS = ("bb_latent_quantize_packed", "bb_latent_dequantize_packed", "bb_compress_host_packed",
           "bb_decompress_host_packed")


def test_symbols_declared_bound_and_exported():
    build.build()
    hdr = open(os.path.join(ROOT, "include", "baler_b200.h")).read()
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    for name in SYMBOLS:
        assert name + "(" in hdr and name in _lib.exported_symbols() and (" T " + name) in out, name
    assert "#define BB_LATENT_MIN_BITS 2" in hdr and "#define BB_LATENT_MAX_BITS 8" in hdr
    assert (latent_q8.MIN_BITS, latent_q8.MAX_BITS) == (2, 8)


@pytest.mark.parametrize("bits,z,row,want", [
    # z * b a multiple of 8
    (4, 2, [0x3, 0xA], [0xA3]),
    (2, 4, [1, 2, 3, 0], [0b00111001]),
    (8, 3, [1, 200, 255], [1, 200, 255]),
    (4, 4, [0xF, 0x1, 0x2, 0x3], [0x1F, 0x32]),
    # z * b not a multiple of 8: codes straddle bytes, the last byte's high bits stay 0
    (3, 3, [0b101, 0b011, 0b111], [0b11011101, 0b1]),
    (5, 2, [0b10011, 0b01110], [0b11010011, 0b01]),
    (7, 2, [0x7F, 0x01], [0xFF, 0x00]),
    (7, 3, [0x01, 0x7E, 0x55], [0x01, 0x7F, 0x15]),
    (6, 1, [0b111111], [0b00111111]),
    (2, 5, [3, 3, 3, 3, 3], [0xFF, 0x03]),
])
def test_bit_layout_on_hand_made_rows(bits, z, row, want):
    codes = np.array([row, row[::-1]], np.uint8)
    packed = ref.pack(codes, bits)
    assert packed.shape == (2, latent_q8.row_bytes(z, bits)) == (2, (z * bits + 7) // 8)
    # the layout spelled out: bit k of the row is bit k % 8 of byte k // 8
    for r in range(2):
        bitstring = 0
        for j, c in enumerate(codes[r]):
            bitstring |= int(c) << (j * bits)
        assert bytes(packed[r]) == bitstring.to_bytes(packed.shape[1], "little")
    assert list(packed[0]) == want
    assert np.array_equal(ref.unpack(packed, z, bits), codes)


@pytest.mark.parametrize("bits", BITS)
def test_pack_unpack_round_trip_and_zero_padding(bits):
    rng = np.random.default_rng(bits)
    for z in (1, 3, 15, 31, 33):
        codes = rng.integers(0, 2 ** bits, (257, z)).astype(np.uint8)
        packed = ref.pack(codes, bits)
        assert np.array_equal(ref.unpack(packed, z, bits), codes)
        spare = packed.shape[1] * 8 - z * bits
        if spare:
            assert (packed[:, -1] >> (8 - spare) == 0).all()


def test_b8_is_the_q8_mirror_byte_for_byte(tmp_path):
    rng = np.random.default_rng(8)
    z = (rng.standard_normal((1000, 15)) * rng.uniform(0.01, 100, 15)).astype(np.float32)
    z[3, 2], z[7, 9], z[8, 9] = np.nan, np.inf, -np.inf
    codes, lo, step = ref.quantize(z, 8)
    c8, lo8, st8 = latent_q8_ref.quantize(z)
    assert np.array_equal(codes, c8) and np.array_equal(lo.view(np.uint32), lo8.view(np.uint32))
    assert np.array_equal(step.view(np.uint32), st8.view(np.uint32))
    assert np.array_equal(ref.pack(codes, 8), c8)
    back, back8 = ref.dequantize(codes, lo, step, 8), latent_q8_ref.dequantize(c8, lo8, st8)
    assert np.array_equal(back.view(np.uint32), back8.view(np.uint32))
    names, feats = np.array(["a"]), np.zeros((2, 24), np.float32)
    ref.write_npz(tmp_path / "p.npz", ref.pack(codes, 8), lo, step, 8, names, feats)
    latent_q8_ref.write_npz(tmp_path / "q.npz", c8, lo8, st8, names, feats)
    np.savez(tmp_path / "pkg.npz", **latent_q8.npz_arrays(latent_q8.PackedLatent(c8, lo8, st8, 8)), names=names,
             normalization_features=feats)
    assert open(tmp_path / "p.npz", "rb").read() == open(tmp_path / "q.npz", "rb").read()
    assert open(tmp_path / "pkg.npz", "rb").read() == open(tmp_path / "q.npz", "rb").read()


def _check_bound(z, bits):
    codes, lo, step = ref.quantize(z, bits)
    assert codes.shape == z.shape and lo.shape == step.shape == (latent_q8.n_blocks(len(z)), z.shape[1])
    back = ref.dequantize(codes, lo, step, bits)
    fin = np.isfinite(z)
    assert np.array_equal(codes == 2 ** bits - 1, ~fin) and np.isnan(back[~fin]).all()
    err = np.abs(back.astype(np.float64) - z.astype(np.float64))
    bound = ref.error_bound(z, step, bits)
    assert (err[fin] <= bound[fin]).all(), float((err - bound)[fin].max())
    assert codes[fin].max(initial=0) <= 2 ** bits - 2
    assert np.array_equal(ref.unpack(ref.pack(codes, bits), z.shape[1], bits), codes)
    return codes, lo, step


@pytest.mark.parametrize("bits", BITS)
def test_bound_random_and_extremes_hit(bits):
    rng = np.random.default_rng(100 + bits)
    z = (rng.standard_normal((1000, 15)) * rng.uniform(0.01, 100, 15)).astype(np.float32)
    codes, lo, step = _check_bound(z, bits)
    for b in range(len(lo)):
        blk = codes[b * 128:(b + 1) * 128]
        assert np.array_equal(lo[b], z[b * 128:(b + 1) * 128].min(axis=0))
        assert (blk.min(axis=0) == 0).all() and (blk.max(axis=0) == 2 ** bits - 2).all()


@pytest.mark.parametrize("bits", BITS)
def test_bound_on_awkward_columns(bits):
    rng = np.random.default_rng(7)
    n = 300  # two whole blocks and a short one of 44 rows
    z = rng.standard_normal((n, 8)).astype(np.float32)
    z[:, 0] = 3.25                                   # constant: step 0, every code 0, exact
    z[:, 1] = np.nan                                 # all NaN: lo = step = 0, every code 2^b - 1
    z[::3, 2] = np.inf                               # +-inf among finite values
    z[1::7, 2] = -np.inf
    z[:, 3] = 1e30 + rng.standard_normal(n).astype(np.float32) * 1e24   # huge offset, small spread
    z[:, 4] = np.float32(-3e38)                      # near the float32 limit
    z[5:, 4] = np.float32(3e38)
    z[:, 5] = 0.0                                    # -0 and +0 only
    z[::2, 5] = -0.0
    z[17, 6] = np.nan                                # one NaN in a random column
    codes, lo, step = _check_bound(z, bits)
    assert (codes[:, 0] == 0).all() and (step[:, 0] == 0).all()
    assert np.array_equal(ref.dequantize(codes, lo, step, bits)[:, 0], z[:, 0])
    assert (codes[:, 1] == 2 ** bits - 1).all() and (lo[:, 1] == 0).all() and (step[:, 1] == 0).all()
    assert np.isfinite(step).all() and np.signbit(lo[:, 5]).all()
    assert codes[17, 6] == 2 ** bits - 1
    assert lo[-1, 7] == z[256:, 7].min()  # the short last block takes only its own rows


@pytest.mark.parametrize("bits", [2, 3, 8])
def test_short_blocks(bits):
    rng = np.random.default_rng(3)
    for n in (1, 2, 127, 129, 255, 257):
        z = rng.uniform(-5, 5, (n, 3)).astype(np.float32)
        codes, lo, step = _check_bound(z, bits)
        assert np.array_equal(lo[-1], z[(len(lo) - 1) * 128:].min(axis=0))


def _arrays(bits, n=300, z=15):
    codes, lo, step = ref.quantize(np.random.default_rng(1).standard_normal((n, z)).astype(np.float32), bits)
    out = dict(data=ref.pack(codes, bits), latent_min=lo, latent_step=step, latent_block_rows=np.int64(128))
    if bits != 8:
        out["latent_bits"] = np.int64(bits)
    return out, codes


@pytest.mark.parametrize("bits", BITS)
def test_reader_round_trip(tmp_path, bits):
    arrays, codes = _arrays(bits)
    np.savez(tmp_path / "c.npz", **arrays)
    q = latent_q8.read(np.load(tmp_path / "c.npz"))
    assert isinstance(q, latent_q8.PackedLatent) and q.bits == bits and q.codes.shape == (300, (15 * bits + 7) // 8)
    assert np.array_equal(ref.unpack(q.codes, 15, bits), codes)
    # the package's writer gives the same keys and arrays; latent_bits only below 8 bits
    pkg = latent_q8.npz_arrays(q)
    assert sorted(pkg) == sorted(arrays) and all(np.array_equal(pkg[k], arrays[k]) for k in arrays)
    assert ("latent_bits" in pkg) == (bits != 8)
    sub = latent_q8.rows(q, 128, 300)
    assert sub.bits == bits and np.array_equal(sub.codes, q.codes[128:]) and np.array_equal(sub.lo, q.lo[1:])
    if bits == 8:
        assert isinstance(latent_q8.from_npz(arrays), latent_q8.Q8Latent)
    else:
        with pytest.raises(ValueError, match="%d-bit latent" % bits):
            latent_q8.from_npz(arrays)


@pytest.mark.parametrize("bits,bad,match", [
    (4, dict(latent_bits=np.int64(1)), "latent_bits must be one integer from 2 to 8"),
    (4, dict(latent_bits=np.int64(9)), "latent_bits must be one integer from 2 to 8"),
    (4, dict(latent_bits=np.array([4, 4])), "latent_bits must be one integer"),
    (4, dict(latent_bits=np.float64(4)), "latent_bits must be one integer"),
    (4, dict(latent_bits=None), "data must be 15 bytes wide"),  # a missing latent_bits reads as 8 bits
    (4, dict(latent_bits=np.int64(3)), "data must be 6 bytes wide"),
    (3, dict(data=np.zeros((300, 5), np.uint8)), "data must be 6 bytes wide"),
    (8, dict(data=np.zeros((300, 8), np.uint8)), "data must be 15 bytes wide"),
    (4, dict(data=np.zeros((300, 8), np.int8)), "uint8"),
    (4, dict(data=np.zeros((300, 8, 1), np.uint8)), "2-D uint8"),
    (4, dict(latent_min=np.zeros((2, 15), np.float32)), "latent_min must be float32 of shape"),
    (4, dict(latent_min=np.zeros(15, np.float32)), "latent_min must be float32 of shape"),
    (4, dict(latent_step=np.zeros((3, 14), np.float32)), "latent_step must be float32 of shape"),
    (4, dict(latent_step=np.zeros((3, 15), np.float64)), "latent_step must be float32"),
    (4, dict(latent_block_rows=np.int64(64)), "blocks of"),
    (4, dict(latent_min=None), "no 'latent_min'"),
])
def test_reader_refuses(bits, bad, match):
    arrays, _ = _arrays(bits)
    arrays.update(bad)
    arrays = {k: v for k, v in arrays.items() if v is not None}
    with pytest.raises(ValueError, match=match):
        latent_q8.read(arrays)


@pytest.mark.parametrize("name,bits", [("q%d" % b, b) for b in BITS] + [("float16", None), ("float64", None), (None, None)])
def test_bits_of_valid(name, bits):
    assert latent_q8.bits_of(name) == bits


@pytest.mark.parametrize("name", ["q1", "q9", "q", "q08", "q4 ", "qx"])
def test_unknown_q_value_is_refused_before_any_file(tmp_path, name):
    with pytest.raises(ValueError, match="latent_dtype"):
        latent_q8.bits_of(name)
    cfg = SimpleNamespace(precision="auto", latent_dtype=name, input_path=str(tmp_path / "missing.npz"),
                          save_error_bounded_deltas=False)
    with pytest.raises(ValueError, match="latent_dtype %r" % name):
        helper.compress(str(tmp_path / "missing.pt"), cfg)
    with pytest.raises(ValueError, match="latent_dtype %r" % name):
        helper.decompress(str(tmp_path / "missing.pt"), str(tmp_path / "missing.npz"), None, None, "AE", cfg, str(tmp_path),
                          None)
    assert os.listdir(tmp_path) == []


@pytest.mark.parametrize("bits", BITS)
def test_fp64_is_refused_before_any_file(tmp_path, bits):
    cfg = SimpleNamespace(precision="fp64", latent_dtype="q%d" % bits, input_path=str(tmp_path / "missing.npz"),
                          save_error_bounded_deltas=True)
    with pytest.raises(NotImplementedError, match="precision='fp64'.*latent_dtype='q%d'" % bits):
        helper.compress(str(tmp_path / "missing.pt"), cfg)
    with pytest.raises(NotImplementedError, match="latent_dtype='q%d'" % bits):
        helper.decompress(str(tmp_path / "missing.pt"), str(tmp_path / "missing.npz"), None, None, "AE", cfg, str(tmp_path),
                          None)
    assert os.listdir(tmp_path) == []


@pytest.mark.parametrize("bits", BITS)
def test_latent_np_dtype(bits):
    cfg = SimpleNamespace(latent_dtype="q%d" % bits, precision="auto")
    assert helper._latent_np_dtype(SimpleNamespace(dtype=torch.float32), cfg) == "q%d" % bits


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    from baler_b200.modules import models
    m = models.AE(24, 15).eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.codec().compress_host_packed(np.zeros((4, 24), np.float32), 4)
    lib = _lib.lib()
    assert lib.bb_latent_quantize_packed(None, None, 0, 15, 4, None, None, None, None) == -1  # BB_ERR_INVALID
    assert lib.bb_compress_host_packed(None, None, 0, None, 0, 4, None, None, None, 0) == -1
