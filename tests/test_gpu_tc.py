"""tcgen05 path (BB_PREC_SPLIT16): step-by-step accumulator dumps against the oracle, then end-to-end parity.
The step dumps localise a wrong descriptor / layout to one MMA of the program."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import rel_l2, rel_max, sub_sd
from oracle import baler_oracle as orc
from baler_b200 import _lib, synth
from baler_b200.modules import models

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ae(golden):
    g = golden("ae_cms.npz")
    m = models.AE(24, 15)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sub_sd(g, "sd").items()})
    return m.eval(), sub_sd(g, "sd"), g


def debug_chain(codec, decode, x, out_dim, step, width, groups=0, fast=0):
    lib = _lib.lib()
    fn = lib.bb_debug_tc_chain
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    n = x.shape[0]
    out = torch.full((n, out_dim), float("nan"), dtype=torch.float32, device="cuda")
    dbg = torch.full((n, max(width, 1)), float("nan"), dtype=torch.float32, device="cuda")
    rc = fn(codec.handle, decode, x.data_ptr(), n, out.data_ptr(), fast, step, dbg.data_ptr() if step >= 0 else None,
            groups, None)
    assert rc == 0, rc
    torch.cuda.synchronize()
    return out.cpu().numpy(), dbg.cpu().numpy()


def pre_activations(sd, names, x):
    """float64 pre-activations of the 4 layers of one direction"""
    outs, h = [], x
    for i, n in enumerate(names):
        a = h @ sd[n + ".weight"].T + sd[n + ".bias"]
        outs.append(a)
        h = orc.leaky_relu(a) if i < 3 else a
    return outs


@pytest.mark.parametrize("groups", [1, 2])
@pytest.mark.parametrize("n", [128, 1000])
def test_encoder_steps(ae, groups, n):
    m, sd, g = ae
    codec = m.codec()
    if codec.auto_precision != "split16":
        pytest.skip("tcgen05 path not available for this shape")
    x = orc.normalize(synth.cms_table(4096, seed=2))[:n]
    pre = pre_activations(sd, ("en1", "en2", "en3", "en4"), x.astype(np.float64))
    xd = torch.from_numpy(x).cuda()
    # (step, width, oracle slice, index of the constant-one column or None)
    plan = [(0, 112, pre[0][:, :112], None), (1, 96, pre[0][:, 112:200], 88), (2, 112, pre[1], 100),
            (3, 64, pre[2], 50), (4, 16, pre[3], None)]
    for step, width, ref, one in plan:
        _, dbg = debug_chain(codec, 0, xd, 15, step, width, groups)
        k = ref.shape[1]
        err = rel_max(dbg[:, :k], ref)
        assert err <= 1e-5, (step, err)
        if one is not None:
            assert np.array_equal(dbg[:, one], np.ones(n, dtype=np.float32)), step
            assert not dbg[:, one + 1:].any(), step
    out, _ = debug_chain(codec, 0, xd, 15, -1, 1, groups)
    assert rel_max(out, pre[3]) <= 1e-5 and rel_l2(out, pre[3]) <= 1e-5


@pytest.mark.parametrize("groups", [1, 2])
def test_decoder_steps(ae, groups):
    m, sd, g = ae
    codec = m.codec()
    if codec.auto_precision != "split16":
        pytest.skip("tcgen05 path not available for this shape")
    z = g["latent"][:200]
    pre = pre_activations(sd, ("de1", "de2", "de3", "de4"), z)
    zd = torch.from_numpy(z.astype(np.float32)).cuda()
    plan = [(0, 64, pre[0], 50), (1, 112, pre[1], 100), (2, 112, pre[2][:, :112], None), (3, 96, pre[2][:, 112:200], 88),
            (4, 32, pre[3], None)]
    for step, width, ref, one in plan:
        _, dbg = debug_chain(codec, 1, zd, 24, step, width, groups)
        k = ref.shape[1]
        err = rel_max(dbg[:, :k], ref)
        assert err <= 1e-5, (step, err)
    out, _ = debug_chain(codec, 1, zd, 24, -1, 1, groups)
    assert rel_max(out, pre[3]) <= 1e-5 and rel_l2(out, pre[3]) <= 1e-5


def test_split16_error_budget(ae):
    """measured error of the 3-product split against float64 on 200k rows, and the fast (1-product) mode"""
    m, sd, _ = ae
    codec = m.codec()
    if codec.auto_precision != "split16":
        pytest.skip("tcgen05 path not available for this shape")
    x = orc.normalize(synth.cms_table(200000, seed=4))
    zr = orc.ae_encode(sd, x)
    xd = torch.from_numpy(x).cuda()
    z = codec.encode(xd, precision="split16").cpu().numpy()
    zf = codec.encode(xd, precision="fp32").cpu().numpy()
    zfast = codec.encode(xd, precision="fast").cpu().numpy()
    e_split, e_f32, e_fast = rel_max(z, zr), rel_max(zf, zr), rel_max(zfast, zr)
    print("\nsplit16 %.2e  fp32 %.2e  fast16 %.2e (max-norm rel. error of the latent vs float64)" % (e_split, e_f32, e_fast))
    assert e_split <= 1e-5 and e_f32 <= 1e-5
    assert 1e-5 < e_fast < 1e-2  # single product: documented as outside the tolerance
    yr = orc.ae_decode(sd, zr)
    y = codec.decode(torch.from_numpy(zr.astype(np.float32)).cuda(), precision="split16").cpu().numpy()
    assert rel_max(y, yr) <= 1e-5 and rel_l2(y, yr) <= 1e-5


def test_range_guard(ae):
    """values beyond the fp16 range poison a row of the split path: the flag is raised and the wrappers fall back"""
    m, sd, _ = ae
    codec = m.codec()
    if codec.auto_precision != "split16":
        pytest.skip("tcgen05 path not available for this shape")
    x = synth.cms_table(1000, seed=6) * 1e4  # |x| up to ~1e6 > 65504
    zr = orc.ae_encode(sd, x.astype(np.float64))
    z = codec.encode(torch.from_numpy(x).cuda(), precision="auto").cpu().numpy()
    assert np.isfinite(z).all()
    assert rel_max(z, zr) <= 1e-5


@pytest.mark.parametrize("n_features,z_dim", [(4, 2), (15, 15), (16, 8), (24, 15), (10, 20), (31, 16), (31, 31)])
def test_tc_shape_family_vs_oracle(n_features, z_dim):
    """every instantiation of the statically shaped tcgen05 kernel (padded first K 16 / 32, padded last N 16 / 32, both
    directions): random reference-initialised AE(n_features, z_dim), fused normalisation / un-normalisation, ragged row
    counts (single rows, tile tails whose byte count is not a multiple of 16, fewer tiles than SMs, many tiles).  The same
    shapes on the fused fp32 chain (precision "fp32") and in single-product mode ("fast": the table-driven kernel except
    on the two CMS instantiations; documented as outside the 1e-5 bar)"""
    torch.manual_seed(100 * n_features + z_dim)
    m = models.AE(n_features, z_dim).eval()
    sd = {k: v.numpy().astype(np.float64) for k, v in m.state_dict().items()}
    codec = m.codec()
    assert codec.auto_precision == "split16"
    rng = np.random.default_rng(n_features * 7 + z_dim)
    for n in (1, 3, 129, 300, 4097, 50021):
        raw = (rng.lognormal(0.0, 1.0, size=(n, n_features)) + rng.integers(0, 5, size=(1, n_features))).astype(np.float32)
        mn = raw.min(axis=0) - 0.25
        rg = (raw.max(axis=0) - mn + 0.5).astype(np.float32)
        xn = ((raw - mn) / rg).astype(np.float64)  # numpy float32 normalisation, then the float64 reference chain
        zr = orc.ae_encode(sd, xn)
        yr = orc.ae_decode(sd, zr) * rg.astype(np.float64) + mn.astype(np.float64)
        x_dev = torch.from_numpy(raw).cuda()
        mn_d, rg_d = torch.from_numpy(mn).cuda(), torch.from_numpy(rg).cuda()
        for precision, tol in (("split16", 1e-5), ("fp32", 1e-5), ("fast", 1e-2)):
            z = codec.encode(x_dev, mn_d, rg_d, precision=precision)
            assert rel_max(z.cpu().numpy(), zr) <= tol and rel_l2(z.cpu().numpy(), zr) <= tol, (n, precision, rel_max(z.cpu().numpy(), zr))
            y = codec.decode(torch.from_numpy(zr.astype(np.float32)).cuda(), mn_d, rg_d, precision=precision)
            assert rel_max(y.cpu().numpy(), yr) <= tol and rel_l2(y.cpu().numpy(), yr) <= tol, (n, precision, rel_max(y.cpu().numpy(), yr))
    assert not codec.range_flag()
