"""Dense encode / decode on every kernel the dispatcher (run_chain, bb_api.cu) can pick, against float64 numpy.

A direction of a dense model runs on one of: the fused fp32 chain (chain_f32_kernel; tile of 80, 64 or 32 rows, the
tallest whose activations fit the shared memory the weights leave), the statically shaped tcgen05 kernel
(chain_tc4_kernel: the AE family), the table-driven tcgen05 kernel (chain_tc_kernel: other 4-layer chains, rows that are
not 16-byte aligned, the single-product "fast" mode) or the per-layer GEMMs (fp32, mma.sync, tcgen05) of models too wide
for shared memory.  The shapes below land on each of them, and the test hook bb_debug_last_route reports the kernel and
tile of every launch: a change of the dispatch rules that moves a case onto another kernel fails here.

Bar: max|d| / max|ref| <= 1e-5 and ||d|| / ||ref|| <= 1e-5 per tensor (1e-2 for "fast", documented as outside it; 1e-3
for a float16 latent).  Inputs are normalised in float32 the way numpy does it, then widened."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import rel_l2, rel_max
from oracle import baler_oracle as orc
from baler_b200 import _lib, engine
from baler_b200.modules import models

pytestmark = pytest.mark.gpu

TOL, FAST_TOL, F16_TOL = 1e-5, 1e-2, 1e-3
# BbRoute (bb_common.cuh)
F32, TC4, TC, LAY_F32, LAY_MMA, LAY_TC5 = 1, 2, 3, 4, 5, 6
ROUTE = {F32: "chain_f32", TC4: "chain_tc4", TC: "chain_tc", LAY_F32: "layered fp32", LAY_MMA: "layered mma.sync",
         LAY_TC5: "layered tcgen05"}
N_BIG = 50021  # the one large row count of every route
HIT = {}       # (kernel, tile rows) -> cases that ran on it (layered GEMMs: tile 0, their chunk follows the row count)
RAN = set()
# every (kernel, tile) the cases below must reach between them
REQUIRED = {(F32, 80), (F32, 64), (F32, 32), (TC4, 256), (TC, 128), (TC, 256), (LAY_F32, 0)}


def last_route(codec, direction):
    fn = _lib.lib().bb_debug_last_route
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    k, t = C.c_int(-1), C.c_int(-1)
    assert fn(codec.handle, direction, C.byref(k), C.byref(t)) == 0
    return k.value, (0 if k.value in (LAY_F32, LAY_MMA, LAY_TC5) else t.value)


def debug_chain(codec, decode, x, out_dim, groups, fast):
    """one direction on the table-driven tcgen05 kernel with 1 or 2 pipelines per CTA (bb_debug_tc_chain, no features)"""
    fn = _lib.lib().bb_debug_tc_chain
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    out = torch.full((x.shape[0], out_dim), float("nan"), dtype=torch.float32, device="cuda")
    assert fn(codec.handle, decode, x.data_ptr(), x.shape[0], out.data_ptr(), fast, -1, None, groups, None) == 0
    torch.cuda.synchronize()
    return out


def dense_ref(layers, v):
    v = np.asarray(v, dtype=np.float64)
    for w, b, a in layers:
        v = v @ w.T + b
        v = np.where(v > 0, v, orc.LEAKY_SLOPE * v) if a == "leaky" else np.maximum(v, 0.0) if a == "relu" else v
    return v


# ------------------------------------------------------------------ cases
# Each case: a model, its float64 reference per direction, and per direction (kind, tile of the fused fp32 chain or None).
# kind "f32": no tensor-core form, the fused fp32 chain; "tc4": the AE family on chain_tc4_kernel; "tc": a 4-layer chain
# outside the family on chain_tc_kernel; "layered": too wide for the fused kernels.  The tiles follow bb_chain_f32_prepare
# with 227 KB of opt-in shared memory.
def _ae(cls, f, z):
    def build():
        torch.manual_seed(1000 * f + z)
        m = cls(f, z)
        if cls is models.AE_Dropout_BN:  # a BatchNorm that is not the identity once folded
            sd = m.state_dict()
            g = torch.Generator().manual_seed(f + z)
            for bn in m.bn_names:
                n = sd[bn + ".weight"].shape
                sd[bn + ".weight"] = (0.5 + torch.rand(n, generator=g)).double()
                sd[bn + ".bias"] = (0.2 * torch.randn(n, generator=g)).double()
                sd[bn + ".running_mean"] = (0.1 * torch.randn(n, generator=g)).double()
                sd[bn + ".running_var"] = (0.5 + torch.rand(n, generator=g)).double()
            m.load_state_dict(sd)
        m.eval()
        sd = {k: v.numpy().astype(np.float64) for k, v in m.state_dict().items()}
        if cls is models.AE_Dropout_BN:
            return m.codec(), sd, (lambda x: orc.dbn_encode(sd, x), lambda z_: orc.dbn_decode(sd, z_))
        return m.codec(), sd, (lambda x: orc.ae_encode(sd, x), lambda z_: orc.ae_decode(sd, z_))
    return build


def _dense(dims_e, acts_e, acts_d, seed):
    def build():
        rng = np.random.default_rng(seed)
        dims_d = dims_e[::-1]

        def layers(dims, acts):
            return [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i]), 0.1 * rng.standard_normal(dims[i + 1]),
                     acts[i]) for i in range(len(dims) - 1)]

        enc, dec = layers(dims_e, acts_e), layers(dims_d, acts_d)
        return engine.DenseCodec(enc, dec), None, (lambda x: dense_ref(enc, x), lambda z_: dense_ref(dec, z_))
    return build


CASES = {
    # fused fp32, tile 80 (AE(24, 40): TN = 2 on the last encoder layer)
    "AE(33,8)": (_ae(models.AE, 33, 8), ("f32", 80), ("f32", 80)),
    "AE(24,40)": (_ae(models.AE, 24, 40), ("f32", 80), ("f32", 80)),
    # fused fp32, tile 64
    "AE(40,10)": (_ae(models.AE, 40, 10), ("f32", 64), ("f32", 64)),
    "AE(24,64)": (_ae(models.AE, 24, 64), ("f32", 64), ("f32", 64)),
    # fused fp32, tile 32 (AE(24, 200): a latent wider than the hidden 50)
    "CFD_dense_AE(64,10)": (_ae(models.CFD_dense_AE, 64, 10), ("f32", 32), ("f32", 32)),
    "AE(96,24)": (_ae(models.AE, 96, 24), ("f32", 32), ("f32", 32)),
    "AE(24,200)": (_ae(models.AE, 24, 200), ("f32", 32), ("f32", 32)),
    # mixed: one direction on tcgen05, the other on the fp32 chain; the fp32 chain at its shared-memory limit (105
    # features) with a layered decoder; the first shape past that limit.  AE(31, 32)'s encoder is in the family, but
    # chain_tc4_kernel's two pipelines of 31-column input and 32-column output stages do not fit shared memory beside its
    # weights, so bb_tc4_launch hands it to the table-driven kernel with one pipeline
    "AE(32,15)": (_ae(models.AE, 32, 15), ("f32", 80), ("tc4", 80)),
    "AE(31,32)": (_ae(models.AE, 31, 32), ("tc", 64), ("f32", 64)),
    "AE(105,15)": (_ae(models.AE, 105, 15), ("f32", 32), ("layered", None)),
    "AE(106,15)": (_ae(models.AE, 106, 15), ("layered", None), ("layered", None)),
    # eval-mode AE_Dropout_BN: LeakyReLU on the latent, folded BatchNorm, ReLU on the output
    "AE_Dropout_BN(40,10)": (_ae(models.AE_Dropout_BN, 40, 10), ("f32", 64), ("f32", 64)),
    "AE_Dropout_BN(64,12)": (_ae(models.AE_Dropout_BN, 64, 12), ("f32", 32), ("f32", 32)),
    # the table-driven tcgen05 kernel on chains outside the family; the widest one leaves room for one pipeline only
    "dense[20,150,90,40,12]": (_dense([20, 150, 90, 40, 12], ["leaky", "relu", "none", "leaky"],
                                      ["relu", "leaky", "none", "relu"], 5), ("tc", 80), ("tc", 80)),
    "dense[31,207,111,111,20]": (_dense([31, 207, 111, 111, 20], ["relu", "leaky", "leaky", "none"],
                                        ["leaky", "none", "relu", "none"], 6), ("tc", 32), ("tc", 32)),
    "dense[3,113,5,7,2]": (_dense([3, 113, 5, 7, 2], ["leaky", "leaky", "relu", "none"],
                                  ["none", "relu", "leaky", "none"], 7), ("tc", 80), ("tc", 80)),
}
TC_GROUPS = {"dense[20,150,90,40,12]": 2, "dense[31,207,111,111,20]": 1, "dense[3,113,5,7,2]": 2}


@pytest.fixture(scope="module")
def built():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = CASES[name][0]()
        return cache[name]

    return get


def _table(n, f, seed):
    rng = np.random.default_rng(seed)
    raw = (rng.lognormal(0.0, 1.0, size=(n, f)) + rng.integers(0, 5, size=(1, f))).astype(np.float32)
    mn = raw.min(axis=0) - 0.25
    rg = (raw.max(axis=0) - mn + 0.5).astype(np.float32)
    return raw, mn, rg


def _close(a, ref, tol, what):
    a = a.detach().float().cpu().numpy() if torch.is_tensor(a) else a
    e_max, e_l2 = rel_max(a, ref), rel_l2(a, ref)
    assert e_max <= tol and e_l2 <= tol, (what, e_max, e_l2)


def _expected(kind, f32_tile, prec, in_dim, out_dim, direction, aligned):
    """(kernel, tile rows or None for "any") a direction must run on at `prec`, or None when it must refuse"""
    if prec == "fp32":
        return (LAY_F32, 0) if kind == "layered" else (F32, f32_tile)
    if kind == "f32":
        return (F32, f32_tile) if prec == "auto" else None
    if kind == "layered":
        return None if prec == "fast" else ("layered", 0)
    if kind == "tc4" and aligned:
        ka, nl = (in_dim + 1 + 15) // 16 * 16, (out_dim + 15) // 16 * 16
        cms = (ka, nl) == ((32, 16) if direction == 0 else (16, 32))  # the two instantiations with a fast form
        if prec != "fast" or cms:
            return (TC4, 256)
    return (TC, None)


def _route_ok(got, want):
    if want[0] == "layered":
        return got in ((LAY_MMA, 0), (LAY_TC5, 0))
    return got[0] == want[0] and (want[1] is None or got[1] == want[1])


@pytest.mark.parametrize("direction", [0, 1], ids=["encode", "decode"])
@pytest.mark.parametrize("case", list(CASES))
def test_route_vs_float64(built, case, direction):
    codec, _, refs = built(case)
    kind, f32_tile = CASES[case][1 + direction]
    sms = codec.ctx.sm_count
    in_dim, out_dim = (codec.n_features, codec.z_dim) if direction == 0 else (codec.z_dim, codec.n_features)
    chain_prec = _lib.lib().bb_model_chain_precision(codec.handle, direction)
    assert chain_prec == (_lib.BB_PREC_FP32 if kind == "f32" else _lib.BB_PREC_SPLIT16), (case, chain_prec)

    # inputs: the encoder reads a raw table (normalised by the kernel, or not at all), the decoder a float32 latent
    n_max = 2 * sms * 256 + 256
    raw, mn, rg = _table(max(n_max, N_BIG), codec.n_features, 11 + direction)
    xn = ((raw - mn) / rg).astype(np.float64)
    if direction == 0:
        x = raw
        ref = {True: refs[0](xn), False: refs[0](raw.astype(np.float64))}
    else:
        x = refs[0](xn).astype(np.float32)
        y = refs[1](x.astype(np.float64))
        ref = {True: y * rg.astype(np.float64) + mn.astype(np.float64), False: y}
    x_dev = torch.from_numpy(x).cuda()
    feats = (torch.from_numpy(mn).cuda(), torch.from_numpy(rg).cuda())

    def run(xd, prec, norm, out=None, out_dtype=torch.float32):
        f = feats if norm else (None, None)
        if direction == 0:
            return codec.encode(xd, f[0], f[1], out_dtype=out_dtype, precision=prec, out=out)
        return codec.decode(xd, f[0], f[1], precision=prec, out=out)

    def route(want, what):
        got = last_route(codec, direction)
        assert _route_ok(got, want), (what, "ran %s / %d, expected %s" % (ROUTE.get(got[0], got[0]), got[1], want))
        HIT.setdefault(got, set()).add(case)
        return got

    for prec in ("auto", "fp32", "split16", "fast"):
        want = _expected(kind, f32_tile, "split16" if prec == "auto" and kind != "f32" else prec, in_dim, out_dim,
                         direction, True)
        if want is None:  # a precision this direction does not have is refused, never run on another kernel
            with pytest.raises(_lib.BalerB200Error):
                run(x_dev[:5], prec, True)
            continue
        tol = FAST_TOL if prec == "fast" else TOL
        got = None
        # row counts around the route's tile T and its wave of SM-count persistent CTAs (tcgen05: 128-row tiles, the
        # hook reports the rows a CTA keeps in flight)
        run(x_dev[:1].clone(), prec, True)
        got = route(want, (case, prec, 1))
        t = got[1] if got[0] == F32 else 128
        per_cta = got[1] if got[0] in (F32, TC4, TC) else 128
        counts = sorted({1, t - 1, t + 1, sms * per_cta - 1, sms * per_cta + 1, 2 * sms * per_cta + t // 2 + 3, N_BIG})
        for n in counts:
            for norm in (True, False):
                out = run(x_dev[:n], prec, norm)
                route(want, (case, prec, n, norm))
                _close(out, ref[norm][:n], tol, (case, prec, n, norm))
        n = counts[-2]
        # float16 latent: the encoder's output to 1e-3; the decoder against the oracle fed the same float16 values
        if direction == 0:
            z16 = run(x_dev[:n], prec, True, out_dtype=torch.float16)
            assert z16.dtype == torch.float16
            route(want, (case, prec, "fp16 out"))
            _close(z16, ref[True][:n], max(tol, F16_TOL), (case, prec, "fp16 latent"))
        else:
            z16 = x[:n].astype(np.float16)
            y16 = run(torch.from_numpy(z16).cuda(), prec, True)
            route(want, (case, prec, "fp16 in"))
            _close(y16, refs[1](z16.astype(np.float64)) * rg.astype(np.float64) + mn.astype(np.float64), tol,
                   (case, prec, "fp16 latent in"))
        # rows that are only 4-byte aligned, in and out, and out alone: chain_tc4_kernel's bulk copies need 16 bytes,
        # so the family shapes move onto the table-driven kernel
        want_u = _expected(kind, f32_tile, "split16" if prec == "auto" and kind != "f32" else prec, in_dim, out_dim,
                           direction, False)
        for in_u in (True, False):
            if in_u:
                flat = torch.empty(n * in_dim + 1, dtype=torch.float32, device="cuda")
                flat[1:].copy_(x_dev[:n].reshape(-1))
                xu = flat[1:].view(n, in_dim)
                assert xu.data_ptr() % 16 == 4
            else:
                xu = x_dev[:n]
            oflat = torch.full((n * out_dim + 1,), float("nan"), dtype=torch.float32, device="cuda")
            ou = oflat[1:].view(n, out_dim)
            res = run(xu, prec, True, out=ou)
            assert res.data_ptr() == ou.data_ptr()
            route(want_u, (case, prec, "unaligned", in_u))
            _close(ou, ref[True][:n], tol, (case, prec, "unaligned", in_u))
        # the fused kernels treat rows independently: a slice gives the bits of the whole, identical rows identical bits
        # (not on the layered GEMMs, whose mode depends on the row count)
        if got[0] in (F32, TC4, TC):
            full = run(x_dev[:N_BIG], prec, True)
            a = 3 * t + 5
            b = a + sms * t + 7
            part = run(x_dev[a:b].clone(), prec, True)
            route(want, (case, prec, "slice"))
            assert torch.equal(part, full[a:b]), (case, prec, "slice differs from the whole")
            rep = run(x_dev[:t + 3].repeat(3, 1), prec, True)
            assert torch.equal(rep[:t + 3], rep[t + 3:2 * t + 6]) and torch.equal(rep[:t + 3], rep[2 * t + 6:])
            assert torch.equal(rep[:t + 3], full[:t + 3])
    assert not codec.range_flag()
    RAN.add((case, direction))


@pytest.mark.parametrize("direction", [0, 1], ids=["encode", "decode"])
@pytest.mark.parametrize("case", list(TC_GROUPS))
def test_table_driven_pipelines_vs_float64(built, case, direction):
    """chain_tc_kernel with one and with two pipelines per CTA (bb_debug_tc_chain's force_groups), exact and single
    product; two pipelines where the chain's weights leave room for them"""
    codec, _, refs = built(case)
    sms = codec.ctx.sm_count
    raw, _, _ = _table(2 * sms * 256 + 256, codec.n_features, 21 + direction)
    x = raw if direction == 0 else refs[0](raw.astype(np.float64)).astype(np.float32)
    ref = refs[direction](x.astype(np.float64))
    x_dev = torch.from_numpy(x).cuda()
    out_dim = codec.z_dim if direction == 0 else codec.n_features
    for groups in (1, 2):
        per_cta = 128 * min(groups, TC_GROUPS[case])
        for fast in (0, 1):
            for n in (1, 127, 129, sms * per_cta - 1, sms * per_cta + 1, 2 * sms * per_cta + 67):
                out = debug_chain(codec, direction, x_dev[:n], out_dim, groups, fast)
                got = last_route(codec, direction)
                assert got == (TC, per_cta), (case, groups, got)
                HIT.setdefault(got, set()).add(case)
                _close(out, ref[:n], FAST_TOL if fast else TOL, (case, groups, fast, n))
    assert not codec.range_flag()


# ------------------------------------------------------------------ host pipelines
PIPE_CASES = ["AE(32,15)", "AE(31,32)", "AE(105,15)", "AE(106,15)", "AE(40,10)"]


@pytest.mark.parametrize("case", PIPE_CASES)
def test_host_pipelines(built, case):
    """compress_host / decompress_host over more rows than one pipeline chunk (2^21), latents float32 / float64 /
    float16 and reconstructions float32 / float64, checked on sampled rows against the oracle"""
    codec, sd, refs = built(case)
    f = codec.n_features
    n = (1 << 22) + 12345
    rng = np.random.default_rng(f)
    base, _, _ = _table(1 << 16, f, 31)
    table = np.ascontiguousarray(base[rng.integers(0, len(base), size=n)])
    idx = np.unique(np.concatenate([np.arange(64), (1 << 21) + np.arange(-64, 64), (1 << 22) + np.arange(-64, 64),
                                    np.arange(n - 64, n), rng.integers(0, n, size=4096)]))
    zs = {}
    for z_dtype in (np.float32, np.float64, np.float16):
        z, feats = codec.compress_host(table, recompute_minmax=True, z_dtype=z_dtype)
        assert z.dtype == z_dtype and np.array_equal(feats, orc.find_minmax(table))
        xn = ((table[idx] - feats[0]) / feats[1]).astype(np.float64)
        _close(z[idx], refs[0](xn), F16_TOL if z_dtype == np.float16 else TOL, (case, z_dtype))
        zs[z_dtype] = z
    assert np.array_equal(zs[np.float64], zs[np.float32].astype(np.float64))  # widened on the host, exactly
    for y_dtype in (np.float32, np.float64):
        y = codec.decompress_host(zs[np.float32], features=feats, y_dtype=y_dtype)
        assert y.dtype == y_dtype
        yr = orc.renormalize(refs[1](zs[np.float32][idx].astype(np.float64)), feats[0], feats[1])
        _close(y[idx], yr, TOL, (case, y_dtype))
    assert not codec.range_flag()


@pytest.mark.parametrize("case", ["AE(32,15)", "AE(31,32)", "AE(105,15)", "AE(106,15)"])
def test_host_pipeline_range_fallback(built, case):
    """values beyond the fp16 range: with precision "auto" the tensor-core direction re-runs on the fp32 kernels and
    matches the oracle; a direction on the fp32 chain runs once and raises no flag"""
    codec, _, refs = built(case)
    kinds = (CASES[case][1][0], CASES[case][2][0])
    raw, _, _ = _table(5000, codec.n_features, 41)
    table = raw * np.float32(3e4)  # |x| up to ~2e6
    z, _ = codec.compress_host(table, z_dtype=np.float32)
    _close(z, refs[0](table.astype(np.float64)), TOL, (case, "encode"))
    fp32_route = (LAY_F32, 0) if kinds[0] == "layered" else (F32, CASES[case][1][1])
    assert last_route(codec, 0) == fp32_route, (case, last_route(codec, 0))
    zbig = (np.random.default_rng(3).standard_normal((5000, codec.z_dim)) * 1e6).astype(np.float32)
    y = codec.decompress_host(zbig, y_dtype=np.float32)
    _close(y, refs[1](zbig.astype(np.float64)), TOL, (case, "decode"))
    fp32_route = (LAY_F32, 0) if kinds[1] == "layered" else (F32, CASES[case][2][1])
    assert last_route(codec, 1) == fp32_route, (case, last_route(codec, 1))
    assert not codec.range_flag()
    # in range, the tensor-core directions stay on their kernels
    z, feats = codec.compress_host(raw, recompute_minmax=True, z_dtype=np.float32)
    codec.decompress_host(z, features=feats, y_dtype=np.float32)
    for d, kind in enumerate(kinds):
        want = _expected(kind, CASES[case][1 + d][1], "split16" if kind != "f32" else "auto", 0, 0, d, True)
        got = last_route(codec, d)
        assert _route_ok(got, (want[0], None) if want[0] == TC4 else want), (case, d, got)
        HIT.setdefault(got, set()).add(case)


def test_every_route_was_hit():
    """runs last: every (kernel, tile) the cases above are there for was reached"""
    if len(RAN) < 2 * len(CASES):
        pytest.skip("only part of this file ran")
    print("\nroutes hit:")
    for (k, t), cases in sorted(HIT.items()):
        print("  %-18s tile %4d  %s" % (ROUTE[k], t, ", ".join(sorted(cases))))
    missing = sorted(REQUIRED - set(HIT))
    assert not missing, [(ROUTE[k], t) for k, t in missing]
    assert (LAY_TC5, 0) in HIT or (LAY_MMA, 0) in HIT
