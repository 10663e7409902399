"""GPU: the codec's rate estimate (FusedCodec.estimate, lic360_codec_estimate) against the float64 bits of the tables the coder
uses -- exact ones from the probe networks, and the per-op path's at random weights --, against the bytes encode writes (the
bound derived in test_rate_estimate.py), and its determinism, its independence from the codec's other state, and its errors."""
import functools
import math

import numpy as np
import pytest
import torch

import probe_nets as pn
from test_gpu_probe_codec import SHAPES
from test_rate_estimate import assert_within_bound, bits_from_tables
from util import n, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RANDOM_SHAPES = [(8, 16), (10, 14), (6, 130), (64, 128)]


def _maps(bits_code, bits_imp, H, W):
    """per-symbol bits in coding order -> (1,48,H,W) and (1,1,H/2,W/2) maps"""
    code = np.zeros((1, pn.G, H, W))
    c, h, w = pn.coding_order(H, W, pn.G).T
    code[0, c, h, w] = bits_code
    imp = np.zeros((1, 1, H // 2, W // 2))
    _, h, w = pn.coding_order(H // 2, W // 2, 1).T
    imp[0, 0, h, w] = bits_imp
    return code, imp


def _assert_estimate(est, Tc, lab_c, msk, Ti, lab_i, mask, H, W):
    bc, bi = bits_from_tables(Tc, lab_c, msk), bits_from_tables(Ti, lab_i)
    for key, total, want in zip(("code", "imp"), (bc, bi), _maps(bc, bi, H, W)):
        got = n(est[key + "_map"])
        assert got.dtype == np.float32 and got.shape == want.shape, key
        w32 = want.astype(np.float32)
        bad = np.argwhere(np.abs(got.astype(np.float64) - w32) > np.spacing(np.abs(w32)))
        assert len(bad) == 0, "%s map: %d entries off by more than 1 ulp, first %s: %r vs %r" % (
            key, len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])
        ref = math.fsum(total)
        assert abs(est[key + "_bits"] - ref) <= 1e-9 * ref, "%s total %.9f vs %.9f" % (key, est[key + "_bits"], ref)
    assert (n(est["code_map"])[mask < 0.5] == 0).all(), "a masked code symbol has a cost"


def _assert_streams_within_bound(est, streams, mask):
    assert_within_bound(len(streams[0]), est["imp_bits"], est["imp_map"].numel(), "importance stream")
    assert_within_bound(len(streams[1]), est["code_bits"], int((mask >= 0.5).sum()), "code stream")


@functools.lru_cache(maxsize=None)
def _probe_case(name, H, W):
    params = pn.probe_params(name)
    q, mask, lv = synthetic_latent(400 + H + W, H=H, W=W)
    return (q, mask, lv), pn.expected_tables(params, q, mask, lv)


@pytest.mark.parametrize("H,W", [s for s in SHAPES if s[0] * s[1] <= 64 * 128])
@pytest.mark.parametrize("name", pn.PROBES)
def test_probe_networks_exact_bits(name, H, W):
    """exact tables: every entry of both maps within 1 ulp of the float64 bits, both totals to 1e-9, and encode's streams within
    the bound of the totals"""
    import lic360_pipeline as pl
    (q, mask, lv), tables = _probe_case(name, H, W)
    codec = pl.FusedCodec(pn.to_torch(pn.probe_params(name), DEV), H=H, W=W)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    est = codec.estimate(tq, tm, tl)
    _assert_estimate(est, *tables, mask, H, W)
    _assert_streams_within_bound(est, codec.encode(tq, tm, tl), mask)


def _per_op_tables(params, tq, tm, tl):
    """(code tables, labels, mask, importance tables, labels) in coding order from the per-op path: the whole-frame networks,
    then per wavefront step TileExtract + EntropyGmmTable / EntropyTable, what lic360_codec_ops.EntEncoder / ImpEntEncoder hand
    to the coder"""
    import lic360
    import lic360_codec_ops as ops
    H, W = tq.shape[2:]
    enc = ops.EntEncoder(lic360, params["code"])
    ctx = ops._plan(lic360, tq, 0, [enc.ext, enc.ext_label, enc.ext_mask])
    x = ((tq - enc.bias) * tm).contiguous()
    y = enc.net(torch.cat([x, x, x], dim=0).contiguous())
    tc, lc, mc = [], [], []
    for _ in range(H + W + pn.G - 2):
        z, le = enc.ext.forward_batch(y)
        vec = enc.gmm.forward_batch(z, le)[0]
        ln = int(le[0].item())
        tc.append(n(vec).reshape(-1, 9)[:ln])
        lc.append(n(enc.ext_label.forward(tq)[0]).reshape(-1)[:ln])
        mc.append(n(enc.ext_mask.forward(tm)[0]).reshape(-1)[:ln])
    ienc = ops.ImpEntEncoder(lic360, params["imp"])
    ictx = ops._plan(lic360, tl, 0, [ienc.ext, ienc.ext_label])
    y = ienc.net(ienc.scale.forward(tl)[0])
    ti, li = [], []
    for _ in range(H // 2 + W // 2 - 1):
        z, le = ienc.ext.forward(y)
        vec = ienc.table.forward(z, le)[0]
        ln = int(le[0].item())
        ti.append(n(vec).reshape(-1, 50)[:ln])
        li.append(n(ienc.ext_label.forward(tl)[0]).reshape(-1)[:ln])
    del ctx, ictx
    cat = np.concatenate
    return cat(tc).astype(np.int32), cat(lc).astype(np.int32), cat(mc), cat(ti).astype(np.int32), cat(li).astype(np.int32)


@pytest.mark.parametrize("H,W", RANDOM_SHAPES)
def test_random_weights_match_the_per_op_tables(H, W):
    """network arithmetic that is not exact: the estimate costs the tables the per-op path (and so the coder) uses"""
    import lic360_pipeline as pl
    params = pl.make_codec_params(DEV, seed=600 + H)
    q, mask, lv = synthetic_latent(601 + W, H=H, W=W)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    tables = _per_op_tables(params, tq, tm, tl)
    c, h, w = pn.coding_order(H, W, pn.G).T
    assert np.array_equal(tables[1], q[0, c, h, w]) and np.array_equal(tables[2], mask[0, c, h, w])
    codec = pl.FusedCodec(params, H=H, W=W)
    est = codec.estimate(tq, tm, tl)
    _assert_estimate(est, *tables, mask, H, W)
    _assert_streams_within_bound(est, codec.encode(tq, tm, tl), mask)


@pytest.mark.parametrize("kind", ["random"] + list(pn.PROBES))
def test_streams_within_bound_at_128x256(kind):
    import lic360_pipeline as pl
    H, W = 128, 256
    params = pl.make_codec_params(DEV, seed=700) if kind == "random" else pn.to_torch(pn.probe_params(kind), DEV)
    q, mask, lv = synthetic_latent(701, H=H, W=W)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    codec = pl.FusedCodec(params, H=H, W=W)
    est = codec.estimate(tq, tm, tl)
    assert est["code_bits"] > 1e5 and est["imp_bits"] > 1e3
    _assert_streams_within_bound(est, codec.encode(tq, tm, tl), mask)


def _same(a, b):
    return (a["code_bits"] == b["code_bits"] and a["imp_bits"] == b["imp_bits"] and torch.equal(a["code_map"], b["code_map"])
            and torch.equal(a["imp_map"], b["imp_map"]))


def test_estimate_is_deterministic_and_leaves_the_codec_alone():
    import lic360_pipeline as pl
    H, W = 24, 72
    params = pl.make_codec_params(DEV, seed=800)
    q, mask, lv = synthetic_latent(801, H=H, W=W)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    want = pl.FusedCodec(params, H=H, W=W).encode(tq, tm, tl)
    codec = pl.FusedCodec(params, H=H, W=W)
    e1 = codec.estimate(tq, tm, tl)
    timing = codec.last_timing()
    assert timing["total_ms"] > 0 and timing["total_ms"] >= timing["gpu_wait_ms"] >= 0
    assert timing["host_coder_ms"] == timing["imp_stream_ms"] == timing["gpu_steps_ms"] == timing["imp_gpu_steps_ms"] == 0
    assert _same(e1, codec.estimate(tq, tm, tl)), "second estimate on the same codec"
    assert _same(e1, pl.FusedCodec(params, H=H, W=W).estimate(tq, tm, tl)), "estimate on a second codec"
    # encode -> estimate -> decode on one codec: the estimate touches nothing the encoder's bytes or the decoder depend on
    got = codec.encode(tq, tm, tl)
    assert got == want
    assert _same(e1, codec.estimate(tq, tm, tl))
    code, mup = codec.decode(*got)
    assert np.array_equal(n(mup), mask) and np.array_equal(n(code), q * mask)
    assert codec.encode(tq, tm, tl) == want
    codec.set_mode(2)
    assert _same(e1, codec.estimate(tq, tm, tl)), "estimate in mode 2"


def _raised(fn, *args):
    try:
        fn(*args)
    except RuntimeError as e:
        return str(e)
    return None


def test_errors_match_encode():
    """the same inputs are refused by estimate and encode, with the same message, and the same inputs pass both"""
    import lic360_pipeline as pl
    H, W = 8, 16
    params = pl.make_codec_params(DEV, seed=900)
    q, mask, lv = synthetic_latent(901, H=H, W=W)
    codec = pl.FusedCodec(params, H=H, W=W)
    kept, skipped = tuple(np.argwhere(mask[0] > 0.5)[5]), tuple(np.argwhere(mask[0] < 0.5)[5])

    def both(qq, ll):
        return _raised(codec.estimate, t(qq, DEV), t(mask, DEV), t(ll, DEV)), _raised(codec.encode, t(qq, DEV), t(mask, DEV), t(ll, DEV))

    for where, value, refused in ((kept, 8.0, True), (kept, -0.5, True), (kept, np.nan, True), (kept, 7.9, False),
                                  (skipped, 8.0, False), (skipped, -3.0, False)):
        qq = q.copy()
        qq[0][where] = value
        est, enc = both(qq, lv)
        assert est == enc, (where, value)
        assert (est is not None) == refused, (where, value, est)
        if refused:
            assert "coder: symbol out of range" in est
    for value, refused in ((49.0, True), (-1.0, True), (48.9, False)):
        ll = lv.copy()
        ll[0, 0, 1, 2] = value
        est, enc = both(q, ll)
        assert est == enc, value
        assert (est is not None) == refused, (value, est)
        if refused:
            assert "importance level" in est
    # a symbol on a skipped position costs nothing
    qq = q.copy()
    qq[0][skipped] = 8.0
    assert n(codec.estimate(t(qq, DEV), t(mask, DEV), t(lv, DEV))["code_map"])[0][skipped] == 0
    # wrong shape, dtype or device
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    for args in ((tq[..., :-2], tm, tl), (tq, tm.double(), tl), (tq, tm, tl.cpu()), (tq, tm, tl[..., :-1])):
        with pytest.raises(RuntimeError):
            codec.estimate(*args)
    assert codec.estimate(tq, tm, tl)["code_bits"] > 0
