"""GPU: every context-conv kernel against canon_conv, the CPU model of the canonical fp32 order (header of
csrc/conv.cu), bit for bit.  The per-op encoder (CconvEc: P pass with and without tile pairing, the rq_tile / rq<4> /
rq<0> / rqb R-Q passes) and decoder (CconvDc) at shapes chosen from the launchers' dispatch conditions, the 12-layer
stacks, and the product codec (FusedCodec, whose fused decoder kernels are seen through its streams) at random
weights, with the expected bytes built from the model's network outputs.  Then the tensor-core switch: within a
float64 bound per op, and never used by the codec."""
import ctypes
import functools
import os

import numpy as np
import pytest
import torch

import canon_conv as cc
import probe_nets as pn
from util import n, rng, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _assert_bits(got, want, what):
    """int32-view equality; on failure the count and the first differing (n, o, h, w) with both values"""
    got, want = np.ascontiguousarray(got, np.float32), np.ascontiguousarray(want, np.float32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = got.view(np.int32) != want.view(np.int32)
    if bad.any():
        i = tuple(int(v) for v in np.argwhere(bad)[0])
        pytest.fail("%s: %d of %d outputs differ from the canonical order; first (n,o,h,w)=%s: kernel %r (0x%08x), "
                    "model %r (0x%08x)" % (what, int(bad.sum()), bad.size, i, float(got[i]), got.view(np.uint32)[i],
                                           float(want[i]), want.view(np.uint32)[i]))


# ---- per-op layers --------------------------------------------------------------------------------------------------
# name: (N, nsets, G, cin_g, cout_g, H, W, constrain, act, options); options: "resid" (EC residual through
# lic360_cconv_ec_forward), "misaligned" (x at a 4-byte, not 16-byte, offset), "nodc" (EC only)
CASES = {
    "g48_first_24x72": (3, 3, 48, 1, 4, 24, 72, 5, True, ""),              # P over 3 blocks of Cin, rq<0>, no pairing
    "g48_hidden_64x128": (3, 3, 48, 4, 4, 64, 128, 6, True, "resid"),      # tile pairing, rq_tile
    "g48_last_64x128": (3, 3, 48, 4, 3, 64, 128, 6, False, ""),            # padded output channel (cout_g 3)
    "g40_hidden_64x128": (3, 3, 40, 4, 4, 64, 128, 6, True, ""),           # pairing with an odd y-tile count
    "g48_hidden_20x42": (3, 3, 48, 4, 4, 20, 42, 6, True, ""),             # W % 4 != 0: rq<4>
    "g48_hidden_misaligned": (3, 3, 48, 4, 4, 64, 128, 6, True, "misaligned nodc"),  # unaligned x: rq<4>
    "g10_hidden_13x36": (1, 1, 10, 4, 4, 13, 36, 6, True, ""),             # partial RQ4_G tile, partial h / w tiles
    "g9_hidden_13x36": (1, 1, 9, 4, 4, 13, 36, 6, True, ""),               # odd group pair
    "imp_first_32x64": (1, 1, 1, 1, 144, 32, 64, 5, True, ""),             # Cin = 1 stage
    "imp_hidden_32x64": (1, 1, 1, 144, 144, 32, 64, 6, True, ""),          # rqb, nqb = 9
    "imp_last_32x64": (1, 1, 1, 144, 49, 32, 64, 6, False, ""),            # cout_g 49
    "cin6_11x19": (2, 1, 2, 6, 5, 11, 19, 6, True, ""),                    # rq<0> 2-channel chunk tail
    "cin16_11x19": (1, 1, 3, 16, 4, 11, 19, 6, True, ""),                  # exactly one block per group
    "cin17_11x19": (1, 1, 2, 17, 3, 11, 19, 6, False, ""),                 # 16/1 block boundary, rqb scalar tail
    "cin18_11x19": (1, 1, 2, 18, 4, 11, 19, 6, True, ""),                  # rqb 2-channel tail
    "cin160_9x13": (1, 1, 1, 160, 8, 9, 13, 6, True, ""),                  # the largest group rqb and DC accept
    "per2_g6_9x13": (6, 3, 6, 4, 4, 9, 13, 6, True, ""),                   # two images per parameter set
    "g6_1x7": (1, 1, 6, 4, 4, 1, 7, 6, True, ""),                          # degenerate frames
    "g6_5x1": (1, 1, 6, 4, 4, 5, 1, 6, True, ""),
    "g48_hidden_40x72": (3, 3, 48, 4, 4, 40, 72, 6, True, ""),             # DC: multi-part diagonals
}


@functools.lru_cache(maxsize=None)
def _layer_case(name):
    N, nsets, G, cin_g, cout_g, H, W, constrain, act, opts = CASES[name]
    r = rng(sum(map(ord, name)))
    x = cc.dynamic_input(r, (N, G * cin_g, H, W))
    w, b, a = cc.layer_params(r, nsets, G, G * cin_g, G * cout_g, constrain)
    if nsets == 1:
        w, b, a = w[0], b[0], a[0]
    a = a if act else None
    res = cc.dynamic_input(r, (N, G * cout_g, H, W)) if "resid" in opts else None
    want = cc.layer(x, w, b, a, G, constrain, nsets, res)
    return x, w, b, a, res, want


def _call(op, x, w, b, a, nsets):
    sfx = "_batch" if nsets > 1 else ""
    if a is not None:
        return getattr(op, "forward_act" + sfx)(x, w, b, a)[0]
    return getattr(op, "forward" + sfx)(x, w, b)[0]


def _device_x(x, misaligned):
    if not misaligned:
        return t(x, DEV)
    buf = torch.empty(x.size + 1, dtype=torch.float32, device=DEV)  # 4 bytes past a 16-byte boundary
    xm = buf[1:].view(x.shape)
    xm.copy_(t(x, DEV))
    assert xm.is_contiguous() and xm.data_ptr() % 16 == 4
    return xm


def _run_ec(name):
    import lic360
    from lic360._lib import LIB, check, cstream
    N, nsets, G, cin_g, cout_g, H, W, constrain, act, opts = CASES[name]
    x, w, b, a, res, _ = _layer_case(name)
    xd, wd, bd = _device_x(x, "misaligned" in opts), t(w, DEV), t(b, DEV)
    ad = None if a is None else t(a, DEV)
    op = lic360.CconvEcOp(G * cin_g, G, G * cout_g, 5, constrain, 0, False)
    if res is None:
        return n(_call(op, xd, wd, bd, ad, nsets))
    wp, wq = op._pack(wd, nsets)
    rd = t(res, DEV)
    out = torch.empty((N, G * cout_g, H, W), dtype=torch.float32, device=DEV)
    p = lambda v: ctypes.c_void_p(v.data_ptr())
    check(LIB.lic360_cconv_ec_forward(p(xd), p(wp), p(wq), p(bd), None if ad is None else p(ad), p(rd), p(out), N,
                                      G * cin_g, H, W, G * cout_g, G, constrain, nsets, cstream(xd)))
    return n(out)


def _run_dc(name):
    import lic360
    import lic360_codec_ops as ops
    N, nsets, G, cin_g, cout_g, H, W, constrain, act, opts = CASES[name]
    x, w, b, a, _, _ = _layer_case(name)
    xd, wd, bd = t(x, DEV), t(w, DEV), t(b, DEV)
    ad = None if a is None else t(a, DEV)
    op = lic360.CconvDcOp(G * cin_g, G, G * cout_g, 5, constrain, 0, False)
    ops._plan(lic360, torch.zeros((1, 1, H, W), device=DEV), 0, [op])
    out = None
    for _ in range(H + W + G - 2):
        out = _call(op, xd, wd, bd, ad, nsets)
    return n(out)


@pytest.mark.parametrize("name", list(CASES))
def test_cconv_ec_is_canonical(name):
    _assert_bits(_run_ec(name), _layer_case(name)[-1], "CconvEc " + name)


@pytest.mark.parametrize("name", [k for k, v in CASES.items() if "nodc" not in v[-1] and "resid" not in v[-1]])
def test_cconv_dc_is_canonical(name):
    _assert_bits(_run_dc(name), _layer_case(name)[-1], "CconvDc " + name)


def test_dc_residual_case_without_residual_is_canonical():
    """the residual row's layer through the decoder (whose per-op form has no residual input)"""
    x, w, b, a, res, want = _layer_case("g48_hidden_64x128")
    _assert_bits(_run_dc("g48_hidden_64x128"), cc.layer(x, w, b, a, 48, 6, 3), "CconvDc g48_hidden_64x128")


@pytest.mark.parametrize("cin", [161, 200])
def test_group_too_wide_is_an_error_from_both_ops(cin):
    """cin_g > 160 is beyond the encoder's block-parallel R / Q kernel and the decoder's 32 warps: both refuse"""
    import lic360
    import lic360_codec_ops as ops
    r = rng(cin)
    x = t(cc.dynamic_input(r, (1, cin, 9, 13)), DEV)
    w, b, a = (t(v[0], DEV) for v in cc.layer_params(r, 1, 1, cin, 8, 6))
    with pytest.raises(RuntimeError):
        lic360.CconvEcOp(cin, 1, 8, 5, 6, 0, False).forward_act(x, w, b, a)
    op = lic360.CconvDcOp(cin, 1, 8, 5, 6, 0, False)
    ops._plan(lic360, torch.zeros((1, 1, 9, 13), device=DEV), 0, [op])
    with pytest.raises(RuntimeError):
        op.forward_act(x, w, b, a)
    torch.cuda.synchronize()  # nothing asynchronous went wrong either


# ---- 12-layer stacks ------------------------------------------------------------------------------------------------
def _random_biases(params, seed, scale=0.1):
    """make_entropy_params leaves the biases at zero (but the delta net's 2): add random ones, in place"""
    r = rng(seed)
    for k, v in params.items():
        if k.endswith(".bias"):
            v += t((r.standard_normal(tuple(v.shape)) * scale).astype(np.float32), v.device)
    return params


def _np(params):
    return {k: n(v) for k, v in params.items()}


@pytest.mark.parametrize("geom,H,W", [((48, 4, 3, 3), 40, 72), ((1, 144, 49, None), 32, 64)], ids=["code", "imp"])
def test_twelve_layer_stacks_are_canonical(geom, H, W):
    import lic360
    import lic360_codec_ops as ops
    ngroup, cpg, nlast, batch = geom
    params = _random_biases(ops.make_entropy_params(ngroup, cpg, nlast, batch, 77, DEV), 78)
    q, mask, lv = synthetic_latent(79, H=H if batch else 2 * H, W=W if batch else 2 * W)
    x = pn.code_input(q, mask) if batch else pn.imp_input(lv)[None]
    want = cc.net(_np(params), x, ngroup, batch or 1)
    ec = ops._Net(lic360, params, ngroup, cpg, nlast, batch, False, 0)
    dc = ops._Net(lic360, params, ngroup, cpg, nlast, batch, True, 0)
    ops._plan(lic360, torch.zeros((1, 1, H, W), device=DEV), 0, dc.stateful())
    xd = t(x, DEV)
    _assert_bits(n(ec(xd)), want, "EC net")
    y = None
    for _ in range(H + W + ngroup - 2):
        y = dc(xd)
    _assert_bits(n(y), want, "DC net")


# ---- the product codec at random weights -----------------------------------------------------------------------------
CODEC_SHAPES = [(8, 16), (34, 66), (64, 128), (128, 256)]


@functools.lru_cache(maxsize=None)
def _codec_case(H, W):
    """(torch params, latent, expected streams): the per-op encoders' table ops and coder, fed the model's network
    outputs instead of running the networks"""
    import tempfile

    import lic360
    import lic360_codec_ops as ops
    import lic360_pipeline as pl
    seed = 500 + H
    params = pl.make_codec_params(DEV, seed=seed)
    _random_biases(params["code"], seed + 1)
    _random_biases(params["imp"], seed + 2)
    q, mask, lv = synthetic_latent(seed, H=H, W=W)
    y_code = t(cc.net(_np(params["code"]), pn.code_input(q, mask), 48, 3), DEV)
    y_imp = t(cc.net(_np(params["imp"]), pn.imp_input(lv)[None], 1, 1), DEV)
    d = tempfile.mkdtemp(prefix="lic360_canon_")
    enc_i = ops.ImpEntEncoder(lic360, params["imp"])
    enc_i.net = lambda _: y_imp.clone()
    enc_i.encode(t(lv, DEV), os.path.join(d, "imp"))
    enc_c = ops.EntEncoder(lic360, params["code"])
    enc_c.net = lambda _: y_code.clone()
    enc_c.encode(t(q, DEV), t(mask, DEV), os.path.join(d, "code"))
    streams = []
    for f in ("imp", "code"):
        with open(os.path.join(d, f), "rb") as fh:
            streams.append(fh.read())
        os.remove(os.path.join(d, f))
    os.rmdir(d)
    return params, (q, mask, lv), tuple(streams)


def _decode_ok(codec, streams, q, mask):
    code, mup = codec.decode(*streams)
    return np.array_equal(n(mup), mask) and np.array_equal(n(code), q * mask)


@pytest.mark.parametrize("H,W", CODEC_SHAPES)
def test_fused_codec_writes_the_canonical_streams(H, W):
    """FusedCodec (whole-frame encoder nets, fused wavefront decoder) against the specification, not against itself"""
    import lic360
    import lic360_pipeline as pl
    params, (q, mask, lv), want = _codec_case(H, W)
    fused = pl.FusedCodec(params, H=H, W=W)
    got = fused.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
    assert got[0] == want[0], "importance stream differs (%d vs %d bytes)" % (len(got[0]), len(want[0]))
    assert got[1] == want[1], "code stream differs (%d vs %d bytes)" % (len(got[1]), len(want[1]))
    assert _decode_ok(fused, want, q, mask), "mode 0 decode"
    fused.set_mode(2)
    assert _decode_ok(fused, want, q, mask), "mode 2 decode"
    if H * W <= 8 * 16:
        code, mup = pl.PerOpCodec(lic360, params).decode(*want, H // 2, W // 2)
        assert np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask), "per-op decode"


# ---- the tensor-core switch -----------------------------------------------------------------------------------------
def _mma_gamma(w, G, constrain):
    """Error model of the LIC360_EC_MMA=1 old-term pass (csrc/conv_mma.cu), per output channel.
    Split: v_hi = v truncated to 11 significant bits, so |v - v_hi| < 2^-10 |v|; v_lo = (v - v_hi) truncated, so
    |v - v_hi - v_lo| < 2^-20 |v| and |v_lo| < 2^-10 |v|.  The three products x_lo w_hi + x_hi w_lo + x_hi w_hi miss
    x_lo w_lo and the two truncation remainders: < (2^-20 + 2^-20 + 2^-20 (1 + 2^-10)) |x w| < 3.01 * 2^-20 |x w|.
    Accumulation: the tensor core multiplies tf32 exactly and adds with truncation (round toward zero, unit 2^-23);
    counting two truncations per split product (its alignment in the MMA and the accumulator's normalisation), k kept
    P taps give at most 6k roundings of unit 2^-23, on addends of total magnitude <= (1 + 2^-9) sum |x w|.  The block
    folds, the R / Q chains and the epilogue are the fp32 ones of the canonical order (covered by the same count)."""
    Cout, Cin = w.shape[-4:-2]
    k = cc.allowed(Cout, Cin, G, constrain).reshape(Cout, -1).sum(1)
    nops = 6 * k + (Cin + 15) // 16 + 2 * ((Cin // G + 15) // 16) + 8
    return cc.gamma(nops, 2.0 ** -23) * (1 + 2.0 ** -9) + 3.01 * 2.0 ** -20


@pytest.mark.parametrize("name", ["g48_hidden_40x72", "imp_hidden_32x64", "cin17_11x19"])
def test_tensor_core_pass_within_float64_bound(monkeypatch, name):
    """LIC360_EC_MMA=1 (per-op CconvEc only): within the bound of _mma_gamma of float64; the same bound against a
    reference with one old-term product dropped fails, so the bound can see one missing product"""
    N, nsets, G, cin_g, cout_g, H, W, constrain, act, opts = CASES[name]
    x, w, b, a, res, want = _layer_case(name)
    monkeypatch.setenv("LIC360_EC_MMA", "1")
    got = _run_ec(name)
    assert np.isfinite(got).all()
    cg = _mma_gamma(w, G, constrain)
    S, A, nops = cc.exact64(x, w, b, G, constrain, nsets)
    ref, E = cc.error_bound(S, A, nops, a, None, nsets, conv_gamma=cg)
    assert (np.abs(got - ref) <= E).all(), "%d outputs outside the bound" % int((np.abs(got - ref) > E).sum())
    # an old term (wavefront <= p-2) of the last output channel: input group 0 at the tap (0, 0)
    Cout = G * cout_g
    wd = w.copy()
    wd[..., Cout - 1, 0, 0, 0] = 0
    S, A, nops = cc.exact64(x, wd, b, G, constrain, nsets)
    ref, E = cc.error_bound(S, A, nops, a, None, nsets, conv_gamma=cg)
    assert (np.abs(got[:, Cout - 1] - ref[:, Cout - 1]) > E[:, Cout - 1]).any(), "the bound does not see one product"


def test_fused_codec_ignores_the_tensor_core_switch(monkeypatch):
    """LIC360_EC_MMA=1 is a per-op measurement switch: the codec's encoder nets keep the canonical P pass, so the streams
    are the ones its decoder reproduces"""
    import lic360_pipeline as pl
    H, W = 64, 128
    params, (q, mask, lv), want = _codec_case(H, W)
    monkeypatch.setenv("LIC360_EC_MMA", "1")
    fused = pl.FusedCodec(params, H=H, W=W)
    got = fused.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
    assert got == want, "streams differ with LIC360_EC_MMA=1 (%d/%d vs %d/%d bytes)" % (
        len(got[0]), len(got[1]), len(want[0]), len(want[1]))
