"""CPU: canon_conv, the bit-exact model of the canonical fp32 order of the context conv, against float64 (an error
bound that one dropped or duplicated tap breaks), against the exact closed form of the probe networks (bit for bit),
and against the oracle; and proof that it tells the canonical order apart from nearby orders on the test data, so the
GPU tests that compare kernels with it bit for bit (test_gpu_canonical_conv.py) can see an order change."""
import numpy as np
import pytest

import canon_conv as cc
import probe_nets as pn
from oracle import oracle as O
from util import rel_err, rng, synthetic_latent

# (N, G, cin_g, cout_g, H, W, constrain, act, resid, nsets)
FORMS = [
    (2, 6, 1, 4, 9, 13, 5, True, False, 1),      # first layer: P and R only
    (1, 6, 4, 4, 9, 13, 6, True, False, 1),      # hidden: P, R, Q
    (1, 6, 4, 3, 7, 10, 6, False, False, 1),     # last: no PReLU, padded output chunk
    (3, 5, 4, 4, 8, 11, 6, True, True, 3),       # residual, three parameter sets
    (6, 4, 4, 4, 6, 9, 6, True, True, 3),        # two images per parameter set
    (1, 1, 24, 24, 8, 16, 6, True, False, 1),    # one group: 2 P blocks, 2 R / Q blocks, a 4-channel chunk tail
    (1, 2, 18, 5, 6, 7, 6, False, True, 1),      # 2-channel chunk tail, 16/2 block split of the group
]


def _form(form, seed):
    N, G, cin_g, cout_g, H, W, constrain, act, resid, nsets = form
    r = rng(seed)
    x = cc.dynamic_input(r, (N, G * cin_g, H, W))
    w, b, a = cc.layer_params(r, nsets, G, G * cin_g, G * cout_g, constrain)
    res = cc.dynamic_input(r, (N, G * cout_g, H, W)) if resid else None
    return x, w, b, (a if act else None), res, G, constrain, nsets


def _violations(got, ref, E):
    return int((np.abs(np.asarray(got, np.float64) - ref) > E).sum())


@pytest.mark.parametrize("form", FORMS)
def test_model_within_float64_bound(form):
    x, w, b, a, res, G, constrain, nsets = _form(form, 1)
    got = cc.layer(x, w, b, a, G, constrain, nsets, res)
    assert np.isfinite(got).all()
    S, A, nops = cc.exact64(x, w, b, G, constrain, nsets)
    ref, E = cc.error_bound(S, A, nops, a, res, nsets)
    assert _violations(got, ref, E) == 0


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("factor", [0.0, 2.0], ids=["dropped", "duplicated"])
def test_bound_catches_one_dropped_or_duplicated_tap(form, factor):
    """the bound is tight enough to see one term: the model run with one kept tap removed (factor 0) or counted twice
    (factor 2) breaks it somewhere"""
    x, w, b, a, res, G, constrain, nsets = _form(form, 1)
    S, A, nops = cc.exact64(x, w, b, G, constrain, nsets)
    ref, E = cc.error_bound(S, A, nops, a, res, nsets)
    Cout, Cin = w.shape[-4:-2]
    keep = cc.allowed(Cout, Cin, G, constrain)
    o = Cout - 1
    for ci, kh, kw in [(Cin - 1, 2, 1), (0, 2, 2), (Cin // 2, 1, 2)]:  # an R / Q tap, a P tap, one in between
        if not keep[o, ci, kh, kw]:
            continue
        wm = w.copy()
        wm[..., o, ci, kh, kw] *= factor
        got = cc.layer(x, wm, b, a, G, constrain, nsets, res)
        assert _violations(got[:, o], ref[:, o], E[:, o]) > 0, (ci, kh, kw)


@pytest.mark.parametrize("shape", [(8, 16), (10, 14)])
@pytest.mark.parametrize("name", pn.PROBES)
def test_model_equals_probe_closed_form(name, shape):
    """bit for bit on the probe networks, whose fp32 arithmetic is exact in any order (probe_nets.closed_form)"""
    H, W = shape
    params = pn.probe_params(name)
    q, mask, lv = synthetic_latent(7 + H, H=H, W=W)
    y_code, y_imp = pn.closed_form(params, q, mask, lv)
    got_code = cc.net(params["code"], pn.code_input(q, mask), pn.G, 3)
    got_imp = cc.net(params["imp"], pn.imp_input(lv)[None], 1, 1)[0]
    assert np.array_equal(got_code.view(np.int32), y_code.view(np.int32))
    assert np.array_equal(got_imp.view(np.int32), y_imp.view(np.int32))


# the conv op cases of op_cases.py: (N, G, cin_g, cout_g, H, W, constrain, act, nsets)
OP_CASES = [
    (2, 6, 1, 4, 9, 13, 5, True, 1), (1, 6, 4, 4, 9, 13, 6, True, 1), (1, 6, 4, 3, 7, 10, 6, False, 1),
    (3, 5, 1, 4, 8, 33, 5, True, 3), (6, 12, 4, 4, 10, 12, 6, True, 3), (3, 5, 4, 3, 8, 9, 6, False, 3),
    (1, 1, 1, 24, 8, 16, 5, True, 1), (1, 1, 24, 24, 8, 16, 6, True, 1), (1, 1, 24, 9, 8, 16, 6, False, 1),
    (3, 48, 4, 4, 6, 8, 6, True, 3), (3, 48, 1, 4, 64, 128, 5, True, 3), (3, 48, 4, 4, 64, 128, 6, True, 3),
    (3, 48, 4, 3, 64, 128, 6, False, 3), (1, 1, 1, 144, 32, 64, 5, True, 1), (1, 1, 144, 144, 32, 64, 6, True, 1),
    (1, 1, 144, 49, 32, 64, 6, False, 1),
]


@pytest.mark.parametrize("case", OP_CASES)
def test_model_against_oracle(case):
    N, G, cin_g, cout_g, H, W, constrain, act, nsets = case
    r = rng(300 + H + G + cin_g)
    x = r.standard_normal((N, G * cin_g, H, W)).astype(np.float32)
    w, b, a = cc.layer_params(r, nsets, G, G * cin_g, G * cout_g, constrain)
    a = a if act else None
    want = O.cconv_ec(x, np.nan_to_num(w, nan=0.0), b, a, G, constrain, nsets)  # the oracle multiplies masked taps by 0
    got = cc.layer(x, w, b, a, G, constrain, nsets)
    assert rel_err(got, want) <= 1e-6


# least fraction of outputs in which each nearby order gives other bits than the canonical one, on dynamic-range data;
# measured (fp32 of the exact sum / flat chain / (P+Q)+R): 0.79/0.90/0.28, 0.89/0.95/0.26, 0.82/0.88/0.31, 0.85/0.84/0,
# 0.83/0.95/0.29
TEETH = [(1, 24, 24, 6, 0.5, 0.5, 0.15), (48, 4, 4, 6, 0.5, 0.5, 0.15), (6, 4, 4, 6, 0.5, 0.5, 0.15),
         (48, 1, 4, 5, 0.5, 0.5, 0.0), (1, 144, 49, 6, 0.5, 0.5, 0.15)]


@pytest.mark.parametrize("G,cin_g,cout_g,constrain,f_f64,f_flat,f_pqr", TEETH)
def test_model_tells_orders_apart(G, cin_g, cout_g, constrain, f_f64, f_flat, f_pqr):
    """The model differs, in at least the stated fraction of outputs, from the fp32 rounding of the exact sum, from one
    flat fmaf chain without blocks and from ((P + Q) + R): a kernel that used one of those orders could not pass the
    bitwise GPU checks.  (Constrain 5 has no Q terms: there the last order is the canonical one.)"""
    r = rng(11 + G)
    N, H, W = 2, 12, 20
    x = cc.dynamic_input(r, (N, G * cin_g, H, W))
    w, b, a = cc.layer_params(r, 1, G, G * cin_g, G * cout_g, constrain)
    got = cc.layer(x, w, b, None, G, constrain).view(np.int32)
    S, _, _ = cc.exact64(x, w, b, G, constrain)
    frac = lambda y: float((np.asarray(y, np.float32).view(np.int32) != got).mean())
    fr = frac(S.astype(np.float32)), frac(cc.layer(x, w, b, None, G, constrain, variant=cc.FLAT_CHAIN)), \
        frac(cc.layer(x, w, b, None, G, constrain, variant=cc.PQR))
    assert fr[0] >= f_f64 and fr[1] >= f_flat and fr[2] >= f_pqr, fr
    if constrain == 5:
        assert fr[2] == 0.0


@pytest.mark.parametrize("G,cin_g,cout_g,constrain", [(48, 4, 4, 6), (48, 1, 4, 5), (1, 144, 49, 6), (5, 4, 3, 6)])
def test_forbidden_taps_are_never_read(G, cin_g, cout_g, constrain):
    r = rng(5)
    x = cc.dynamic_input(r, (1, G * cin_g, 9, 11))
    w, b, a = cc.layer_params(r, 1, G, G * cin_g, G * cout_g, constrain)
    assert np.isnan(w).sum() > 0
    assert np.isfinite(cc.layer(x, w, b, a, G, constrain)).all()
