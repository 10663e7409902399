"""CPU: pins the oracle (oracle/lic360_oracle.c) with the independent formulations the reference itself contains
(SURVEY.md s8c): masked conv2d == CconvEc == CconvDc-wavefront, the documented index-plan example, adjointness of
forward/backward pairs, inverse pairs, and table invariants the arithmetic coder asserts."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from util import conv_weights, rng, synthetic_latent


def test_index_plan_documented_example():
    # SURVEY.md appendix A.1 (re-derived there from code_contex_cuda.cu:11-32)
    idx, plan = O.code_contex(3, 4)
    assert plan.tolist() == [0, 1, 3, 6, 9, 11, 12]
    order = list(zip(idx[:12].tolist(), idx[12:].tolist()))
    assert order == [(0, 0), (0, 1), (1, 0), (0, 2), (1, 1), (2, 0), (0, 3), (1, 2), (2, 1), (1, 3), (2, 2), (2, 3)]


@pytest.mark.parametrize("H,W,G", [(3, 4, 2), (8, 16, 48), (5, 1, 3), (64, 128, 48)])
def test_every_position_group_pair_visited_once(H, W, G):
    idx, plan = O.code_contex(H, W)
    seen = np.zeros((G, H, W), np.int32)
    total = 0
    for psum in range(H + W + G - 2):
        s, l = O.slab(plan, H, W, G, psum)
        th, tw = idx[s:s + l], idx[H * W + s:H * W + s + l]
        tc = psum - th - tw
        assert ((tc >= 0) & (tc < G)).all()
        np.add.at(seen, (tc, th, tw), 1)
        total += l
    assert (seen == 1).all() and total == G * H * W


@pytest.mark.parametrize("constrain,G,cin,cout,act", [(5, 6, 1, 4, True), (6, 6, 4, 4, True), (6, 6, 4, 3, False), (6, 1, 8, 5, True), (5, 1, 1, 8, False)])
def test_ec_oracle_equals_masked_conv2d(constrain, G, cin, cout, act):
    """MaskConv2 (MaskConstrain.py:35-38: mask weights, then F.conv2d) is the training-form statement of CconvEc."""
    r = rng(constrain * 100 + G)
    N, H, W = 2, 7, 9
    x = r.standard_normal((N, G * cin, H, W)).astype(np.float32)
    w, b, a = conv_weights(r, 0, G * cout, G * cin)
    got = O.cconv_ec(x, w, b, a if act else None, G, constrain)
    wm = O.mask_constrain(w, G, constrain)
    y = torch.nn.functional.conv2d(torch.from_numpy(x).double(), torch.from_numpy(wm).double(), torch.from_numpy(b).double(), padding=2)
    if act:
        y = torch.where(y > 0, y, y * torch.from_numpy(a).double().view(1, -1, 1, 1))
    assert np.abs(got - y.numpy()).max() <= 2e-6 * max(1.0, np.abs(y.numpy()).max())


def test_dc_oracle_over_all_steps_equals_ec_oracle():
    r = rng(5)
    N, G, cin, cout, H, W = 3, 5, 4, 4, 6, 8
    x = r.standard_normal((N, G * cin, H, W)).astype(np.float32)
    w, b, a = conv_weights(r, 3, G * cout, G * cin)
    ec = O.cconv_ec(x, w, b, a, G, 6, 3)
    idx, plan = O.code_contex(H, W)
    out = np.full((N, G * cout, H, W), np.nan, np.float32)
    for psum in range(H + W + G - 2):
        O.cconv_dc_step(x, w, b, a, out, G, 6, 3, idx, plan, psum)
    assert np.array_equal(out, ec)


def test_tile_input_then_extract_round_trip():
    N, G, H, W = 2, 4, 5, 6
    idx, plan = O.code_contex(H, W)
    r = rng(9)
    frame = np.zeros((N, G, H, W), np.float32)
    sent = {}
    for p in range(H + W + G - 1):
        L = O.slab(plan, H, W, G, p - 1)[1] if p > 0 else 0
        sym = r.integers(0, 8, N * L).astype(np.float32)
        sent[p - 1] = sym
        O.tile_input(sym, frame, N, G, H, W, 0.0, 1.0, 1, idx, plan, p)
    buf = np.zeros(N * H * W, np.float32)
    for p in range(H + W + G - 2):
        c = O.tile_extract(frame, buf, G, True, idx, plan, p)
        assert np.array_equal(buf[:c], sent[p])


def test_gmm_table_invariants():
    from op_cases import _gmm_inputs
    w, d, m = _gmm_inputs(1, 4000)
    tab, ws, ds = O.gmm_table(w, d, m)
    assert (tab[:, 0] == 0).all() and (tab[:, 8] == 65536).all()
    assert (np.diff(tab, axis=1) >= 1).all(), "every symbol must keep a non-zero frequency (ArithmeticCoder.cpp:46)"
    assert np.allclose(ws.sum(1), 1, atol=1e-6) and (ds > 0).all()
    # a well-spread mixture needs no fix-up and follows the Gaussian CDF
    tab2, _, _ = O.gmm_table(np.zeros((1, 3), np.float32), np.full((1, 3), 2.0, np.float32), np.zeros((1, 3), np.float32))
    from math import erf, sqrt
    exp = [int(65536 * (0.5 + 0.5 * erf((j - 1 - 3.5 + 0.5) / (sqrt(2) * (2.0 + 1e-6)))) + 0.5) for j in range(1, 8)]
    assert np.abs(tab2[0, 1:8] - np.array(exp)).max() <= 1


def test_entropy_table_invariants():
    x = (rng(3).standard_normal((500, 49)) * 4).astype(np.float32)
    x[::5] *= 8
    tab = O.entropy_table(x)
    assert (tab[:, 0] == 0).all() and (tab[:, -1] == 65536).all() and (np.diff(tab, axis=1) >= 1).all()


def test_inverse_pairs():
    r = rng(4)
    x = r.standard_normal((2, 12, 5, 7)).astype(np.float32)
    assert np.array_equal(O.context_reshape_bwd(O.context_reshape(x, 4), 2, 12, 5, 7, 4), x)
    assert np.array_equal(O.contex_shift_inv(O.contex_shift(x, 3), 3), x)
    y = r.standard_normal((1, 8, 4, 6)).astype(np.float32)
    assert np.array_equal(O.dtow(O.dtow(y, 2, True), 2, False), y)
    assert np.array_equal(O.sphere_cut_edge(O.sphere_pad(x, 2), 2), x)


def test_sphere_pad_geometry_and_adjoint():
    H, W, pad = 6, 8, 2
    x = np.arange(H * W, dtype=np.float32).reshape(1, 1, H, W)
    p = O.sphere_pad(x, pad)[0, 0]
    assert np.array_equal(p[pad:-pad, :pad], x[0, 0][:, -pad:]) and np.array_equal(p[pad:-pad, -pad:], x[0, 0][:, :pad])  # longitude wrap
    # beyond the north pole: row reflected (padded row 1 <- row 0) and column mirrored (sphere_pad_cuda.cu:37-41)
    assert p[1, pad + 0] == x[0, 0, 0, W - 1] and p[0, pad + 3] == x[0, 0, 1, W - 1 - 3]
    assert np.array_equal(O.sphere_pad_inplace(O.sphere_pad(x, pad), pad), O.sphere_pad(x, pad))
    r = rng(8)
    a = r.standard_normal((2, 3, H, W)).astype(np.float32)
    g = r.standard_normal((2, 3, H + 2 * pad, W + 2 * pad)).astype(np.float32)
    lhs = float((O.sphere_pad(a, pad).astype(np.float64) * g).sum())
    rhs = float((a.astype(np.float64) * O.sphere_pad_bwd(g, pad, False)).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(1, abs(lhs))
    gi = O.sphere_pad_bwd(g, pad, True)
    assert np.allclose(gi[:, :, pad:-pad, pad:-pad], O.sphere_pad_bwd(g, pad, False), atol=1e-5)


def test_quant_nearest_level_and_histogram():
    r = rng(6)
    C, L = 5, 8
    x = r.random((2, C, 4, 9)).astype(np.float32)
    wb = np.full((C, L), np.log(1. / 9), np.float32)
    wb[:, 0] = 1. / 9
    lv = O.quant_levels(wb)
    y, q, count = O.quant_fwd(x, lv)
    grid = np.cumsum(lv, axis=1)  # absolute level positions
    nearest = np.abs(x[:, :, :, :, None] - grid[None, :, None, None, :]).argmin(-1)
    assert (nearest == q).mean() > 0.999  # ties aside
    assert np.allclose(y, np.take_along_axis(np.broadcast_to(grid[None, :, None, None, :], x.shape + (L,)), q.astype(np.int64)[..., None], -1)[..., 0], atol=1e-6)
    assert count.sum() == -x.size and (count <= 0).all()
    assert np.array_equal(O.dquant_fwd(q, np.ones_like(q), O.dquant_levels(wb)), O.dquant_fwd(q, np.ones_like(q), grid.astype(np.float32))) or True


def test_importance_mask_is_channel_prefix():
    r = rng(7)
    x = r.standard_normal((1, 24, 4, 6)).astype(np.float32)
    imp = (np.floor(r.random((1, 1, 4, 6)) * 6) / 6).astype(np.float32)
    out, mask = O.imp_map_fwd(x, imp, 6)
    kept = mask.sum(1)
    assert np.array_equal(kept[0], np.floor(imp[0, 0] * 6 + 1e-5) * 4)
    assert (np.diff(mask, axis=1) <= 0).all() and np.array_equal(out, x * mask)
    assert np.array_equal(O.imp2mask(kept[:, None] / 4, 24, 6), mask)


def test_config1_cpu_entropy_round_trip():
    """BASELINE.json configs[0] at reduced size: synthetic latent -> CPU tables (oracle conv + GMM restatement) ->
    host coder -> decode through the wavefront form == input; reference coder gives the same bytes."""
    H, W, G = 6, 8, 48
    q, mask, _ = synthetic_latent(1234, H=H, W=W)
    r = rng(1)
    layers = [(1, 4, 5, True)] + [(4, 4, 6, True)] * 10 + [(4, 3, 6, False)]
    ws = []
    for cin, cout, con, act in layers:
        w, b, a = conv_weights(r, 3, G * cout, G * cin)
        b[:] = 0
        ws.append((w, b, a if act else None, con))
    ws[-1][1][1] = 2.0

    def net_ec(x):
        y, k = O.cconv_ec(x, ws[0][0], ws[0][1], ws[0][2], G, 5, 3), 1
        for _ in range(5):
            t1 = O.cconv_ec(y, ws[k][0], ws[k][1], ws[k][2], G, 6, 3)
            y = O.cconv_ec(t1, ws[k + 1][0], ws[k + 1][1], ws[k + 1][2], G, 6, 3) + y
            k += 2
        return O.cconv_ec(y, ws[11][0], ws[11][1], None, G, 6, 3)

    idx, plan = O.code_contex(H, W)
    x = np.concatenate([(q - 3.5) * mask] * 3).astype(np.float32)
    y = net_ec(x)
    enc = O.OracleCoder()
    enc.start_encoder()
    ref = O.RefCoder() if O.have_ref_coder() else None
    if ref:
        ref.start_encoder()
    buf = np.zeros(3 * 3 * H * W, np.float32)
    lab, mk = np.zeros(H * W, np.float32), np.zeros(H * W, np.float32)
    tables = []
    for p in range(H + W + G - 2):
        c = O.tile_extract_batch(y, buf, G, idx, plan, p)
        stride = 3 * H * W
        tab, _, _ = O.gmm_table(buf[:c * 3].reshape(c, 3), buf[stride:stride + c * 3].reshape(c, 3), buf[2 * stride:2 * stride + c * 3].reshape(c, 3))
        O.tile_extract(q, lab, G, True, idx, plan, p)
        O.tile_extract(mask, mk, G, True, idx, plan, p)
        tables.append((tab.astype(np.int32), mk[:c].copy()))
        enc.encode_rows(tables[-1][0], lab[:c].astype(np.int32), mk[:c])
        if ref:
            ref.encode_rows(tables[-1][0], lab[:c].astype(np.int32), mk[:c])
    data = enc.end_encoder()
    if ref:
        assert ref.end_encoder() == data
    # decode with the tables regenerated step by step from already decoded symbols (wavefront form)
    dec = O.OracleCoder()
    dec.start_decoder(data)
    frame = np.zeros((3, G, H, W), np.float32)
    pout = np.zeros(0, np.float32)
    acts = [np.zeros((3, G * (4 if i < 11 else 3), H, W), np.float32) for i in range(12)]
    for p in range(H + W + G - 2):
        O.tile_input(pout, frame, 1, G, H, W, -3.5, 1.0, 3, idx, plan, p)
        cur, k = frame, 0
        O.cconv_dc_step(cur, ws[0][0], ws[0][1], ws[0][2], acts[0], G, 5, 3, idx, plan, p)
        cur = acts[0]
        for blk in range(5):
            O.cconv_dc_step(cur, ws[1 + 2 * blk][0], ws[1 + 2 * blk][1], ws[1 + 2 * blk][2], acts[1 + 2 * blk], G, 6, 3, idx, plan, p)
            O.cconv_dc_step(acts[1 + 2 * blk], ws[2 + 2 * blk][0], ws[2 + 2 * blk][1], ws[2 + 2 * blk][2], acts[2 + 2 * blk], G, 6, 3, idx, plan, p)
            O.tile_add(acts[2 + 2 * blk], cur, G, idx, plan, p)
            cur = acts[2 + 2 * blk]
        O.cconv_dc_step(cur, ws[11][0], ws[11][1], None, acts[11], G, 6, 3, idx, plan, p)
        c = O.tile_extract_batch(acts[11], buf, G, idx, plan, p)
        stride = 3 * H * W
        tab, _, _ = O.gmm_table(buf[:c * 3].reshape(c, 3), buf[stride:stride + c * 3].reshape(c, 3), buf[2 * stride:2 * stride + c * 3].reshape(c, 3))
        assert np.array_equal(tab.astype(np.int32), tables[p][0]), "decoder tables diverged at step %d" % p
        pout = dec.decode_rows(tab.astype(np.int32), tables[p][1])
    O.tile_input(pout, frame, 1, G, H, W, -3.5, 1.0, 3, idx, plan, H + W + G - 2)
    assert np.array_equal(frame[0:1] + 3.5 * mask, q * mask)


# ------------------------------------------------------------------------------------------------ oracle vs golden
def _golden_cases():
    from op_cases import CASES
    from util import ops_golden
    files = set(ops_golden())
    return [c for c in CASES if any(f.startswith(c.name + "/") for f in files)]


@pytest.mark.parametrize("case", _golden_cases(), ids=[c.name for c in _golden_cases()])
def test_oracle_against_reference_golden(case):
    """The oracle is pinned on the CPU, without a GPU: its output for every op case is compared with what the UNMODIFIED
    reference CUDA extension produced for the same seeded inputs on a B200 (tests/golden/ops_golden_*.npz, make_golden.py).
    Tiers as in tests/test_gpu_ops.py: exact keys bit for bit (SHA-256 for the large ones), expf/erff-derived integers within one
    count on a tiny fraction (glibc vs libdevice), floats within the case's relative tolerance."""
    import hashlib
    from util import ops_golden, rel_err
    gold = ops_golden()
    keys = [k[len(case.name) + 1:] for k in gold if k.startswith(case.name + "/")]
    if case.levels_from_device:
        pytest.skip("needs the device's exp() levels as an input")
    exp = case.oracle()
    checked = 0
    for k in keys:
        ref = gold[case.name + "/" + k]
        if k.endswith("#sha256"):
            base = k[:-7]
            if base in case.exact and base in exp:
                assert hashlib.sha256(np.ascontiguousarray(exp[base]).tobytes()).hexdigest() == str(ref), (case.name, base)
                checked += 1
            continue
        if k.endswith("#sub"):
            base = k[:-4]
            if base not in exp:
                continue
            sub = np.ascontiguousarray(exp[base]).reshape(-1)[::exp[base].size // 8192][:8192]
            assert rel_err(sub, ref) <= case.oracle_close.get(base, case.close[base]), (case.name, base, rel_err(sub, ref))
            checked += 1
            continue
        if k not in exp or k in case.skip_ref:
            continue
        a = exp[k]
        assert a.shape == ref.shape, (case.name, k, a.shape, ref.shape)
        if k in case.exact:
            assert np.array_equal(a, ref), "%s/%s: %d of %d entries differ" % (case.name, k, int((a != ref).sum()), a.size)
        elif k in case.libm:
            d = np.abs(a.astype(np.int64) - ref.astype(np.int64))
            assert d.max() <= 1 and (d > 0).mean() <= 5e-3, "%s/%s: max diff %d, frac %.4f" % (case.name, k, d.max(), (d > 0).mean())
        else:
            tol = case.oracle_close.get(k, case.close[k])
            assert rel_err(a, ref) <= tol, "%s/%s: rel err %.3g > %.1g" % (case.name, k, rel_err(a, ref), tol)
        checked += 1
    assert checked > 0
