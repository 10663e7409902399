"""GPU: the PRODUCT path (FusedCodec -> C-ABI -> csrc/codec.cu, wavefront.cu) against the UNMODIFIED reference CUDA extension
(oracle/_ref/lic360_ref*.so driven by the per-op loops of test/lic360_demo.py:95-290) on BASELINE.json's own shapes:
configs[1] (512x1024 image: code latent 64x128, importance map 32x64) and configs[2] (1024x2048: 128x256 / 64x128).

What is asserted (north_star tiers):
  * both bitstreams of both implementations round-trip exactly through their own decoders;
  * stream sizes (bpp) agree within max(2 bytes, 0.1 %);
  * every layer of both context networks agrees with the reference's CconvEc within 1e-5 relative at the full shape;
  * the CDF tables built from the two networks' outputs differ in a bounded, reported fraction of rows, nearly always by one
    count (the conv is float-tier, SURVEY.md A.4: the reduction order differs from the reference's, so the 12-layer outputs differ
    in their last bits and int(65536 p + 0.5) flips wherever p sits next to a rounding boundary);
  * cross-decoding (reference stream -> this decoder and back) is measured and REPORTED, not asserted: an arithmetic decoder
    desynchronises at the first differing bin, so it succeeds only when no table on the coded path differs.
The measured numbers are written to gpurun_out/r2_parity_baseline_<H>x<W>.json (copied to profiles/ and quoted in DESIGN.md).
"""
import json
import os

import numpy as np
import pytest
import torch

from util import n, rel_err, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _layer_outputs(backend, params, ngroup, cpg, nlast, batch, x):
    """the 12 layer outputs of one context network in whole-frame (EC) form, lic360_demo.py:104-112 / :153-161"""
    import lic360_codec_ops as ops
    net = ops._Net(backend, params, ngroup, cpg, nlast, batch, False, 0)
    outs = []
    y = net._conv(net.first, x, 'net.0', True).clone()
    outs.append(y)
    for i, (c1, c2) in enumerate(net.blocks):
        a = net._conv(c1, y, 'net.%d.conv1' % (i + 1), True).clone()
        outs.append(a)
        b = net._conv(c2, a, 'net.%d.conv2' % (i + 1), True).clone()
        y = b + y
        outs.append(y)
    outs.append(net._conv(net.last, y, 'net.6', False).clone())
    return outs


def _gmm_tables(y, G, H, W):
    """int tables (G*H*W, 9) of every symbol from the code-stream network output (3, G*3, H, W) through this repo's table op
    (bit-exact against the reference's given identical inputs, tests/test_gpu_ops.py)"""
    import lic360
    S = G * H * W
    planes = y.view(3, G, 3, H, W).permute(0, 1, 3, 4, 2).reshape(3, S, 3).contiguous()
    op = lic360.EntropyGmmTableOp(8, 3.5, 3, 65536, 1e-6, 0, False)
    cnt = torch.tensor([S], dtype=torch.int32)
    w, d, m = [planes[k].clone().view(S, 3, 1, 1) for k in range(3)]  # rewritten in place by the op
    tab = op.forward(w, d, m, cnt)[0]
    return n(tab).reshape(-1, 9)[:S].astype(np.int64)


def _imp_tables(y, H, W):
    import lic360
    S = H * W
    logits = y.view(49, S).t().contiguous().view(S, 49, 1, 1)
    op = lic360.EntropyTableOp(49, 65536, 0, False)
    tab = op.forward(logits, torch.tensor([S], dtype=torch.int32))[0]
    return n(tab).reshape(-1, 50)[:S].astype(np.int64)


def _first_mismatch(a, b):
    d = np.flatnonzero(a.reshape(-1) != b.reshape(-1))
    return int(d[0]) if d.size else -1


def _against_recorded_reference_streams(H, W, seed):
    """Without the live extension: this repo's streams round-trip and their sizes agree, within the same bound, with the sizes of
    the reference extension's streams for the same seeded input (tests/golden/reference_streams.json)."""
    import lic360_pipeline as pl
    with open(os.path.join(ROOT, "tests", "golden", "reference_streams.json")) as f:
        rec = json.load(f).get("%dx%d_seed%d" % (H, W, seed))
    if rec is None:
        pytest.skip("oracle/_ref/lic360_ref*.so not present and no recorded reference streams for this shape")
    q, mask, lv = synthetic_latent(seed, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=seed)
    fused = pl.FusedCodec(params, H=H, W=W)
    bi, bc = fused.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
    code, mup = fused.decode(bi, bc)
    assert np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask)
    assert abs(len(bi) - rec["imp_bytes"]) <= max(2, 0.001 * rec["imp_bytes"]), (len(bi), rec)
    assert abs(len(bc) - rec["code_bytes"]) <= max(2, 0.001 * rec["code_bytes"]), (len(bc), rec)


@pytest.mark.parametrize("H,W,seed", [(64, 128, 2024), (128, 256, 2025)], ids=["config2_512x1024", "config3_1024x2048"])
def test_fused_codec_against_reference_extension(ref_ext, H, W, seed):
    if ref_ext is None:
        _against_recorded_reference_streams(H, W, seed)
        return
    import lic360
    import lic360_pipeline as pl
    q, mask, lv = synthetic_latent(seed, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=seed)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    fused = pl.FusedCodec(params, H=H, W=W)
    ref = pl.PerOpCodec(ref_ext, params)
    rep = {"latent": [1, 48, H, W], "importance_map": [1, 1, H // 2, W // 2], "seed": seed}

    # ---- streams: each implementation round-trips its own; sizes agree
    l0 = lic360.launch_count()
    bi, bc = fused.encode(tq, tm, tl)
    code, mup = fused.decode(bi, bc)
    assert lic360.launch_count() > l0
    assert np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask)
    rbi, rbc = ref.encode(tq, tm, tl)
    rcode, rmup = ref.decode(rbi, rbc, H // 2, W // 2)
    assert np.array_equal(n(rcode), q * mask) and np.array_equal(n(rmup), mask)
    rep["bytes"] = {"b200": [len(bi), len(bc)], "reference": [len(rbi), len(rbc)],
                    "identical": [bi == rbi, bc == rbc], "bpp_b200": 8.0 * (len(bi) + len(bc)) / (64 * H * W),
                    "bpp_reference": 8.0 * (len(rbi) + len(rbc)) / (64 * H * W)}
    assert abs(len(bi) - len(rbi)) <= max(2, 0.001 * len(rbi)), rep["bytes"]
    assert abs(len(bc) - len(rbc)) <= max(2, 0.001 * len(rbc)), rep["bytes"]

    # ---- every layer of both networks at the full shape: this repo's CconvEc kernels vs the reference's (float tier)
    x_code = torch.cat([(tq - 3.5) * tm] * 3).contiguous()
    mine = _layer_outputs(lic360, params['code'], 48, 4, 3, 3, x_code)
    theirs = _layer_outputs(ref_ext, params['code'], 48, 4, 3, 3, x_code)
    rep["code_layer_rel_err"] = [rel_err(n(a), n(b)) for a, b in zip(mine, theirs)]
    assert max(rep["code_layer_rel_err"]) <= 1e-5, rep["code_layer_rel_err"]
    x_imp = lic360.ScaleOp(-1, float(2. / 47.), 0, False).forward(tl)[0].clone()
    mine_i = _layer_outputs(lic360, params['imp'], 1, 144, 49, None, x_imp)
    theirs_i = _layer_outputs(ref_ext, params['imp'], 1, 144, 49, None, x_imp)
    rep["imp_layer_rel_err"] = [rel_err(n(a), n(b)) for a, b in zip(mine_i, theirs_i)]
    assert max(rep["imp_layer_rel_err"]) <= 1e-5, rep["imp_layer_rel_err"]

    # ---- CDF rows: how many differ between the two implementations' tables (both through the same bit-exact table op)
    ta, tb = _gmm_tables(mine[-1], 48, H, W), _gmm_tables(theirs[-1], 48, H, W)
    coded = (mask.reshape(48, H * W) > 0.5).reshape(-1)
    drow = (ta != tb).any(axis=1)
    rep["code_rows"] = {"total": int(ta.shape[0]), "coded": int(coded.sum()), "differing": int(drow.sum()),
                        "differing_coded": int((drow & coded).sum()), "max_bin_diff": int(np.abs(ta - tb).max())}
    rep["code_rows"]["bins_off_by_more_than_1"] = int((np.abs(ta - tb) > 1).sum())
    # measured on B200 (profiles/r2_parity_baseline_*.json): 2.7 % of the rows carry a bin that differs, almost always by one count;
    # sharp mixtures (delta near its 1e-6 floor) amplify a 1e-6 relative difference of the mean into several counts
    # (measured: 2.7 % / 2.6 % of the rows at 512x1024 / 1024x2048, 5 resp. a few hundred bins off by more than one count; the largest
    # single difference belongs to a near-degenerate mixture and is reported, not bounded)
    assert drow.mean() <= 5e-2 and (np.abs(ta - tb) > 1).mean() <= 1e-3, rep["code_rows"]
    ia, ib = _imp_tables(mine_i[-1], H // 2, W // 2), _imp_tables(theirs_i[-1], H // 2, W // 2)
    irow = (ia != ib).any(axis=1)
    rep["imp_rows"] = {"total": int(ia.shape[0]), "differing": int(irow.sum()), "max_bin_diff": int(np.abs(ia - ib).max())}
    assert irow.mean() <= 0.2 and (np.abs(ia - ib) > 1).mean() <= 1e-3, rep["imp_rows"]

    # ---- cross-decode, reported: the other implementation's streams through this decoder, and this repo's through the reference's
    cross = {}
    try:
        xcode, xmask = fused.decode(rbi, rbc)
        cross["reference_streams_through_b200_decoder"] = {
            "mask_exact": bool(np.array_equal(n(xmask), mask)), "code_exact": bool(np.array_equal(n(xcode), q * mask)),
            "first_wrong_symbol": _first_mismatch(n(xcode), q * mask), "wrong_symbols": int((n(xcode) != q * mask).sum())}
    except RuntimeError as e:
        cross["reference_streams_through_b200_decoder"] = {"error": str(e)[:200]}
    try:
        ycode, ymask = ref.decode(bi, bc, H // 2, W // 2)
        cross["b200_streams_through_reference_decoder"] = {
            "mask_exact": bool(np.array_equal(n(ymask), mask)), "code_exact": bool(np.array_equal(n(ycode), q * mask)),
            "wrong_symbols": int((n(ycode) != q * mask).sum())}
    except Exception as e:  # the reference coder throws C strings on a desynchronised stream
        cross["b200_streams_through_reference_decoder"] = {"error": repr(e)[:200]}
    rep["cross_decode"] = cross
    # when no coded row differs the streams must be byte-identical and cross-decodable (same coder, same order, same tables)
    if rep["code_rows"]["differing_coded"] == 0:
        assert bc == rbc
    if rep["imp_rows"]["differing"] == 0:
        assert bi == rbi
    print("parity report", json.dumps(rep))
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "r2_parity_baseline_%dx%d.json" % (H, W)), "w") as f:
            json.dump(rep, f, indent=1)


def test_importance_stream_against_reference_extension(tmp_path, ref_ext):
    """The 49-symbol importance stream (EntropyTable rows, 144-channel single-group net) at the config-2 size, stream level:
    sizes agree, both round-trip, and the stream-level byte comparison is reported through the assert message when it fails
    the size bound."""
    if ref_ext is None:
        pytest.skip("oracle/_ref/lic360_ref*.so not present")
    import lic360
    import lic360_codec_ops as ops
    _, _, lv = synthetic_latent(77, H=64, W=128)  # levels (1,1,32,64)
    params = ops.make_entropy_params(1, 144, 49, None, seed=78, device=DEV)
    f_mine, f_ref = str(tmp_path / "mine_imp"), str(tmp_path / "ref_imp")
    ops.ImpEntEncoder(lic360, params).encode(t(lv, DEV), f_mine)
    ops.ImpEntEncoder(ref_ext, params).encode(t(lv, DEV), f_ref)
    a, b = os.path.getsize(f_mine), os.path.getsize(f_ref)
    assert abs(a - b) <= max(2, 0.002 * b), (a, b)
    assert np.array_equal(n(ops.ImpEntDecoder(lic360, params).decode(f_mine, 32, 64, DEV)), lv)
    assert np.array_equal(n(ops.ImpEntDecoder(ref_ext, params).decode(f_ref, 32, 64, DEV)), lv)


def test_encode_reports_out_of_range_symbols():
    """A symbol outside 0..7 on a kept position must fail the encode (the per-op path says 'symbol out of range',
    coder.cpp), not wrap into a decodable but wrong stream (ADVICE r1)."""
    import lic360_pipeline as pl
    H, W = 8, 16
    q, mask, lv = synthetic_latent(5, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=5)
    fused = pl.FusedCodec(params, H=H, W=W)
    fused.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
    kept = np.argwhere(mask > 0.5)
    assert len(kept)
    for bad in (9.0, -1.0, float("nan")):
        q2 = q.copy()
        q2[tuple(kept[len(kept) // 2])] = bad
        with pytest.raises(RuntimeError, match="out of range"):
            fused.encode(t(q2, DEV), t(mask, DEV), t(lv, DEV))
    # the same values on a masked-out position are not coded and therefore fine (coder.cpp:79)
    dropped = np.argwhere(mask < 0.5)
    if len(dropped):
        q3 = q.copy()
        q3[tuple(dropped[0])] = 9.0
        fused.encode(t(q3, DEV), t(mask, DEV), t(lv, DEV))


def test_second_device_in_one_process():
    """Ops and a codec on cuda:1 after cuda:0 in the same process (ADVICE r1: shared-memory limits are per device, the
    launch needs the tensor's device current, the codec must not leave the caller on another device)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import lic360
    import lic360_pipeline as pl
    from op_cases import BY_NAME
    H, W = 16, 32
    q, mask, lv = synthetic_latent(9, H=H, W=W)
    outs = []
    for gid in (0, 1):
        dev = "cuda:%d" % gid
        params = pl.make_codec_params(dev, seed=9)
        fused = pl.FusedCodec(params, H=H, W=W, gid=gid)
        assert torch.cuda.current_device() == 0
        bi, bc = fused.encode(t(q, dev), t(mask, dev), t(lv, dev))
        code, mup = fused.decode(bi, bc)
        assert torch.cuda.current_device() == 0
        assert np.array_equal(n(code), q * mask)
        outs.append((bi, bc))
        ec = BY_NAME["cconv_ec_batch_hidden_g12"].run(lic360, dev)["out"]
        outs.append(ec)
    assert outs[0] == outs[2] and np.array_equal(outs[1], outs[3])
