"""GPU: encoder/decoder consistency of the context model (EC == DC bit-for-bit), codec round trips through the
per-op loops (the restated lic360_demo.py drivers), and stream-level comparison with the reference extension."""
import os

import numpy as np
import pytest
import torch

from util import n, rel_err, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _net_pair(ngroup, cpg, nlast, batch, seed, H, W):
    import lic360
    import lic360_codec_ops as ops
    params = ops.make_entropy_params(ngroup, cpg, nlast, batch, seed, DEV)
    ec = ops._Net(lic360, params, ngroup, cpg, nlast, batch, False, 0)
    dc = ops._Net(lic360, params, ngroup, cpg, nlast, batch, True, 0)
    ops._plan(lic360, torch.zeros((1, 1, H, W), device=DEV), 0, dc.stateful())
    return ec, dc


@pytest.mark.parametrize("ngroup,cpg,nlast,batch,H,W", [(48, 4, 3, 3, 8, 16), (12, 4, 3, 3, 13, 9), (1, 24, 9, None, 8, 16)])
def test_full_net_ec_equals_dc_bitwise(ngroup, cpg, nlast, batch, H, W):
    """12 stacked context convs: the wavefront (decoder) form reproduces the whole-frame (encoder) form bit-for-bit;
    otherwise the arithmetic decoder would desynchronise (SURVEY.md s7 hard part 1)."""
    ec, dc = _net_pair(ngroup, cpg, nlast, batch, 5, H, W)
    r = np.random.default_rng(0)
    x1 = (r.integers(0, 8, (1, ngroup, H, W)) - 3.5).astype(np.float32)
    x = t(np.concatenate([x1] * (batch or 1)), DEV)
    y_ec = n(ec(x)).copy()
    y_dc = None
    for _ in range(H + W + ngroup - 2):
        y_dc = dc(x)
    y_dc = n(y_dc)
    assert np.isfinite(y_ec).all() and np.abs(y_ec).max() > 1e-3
    assert np.array_equal(_bits(y_ec), _bits(y_dc)), "EC and DC differ in %d of %d values" % ((_bits(y_ec) != _bits(y_dc)).sum(), y_ec.size)


@pytest.mark.parametrize("H,W,seed", [(8, 16, 1), (6, 10, 2)])
def test_code_stream_round_trip(tmp_path, H, W, seed):
    import lic360
    import lic360_codec_ops as ops
    q, mask, _ = synthetic_latent(seed, H=H, W=W)
    params = ops.make_entropy_params(48, 4, 3, 3, seed=seed, device=DEV)
    fn = str(tmp_path / "code")
    ops.EntEncoder(lic360, params).encode(t(q, DEV), t(mask, DEV), fn)
    rec = n(ops.EntDecoder(lic360, params).decode(t(mask, DEV), fn))
    # EntDecoder returns frame + 3.5*mask: coded symbols where mask == 1, 0 elsewhere (lic360_demo.py:236-237)
    assert np.array_equal(rec, q * mask)
    assert 0 < os.path.getsize(fn) < q.size


def test_code_stream_all_masked_and_all_kept(tmp_path):
    import lic360
    import lic360_codec_ops as ops
    q, mask, _ = synthetic_latent(3, H=6, W=8)
    params = ops.make_entropy_params(48, 4, 3, 3, seed=9, device=DEV)
    for m in (np.zeros_like(mask), np.ones_like(mask)):
        fn = str(tmp_path / ("code%d" % int(m[0, 0, 0, 0])))
        ops.EntEncoder(lic360, params).encode(t(q, DEV), t(m, DEV), fn)
        rec = n(ops.EntDecoder(lic360, params).decode(t(m, DEV), fn))
        assert np.array_equal(rec, q * m)
        if m.sum() == 0:
            assert os.path.getsize(fn) == 1  # only the terminator bit, ArithmeticCoder.cpp:152-154


def test_importance_stream_round_trip(tmp_path):
    import lic360
    import lic360_codec_ops as ops
    _, _, lv = synthetic_latent(4, H=16, W=32)  # levels (1,1,8,16) in 0..48
    params = ops.make_entropy_params(1, 144, 49, None, seed=11, device=DEV)
    fn = str(tmp_path / "code_imp")
    ops.ImpEntEncoder(lic360, params).encode(t(lv, DEV), fn)
    rec = n(ops.ImpEntDecoder(lic360, params).decode(fn, h=8, w=16, device=DEV))
    assert np.array_equal(rec, lv)


def test_streams_against_reference_extension(tmp_path, ref_ext):
    """Same seeded parameters and latent through the reference CUDA extension and through this repo: the conv outputs
    agree to the float tier, so the tables agree except for rare +-1 bins and the stream sizes (bpp) match; each
    implementation decodes its own stream exactly and, being format-identical, the other's stream wherever the tables
    coincide.  Identical tables -> identical bytes is asserted in tests/test_oracle_coder.py."""
    if ref_ext is None:
        pytest.skip("oracle/_ref/lic360_ref*.so not present")
    import lic360
    import lic360_codec_ops as ops
    q, mask, _ = synthetic_latent(5, H=8, W=16)
    params = ops.make_entropy_params(48, 4, 3, 3, seed=21, device=DEV)
    f_mine, f_ref = str(tmp_path / "mine"), str(tmp_path / "ref")
    ops.EntEncoder(lic360, params).encode(t(q, DEV), t(mask, DEV), f_mine)
    ops.EntEncoder(ref_ext, params).encode(t(q, DEV), t(mask, DEV), f_ref)
    a, b = os.path.getsize(f_mine), os.path.getsize(f_ref)
    assert abs(a - b) <= max(2, 0.002 * b), (a, b)
    rec_ref = n(ops.EntDecoder(ref_ext, params).decode(t(mask, DEV), f_ref))
    assert np.array_equal(rec_ref, q * mask)
    # network output parity (float tier) on the same input
    x = t(np.concatenate([(q - 3.5) * mask] * 3), DEV)
    y_mine = n(ops._Net(lic360, params, 48, 4, 3, 3, False, 0)(x))
    y_ref = n(ops._Net(ref_ext, params, 48, 4, 3, 3, False, 0)(x))
    assert rel_err(y_mine, y_ref) <= 1e-5, rel_err(y_mine, y_ref)


@pytest.mark.parametrize("H,W,seed", [(8, 16, 31), (16, 12, 32)])
def test_fused_codec_matches_per_op_path(H, W, seed):
    """The native pipeline (csrc/codec.cu: graph replay per step, packed rows, no Python in the loop) emits exactly
    the bytes of the per-op loops, decodes them, and decodes the per-op path's streams."""
    import lic360
    import lic360_pipeline as pl
    q, mask, lv = synthetic_latent(seed, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=seed)
    per_op = pl.PerOpCodec(lic360, params)
    fused = pl.FusedCodec(params, H=H, W=W)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    bi0, bc0 = per_op.encode(tq, tm, tl)
    l0 = lic360.launch_count()
    bi1, bc1 = fused.encode(tq, tm, tl)
    assert lic360.launch_count() > l0
    assert bi1 == bi0 and bc1 == bc0, "fused and per-op bitstreams differ (%d/%d vs %d/%d bytes)" % (len(bi1), len(bc1), len(bi0), len(bc0))
    code, mup = fused.decode(bi0, bc0)
    # the decoded importance levels regenerate the mask: it equals the encoder's mask iff the mask is the level map's
    lv_mask = n(mup)
    assert np.array_equal(lv_mask, mask)
    assert np.array_equal(n(code), q * mask)
    code2, mup2 = per_op.decode(bi1, bc1, H // 2, W // 2)
    assert np.array_equal(n(code2), q * mask) and np.array_equal(n(mup2), mask)
    # a second image through the same codec object (graph + buffers reused)
    q2, mask2, lv2 = synthetic_latent(seed + 100, H=H, W=W)
    b = fused.encode(t(q2, DEV), t(mask2, DEV), t(lv2, DEV))
    code3, mup3 = fused.decode(*b)
    assert np.array_equal(n(code3), q2 * mask2) and np.array_equal(n(mup3), mask2)


def test_fused_codec_rejects_bad_input():
    import lic360_pipeline as pl
    params = pl.make_codec_params(DEV, seed=1)
    fused = pl.FusedCodec(params, H=8, W=16)
    with pytest.raises(RuntimeError):
        fused.encode(torch.zeros((1, 48, 8, 16)), torch.zeros((1, 48, 8, 16), device=DEV), torch.zeros((1, 1, 4, 8), device=DEV))
    with pytest.raises(RuntimeError):
        fused.encode(torch.zeros((1, 48, 8, 8), device=DEV), torch.zeros((1, 48, 8, 16), device=DEV), torch.zeros((1, 1, 4, 8), device=DEV))
    # a truncated / foreign stream must not hang or crash: it either decodes to garbage or reports a coder error
    q, mask, lv = synthetic_latent(2, H=8, W=16)
    bi, bc = fused.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
    try:
        fused.decode(bi, bc[: len(bc) // 2])
    except RuntimeError as e:
        assert "coder" in str(e)


def test_fused_codec_serialized_mode():
    """The profile mode (kernels launched one by one with events, lic360_codec_set_mode(1)) decodes the same bytes to the
    same symbols as the default pipelined path."""
    import lic360_pipeline as pl
    H, W = 12, 20
    q, mask, lv = synthetic_latent(41, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=41)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    fused = pl.FusedCodec(params, H=H, W=W)
    bi, bc = fused.encode(tq, tm, tl)
    code0, m0 = fused.decode(bi, bc)
    assert np.array_equal(n(code0), q * mask) and np.array_equal(n(m0), mask)
    fused.set_mode(1)
    code1, m1 = fused.decode(bi, bc)
    kt = fused.kernel_times(0)
    assert kt['steps'] == H + W + 48 - 2 and kt['old_ms'] > 0 and kt['chain_ms'] > 0
    assert np.array_equal(n(code1), n(code0)) and np.array_equal(n(m1), n(m0))


def test_fused_codec_1024x2048_latent():
    """LIC3602K shape (configs[2]): latent (1,48,128,256), 430 + 191 wavefront steps, two items per chain thread."""
    import lic360_pipeline as pl
    H, W = 128, 256
    q, mask, lv = synthetic_latent(43, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=43)
    fused = pl.FusedCodec(params, H=H, W=W)
    bi, bc = fused.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
    code, mup = fused.decode(bi, bc)
    assert np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask)
    assert 0 < len(bc) < q.size and 0 < len(bi) < lv.size


def test_fused_codec_stress_many_images_in_flight():
    """Stress of the decoder's cross-CTA data exchange (the code-stream chain reads, with plain L1-allocating loads, values
    that other CTAs of its cluster stored earlier in the same launch, ordered only by the cluster barrier; the three clusters meet
    at a global counter): 3 codecs decode concurrently from 3 host threads, 8 different images each, two latent sizes with long
    diagonals (several items per chain thread).  A single stale or torn read desynchronises the arithmetic decoder, so exact
    round trips of ~10 million symbols are the check."""
    import threading
    import lic360_pipeline as pl
    errors = []
    for H, W, nimg in ((64, 128, 8), (96, 160, 4)):
        params = pl.make_codec_params(DEV, seed=H)
        codecs = [pl.FusedCodec(params, H=H, W=W) for _ in range(3)]
        lat = [synthetic_latent(500 + 10 * k + i, H=H, W=W) for k in range(3) for i in range(nimg)]

        def worker(k):
            try:
                for i in range(nimg):
                    q, mask, lv = lat[k * nimg + i]
                    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
                    bi, bc = codecs[k].encode(tq, tm, tl)
                    code, mup = codecs[k].decode(bi, bc)
                    if not (np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask)):
                        errors.append((H, W, k, i))
            except Exception as e:  # noqa: BLE001
                errors.append((H, W, k, repr(e)))

        th = [threading.Thread(target=worker, args=(k,)) for k in range(3)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        del codecs
    assert not errors, errors


@pytest.mark.parametrize("H,W,seed", [(8, 16, 51), (64, 128, 52), (96, 160, 53)])
def test_fused_codec_low_latency_mode(H, W, seed):
    """lic360_codec_set_mode(2): ONE launch of the code-stream chain kernel walks all wavefront steps (it polls the symbols the host
    publishes, word by word, instead of being re-launched).  Same bytes in, same symbols out as the graph-replay decode; a truncated
    stream ends in a coder error (or garbage), never in a hang; the codec object can switch back."""
    import lic360_pipeline as pl
    q, mask, lv = synthetic_latent(seed, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=seed)
    fused = pl.FusedCodec(params, H=H, W=W, mode=2)
    bi, bc = fused.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
    for _ in range(2):
        code, mup = fused.decode(bi, bc)
        assert np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask)
    try:
        fused.decode(bi, bc[: len(bc) // 2])
    except RuntimeError as e:
        assert "coder" in str(e)
    code, mup = fused.decode(bi, bc)  # the aborted decode left nothing behind
    assert np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask)
    fused.set_mode(0)
    code0, mup0 = fused.decode(bi, bc)
    assert np.array_equal(n(code0), n(code)) and np.array_equal(n(mup0), n(mup))


@pytest.mark.parametrize("ncodec", [2, 7])
def test_fused_codec_low_latency_mode_several_decodes_at_once(ncodec):
    """Persistent decodes on one GPU from several host threads (3 resident clusters = 24 SMs each): all finish, all exact.  Seven is more
    than the device can keep resident next to the importance streams' clusters: the surplus decodes queue on the host (codec.cu)."""
    import threading
    import lic360_pipeline as pl
    H, W = 64, 128
    params = pl.make_codec_params(DEV, seed=61)
    codecs = [pl.FusedCodec(params, H=H, W=W, mode=2) for _ in range(ncodec)]
    lat = [synthetic_latent(600 + k, H=H, W=W) for k in range(ncodec)]
    errors = []

    def worker(k):
        try:
            q, mask, lv = lat[k]
            bi, bc = codecs[k].encode(t(q, DEV), t(mask, DEV), t(lv, DEV))
            for _ in range(3):
                code, mup = codecs[k].decode(bi, bc)
                if not (np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask)):
                    errors.append((k, "mismatch"))
        except Exception as e:  # noqa: BLE001
            errors.append((k, repr(e)))

    th = [threading.Thread(target=worker, args=(k,)) for k in range(ncodec)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    assert not errors, errors


def test_band_codec_round_trip():
    """One image as independently coded latitude bands (lic360_shard.BandCodec: BASELINE.json configs[3], a format extension -- SURVEY.md
    s8e option 3): every band's two streams are exactly the bytes the codec emits for that band as an image of its own, the container
    decodes to the image, and the price of the lost context at the band edges stays small."""
    import lic360_pipeline as pl
    import lic360_shard as sh
    H, W, NB = 64, 128, 4
    q, mask, lv = synthetic_latent(81, H=H, W=W)
    params = pl.make_codec_params(DEV, seed=81)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    bc = sh.BandCodec(lambda h, w: pl.FusedCodec(params, H=h, W=w), H, W, NB, in_flight=2)
    blob = bc.encode(tq, tm, tl)
    h, w, streams = sh.unpack_band_streams(blob)
    assert (h, w, len(streams)) == (H, W, NB)
    one = pl.FusedCodec(params, H=H // NB, W=W)
    for b, (r0, r1) in enumerate(sh.band_rows(H, NB)):
        alone = one.encode(tq[:, :, r0:r1].contiguous(), tm[:, :, r0:r1].contiguous(), tl[:, :, r0 // 2:r1 // 2].contiguous())
        assert streams[b] == alone
    code, m = bc.decode(blob, like=tq)
    assert np.array_equal(n(code), q * mask) and np.array_equal(n(m), mask)
    single = pl.FusedCodec(params, H=H, W=W).encode(tq, tm, tl)
    total, ref = sum(len(a) + len(b) for a, b in streams), len(single[0]) + len(single[1])
    assert 0.9 * ref <= total <= 1.1 * ref, (total, ref)
