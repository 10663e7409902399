"""GPU: the product codec (FusedCodec: csrc/codec.cu, csrc/wavefront.cu, the packed-row coder) and the per-op path on the
probe networks of probe_nets.py, whose streams are known exactly from a closed form, float64 tables and the host coder.
Unlike a round trip, this fails when the encoder and the decoder share a wrong table, mask rule or coding order."""
import functools

import numpy as np
import pytest

import probe_nets as pn
from util import n, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SHAPES = [(2, 2), (8, 16), (10, 14), (16, 12), (6, 130), (24, 72), (64, 128), (128, 256)]


@functools.lru_cache(maxsize=None)
def _case(name, H, W, seed):
    params = pn.probe_params(name)
    q, mask, lv = synthetic_latent(seed, H=H, W=W)
    return params, (q, mask, lv), pn.expected_streams(params, q, mask, lv)


@functools.lru_cache(maxsize=None)
def _torch_params(name):
    return pn.to_torch(pn.probe_params(name), DEV)


def _decode_ok(codec, streams, q, mask):
    code, mup = codec.decode(*streams)
    return np.array_equal(n(mup), mask) and np.array_equal(n(code), q * mask)


@pytest.mark.parametrize("H,W", SHAPES)
@pytest.mark.parametrize("name", pn.PROBES)
def test_fused_codec_writes_the_expected_streams(name, H, W):
    import lic360
    import lic360_pipeline as pl
    _, (q, mask, lv), want = _case(name, H, W, 100 + H + W)
    params = _torch_params(name)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    fused = pl.FusedCodec(params, H=H, W=W)
    got = fused.encode(tq, tm, tl)
    assert got[0] == want[0], "importance stream differs (%d vs %d bytes)" % (len(got[0]), len(want[0]))
    assert got[1] == want[1], "code stream differs (%d vs %d bytes)" % (len(got[1]), len(want[1]))
    if H * W <= 64 * 128:
        assert pl.PerOpCodec(lic360, params).encode(tq, tm, tl) == want
    assert _decode_ok(fused, want, q, mask)
    fused.set_mode(2)
    assert _decode_ok(fused, want, q, mask)
    # a second image through the same codec object
    _, (q2, mask2, lv2), want2 = _case(name, H, W, 200 + H + W)
    fused.set_mode(0)
    assert fused.encode(t(q2, DEV), t(mask2, DEV), t(lv2, DEV)) == want2
    assert _decode_ok(fused, want2, q2, mask2)


def test_out_of_range_symbol_is_a_coder_error():
    """No table the fix-up emits has an empty bin (test_ref64), so a symbol the coder cannot code is one outside 0..7:
    both paths refuse it and return no stream."""
    import lic360
    import lic360_pipeline as pl
    H, W = 8, 16
    _, (q, mask, lv), _ = _case("E", H, W, 100 + H + W)
    q = q.copy()
    c, h, w = np.argwhere(mask[0] > 0.5)[5]
    q[0, c, h, w] = 8
    params = _torch_params("E")
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    with pytest.raises(RuntimeError, match="coder|range"):
        pl.FusedCodec(params, H=H, W=W).encode(tq, tm, tl)
    with pytest.raises(RuntimeError):
        pl.PerOpCodec(lic360, params).encode(tq, tm, tl)


@pytest.mark.parametrize("H,W", [(8, 16), (64, 128), (128, 256)])
def test_interop_with_reference_extension(ref_ext, H, W):
    """Where the arithmetic is exact by construction, the reference extension's per-op codec writes the same bytes, and each
    implementation decodes the other's streams."""
    if ref_ext is None:
        pytest.skip("oracle/_ref/lic360_ref*.so not present: the expected streams above still pin the product path")
    import lic360_pipeline as pl
    for name in pn.PROBES:
        _, (q, mask, lv), want = _case(name, H, W, 100 + H + W)
        params = _torch_params(name)
        ref = pl.PerOpCodec(ref_ext, params)
        assert ref.encode(t(q, DEV), t(mask, DEV), t(lv, DEV)) == want, name
        code, mup = ref.decode(*want, H // 2, W // 2)
        assert np.array_equal(n(code), q * mask) and np.array_equal(n(mup), mask), name
        assert _decode_ok(pl.FusedCodec(params, H=H, W=W), want, q, mask), name
