"""GPU: the fused decoder at every latent size and cluster setting where the wavefront engine picks a different chain kernel.

wf_init (csrc/wavefront.cu) chooses the importance stream's chain kernel from its longest diagonal and the cluster size:
wf_chain1_kernel with activations exchanged through distributed shared memory (DSM), the same kernel with its tile reloaded
from the frame every layer, or the generic wf_chain_kernel, whose threads loop over their tasks.  The encoder does not depend
on that choice, so a broken variant writes streams that look fine and do not decode.  Every case asserts the variant it is
named for (FusedCodec.engine_info: a retuned threshold fails here instead of quietly covering another kernel), that the
importance stream is the byte string of the CPU model of the canonical fp32 order (canon_conv), and that decoding the
model's bytes gives back the latent exactly.  Codecs of up to 256x512 hold about 13 GB of frames: one is alive at a time."""
import contextlib
import os
import tempfile

import numpy as np
import pytest

import canon_conv as cc
import probe_nets as pn
from test_gpu_canonical_conv import _np, _random_biases
from util import n, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

CHAIN1_DSM16 = dict(chain="chain1", dsm=True, cluster=16, c1_kpc=3)
CHAIN1_TILE16 = dict(chain="chain1", dsm=False, cluster=16, c1_kpc=3)
# name: (H, W, environment switch, stream whose engine the case is about (0 code, 1 importance), expected engine_info)
CASES = {
    "dsm_lenp64_128x256": (128, 256, None, 1, dict(CHAIN1_DSM16, max_len=64, c1_lenp=64)),  # control: the largest size tested before
    "dsm_lenp96_130x260": (130, 260, None, 1, dict(CHAIN1_DSM16, max_len=65, c1_lenp=96, chain_smem=228992)),
    "dsm_lenp96_192x384": (192, 384, None, 1, dict(CHAIN1_DSM16, max_len=96, c1_lenp=96, chain_smem=228992)),
    "tile_lenp128_196x194": (196, 194, None, 1, dict(CHAIN1_TILE16, max_len=97, c1_lenp=128, chain_smem=202560)),  # H > W
    "tile_lenp128_256x512": (256, 512, None, 1, dict(CHAIN1_TILE16, max_len=128, c1_lenp=128, chain_smem=202560)),
    "generic_258x260": (258, 260, None, 1, dict(chain="generic", cluster=16, max_len=129)),
    "imp8_dsm_64x128": (64, 128, "LIC360_WF_CLUSTER_IMP=8", 1, dict(chain="chain1", dsm=True, cluster=8, c1_kpc=5, c1_lenp=32)),
    "imp8_tile_66x132": (66, 132, "LIC360_WF_CLUSTER_IMP=8", 1, dict(chain="chain1", dsm=False, cluster=8, c1_kpc=5, c1_lenp=64)),
    "imp8_generic_130x260": (130, 260, "LIC360_WF_CLUSTER_IMP=8", 1, dict(chain="generic", cluster=8, max_len=65)),
    "code4_tail_24x72": (24, 72, "LIC360_WF_CLUSTER_CODE=4", 0, dict(chain="chain4", cluster=4, tail_rounds=3)),
}
BOTH_STREAMS = {"dsm_lenp96_130x260"}  # the first size the shared-memory limit opens: the code stream against the model too
MODE2 = {"tile_lenp128_256x512"}  # also decoded in the low-latency mode


@pytest.fixture(scope="module")
def params():
    import lic360_pipeline as pl
    p = pl.make_codec_params(DEV, seed=910)
    _random_biases(p["code"], 911)
    _random_biases(p["imp"], 912)
    return p


@contextlib.contextmanager
def _codec(params, H, W):
    import lic360_pipeline as pl
    c = pl.FusedCodec(params, H=H, W=W)
    try:
        yield c
    finally:
        c.__del__()  # its frames go now, even when a failed assertion keeps this frame (and the codec) referenced


def _model_streams(params, q, mask, lv, code):
    """the importance stream (and with code=True the code stream) built from canon_conv's network outputs by the per-op
    encoders' table ops and coder, as test_gpu_canonical_conv._codec_case does; None for a stream not built"""
    import lic360
    import lic360_codec_ops as ops
    d = tempfile.mkdtemp(prefix="lic360_geom_")
    out = []
    try:
        y_imp = t(cc.net(_np(params["imp"]), pn.imp_input(lv)[None], 1, 1), DEV)
        enc_i = ops.ImpEntEncoder(lic360, params["imp"])
        enc_i.net = lambda _: y_imp.clone()
        enc_i.encode(t(lv, DEV), os.path.join(d, "imp"))
        if code:
            y_code = t(cc.net(_np(params["code"]), pn.code_input(q, mask), 48, 3), DEV)
            enc_c = ops.EntEncoder(lic360, params["code"])
            enc_c.net = lambda _: y_code.clone()
            enc_c.encode(t(q, DEV), t(mask, DEV), os.path.join(d, "code"))
        for f in ("imp", "code"):
            p = os.path.join(d, f)
            if os.path.exists(p):
                with open(p, "rb") as fh:
                    out.append(fh.read())
                os.remove(p)
            else:
                out.append(None)
    finally:
        os.rmdir(d)
    return tuple(out)


def _assert_decodes(codec, streams, q, mask, what):
    code, mup = codec.decode(*streams)
    mup, code = n(mup), n(code)
    assert np.array_equal(mup, mask), "%s: decoded mask differs at %d positions" % (what, int((mup != mask).sum()))
    assert np.array_equal(code, q * mask), "%s: decoded symbols differ at %d positions" % (what, int((code != q * mask).sum()))


def _assert_engine(info, want, what):
    got = {k: info[k] for k in want}
    assert got == want, "%s: engine %s, expected %s (full: %s)" % (what, got, want, info)
    if want["chain"] == "generic":  # the case is there for the thread loop over tasks: it must be entered
        assert info["chain_tasks"] > info["chain_threads"], (what, info)


def _check_decoder(codec, name, streams, q, mask):
    """engine_info as the case expects, then the decode of the expected streams (both modes where listed)"""
    H, W, env, sid, want = CASES[name]
    _assert_engine(codec.engine_info(sid), want, name)
    if name == "tile_lenp128_256x512":  # the code stream's chain at the same size: 4 slab items per thread, 4-part old-term tiles
        c = codec.engine_info(0)
        per_cta = -(-c["max_len"] // c["cluster"])
        assert (c["chain"], -(-per_cta // c["chain_threads"]), c["parts4"]) == ("chain4", 4, 4), c
    _assert_decodes(codec, streams, q, mask, name + ", mode 0")
    if name in MODE2:
        codec.set_mode(2)
        _assert_decodes(codec, streams, q, mask, name + ", mode 2")


@pytest.mark.parametrize("name", list(CASES))
def test_decoder_variant(monkeypatch, params, name):
    H, W, env, sid, want = CASES[name]
    q, mask, lv = synthetic_latent(920 + H + W, H=H, W=W)
    tq, tm, tl = t(q, DEV), t(mask, DEV), t(lv, DEV)
    model_imp, model_code = _model_streams(params, q, mask, lv, name in BOTH_STREAMS)
    with _codec(params, H, W) as codec:
        got = codec.encode(tq, tm, tl)
        assert got[0] == model_imp, "importance stream differs from the model (%d vs %d bytes)" % (len(got[0]), len(model_imp))
        if model_code is not None:
            assert got[1] == model_code, "code stream differs from the model (%d vs %d bytes)" % (len(got[1]), len(model_code))
        streams = (model_imp, got[1] if model_code is None else model_code)
        if env is None:
            _check_decoder(codec, name, streams, q, mask)
            return
        if want.get("tail_rounds"):  # 8 CTAs stage the R tail's weight rows in two rounds here: the switch is what reaches a third
            assert codec.engine_info(0)["tail_rounds"] == 2, codec.engine_info(0)
    key, _, value = env.partition("=")
    monkeypatch.setenv(key, value)
    with _codec(params, H, W) as codec:
        assert codec.encode(tq, tm, tl) == got, "%s changes the encoded bytes" % env  # the encoder ignores the decoder's setup
        _check_decoder(codec, name, streams, q, mask)
