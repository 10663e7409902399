"""GPU: the batched encode (FusedCodec.encode_batch, lic360_codec_encode_batch) against single-latent encodes byte for byte, through
decode, across batch sizes and buffer growth, interleaved with the codec's other calls, with errors, and from two threads at once."""
import functools
import threading

import numpy as np
import pytest

import probe_nets as pn
from test_gpu_rate_estimate import _raised
from util import n, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SHAPES = [(8, 16), (10, 14), (6, 130), (24, 72), (64, 128)]


def _pl():
    import lic360_pipeline as pl
    return pl


@functools.lru_cache(maxsize=None)
def _params(kind):
    pl = _pl()
    return pl.make_codec_params(DEV, seed=2000) if kind == "random" else pn.to_torch(pn.probe_params(kind), DEV)


@functools.lru_cache(maxsize=None)
def _codec(kind, H, W):
    return _pl().FusedCodec(_params(kind), H=H, W=W)


def _latents(K, H, W, seed):
    qs, ms, ls = zip(*[synthetic_latent(seed + 17 * k, H=H, W=W) for k in range(K)])
    return np.concatenate(qs), np.concatenate(ms), np.concatenate(ls)


def _singles(codec, q, m, lv):
    return [codec.encode(t(q[k:k + 1], DEV), t(m[k:k + 1], DEV), t(lv[k:k + 1], DEV)) for k in range(q.shape[0])]


def _assert_batch_equals_singles(codec, q, m, lv, decode=False):
    got = codec.encode_batch(t(q, DEV), t(m, DEV), t(lv, DEV))
    K = q.shape[0]
    assert len(got) == K
    assert all(isinstance(a, bytes) and isinstance(b, bytes) for a, b in got)
    assert (codec._stream_bytes(1), codec._stream_bytes(0)) == got[0], "stream_size / stream_copy return latent 0"
    want = _singles(codec, q, m, lv)
    for k in range(K):
        assert got[k] == want[k], "latent %d: imp %d/%d bytes, code %d/%d bytes" % (
            k, len(got[k][0]), len(want[k][0]), len(got[k][1]), len(want[k][1]))
    if decode:
        for k, (imp, code) in enumerate(got):
            cd, mup = codec.decode(imp, code)
            assert np.array_equal(n(mup), m[k:k + 1]), "latent %d: mask" % k
            assert np.array_equal(n(cd), q[k:k + 1] * m[k:k + 1]), "latent %d: code" % k
    return got


@pytest.mark.parametrize("H,W", SHAPES)
@pytest.mark.parametrize("kind", ["random", "P"])
def test_batch_equals_singles_and_decodes(kind, H, W):
    q, m, lv = _latents(5, H, W, 2100 + H + W)
    codec = _codec(kind, H, W)
    _assert_batch_equals_singles(codec, q, m, lv, decode=True)
    tm = codec.last_timing()
    assert tm["total_ms"] >= tm["host_coder_ms"] > 0 and tm["gpu_wait_ms"] >= 0


@pytest.mark.parametrize("K,H,W", [(1, 10, 14), (16, 32, 64)])
def test_batch_k1_k16(K, H, W):
    q, m, lv = _latents(K, H, W, 2200)
    _assert_batch_equals_singles(_codec("random", H, W), q, m, lv)


def test_batch_sizes_and_buffer_growth():
    """a batch beyond what an earlier estimate_batch grew, then a smaller one; a single encode is unchanged after each"""
    pl = _pl()
    H, W = 16, 32
    q, m, lv = _latents(7, H, W, 2300)
    codec = pl.FusedCodec(_params("random"), H=H, W=W)
    one = codec.encode(t(q[:1], DEV), t(m[:1], DEV), t(lv[:1], DEV))
    codec.estimate_batch(t(q[:3], DEV), t(m[:3], DEV), t(lv[:3], DEV), maps=False)
    for lo, hi in ((0, 7), (2, 4), (1, 2), (0, 5)):
        _assert_batch_equals_singles(codec, q[lo:hi], m[lo:hi], lv[lo:hi])
        assert codec.encode(t(q[:1], DEV), t(m[:1], DEV), t(lv[:1], DEV)) == one, (lo, hi)


def test_extreme_latents_in_one_batch():
    """all levels 0 (no code symbol coded) and all levels 48 (every code symbol coded) beside an ordinary latent"""
    pl = _pl()
    H, W = 12, 40
    q, m, lv = _latents(3, H, W, 2400)
    for k, level in ((1, 0.0), (2, 48.0)):
        lv[k] = level
        _, mk = pl.levels_to_mask(t(lv[k:k + 1], DEV), [0])
        m[k] = n(mk)[0]
    assert m[1].sum() == 0 and m[2].min() == 1
    got = _assert_batch_equals_singles(_codec("random", H, W), q, m, lv, decode=True)
    assert len(got[2][1]) > len(got[0][1]) > len(got[1][1])


def test_interleaved_calls_leave_results_unchanged():
    """encode_batch -> estimate_batch -> encode -> decode -> encode_batch on one codec, in mode 0 and in mode 2"""
    pl = _pl()
    H, W = 24, 72
    q, m, lv = _latents(4, H, W, 2500)
    tq, tm, tl = t(q, DEV), t(m, DEV), t(lv, DEV)
    codec = pl.FusedCodec(_params("random"), H=H, W=W)
    want = codec.encode_batch(tq, tm, tl)
    est = codec.estimate_batch(tq, tm, tl, maps=False)
    for mode in (0, 2):
        codec.set_mode(mode)
        assert codec.encode_batch(tq, tm, tl) == want, mode
        e = codec.estimate_batch(tq, tm, tl, maps=False)
        assert [(x["code_bits"], x["imp_bits"]) for x in e] == [(x["code_bits"], x["imp_bits"]) for x in est], mode
        assert codec.encode(tq[2:3], tm[2:3], tl[2:3]) == want[2], mode
        cd, mup = codec.decode(*want[1])
        assert np.array_equal(n(mup), m[1:2]) and np.array_equal(n(cd), q[1:2] * m[1:2]), mode
        assert codec.encode_batch(tq, tm, tl) == want, mode


def test_errors_name_the_first_bad_latent():
    pl = _pl()
    H, W = 8, 16
    codec = pl.FusedCodec(_params("random"), H=H, W=W)
    q, m, lv = _latents(5, H, W, 2600)
    tq, tm, tl = t(q, DEV), t(m, DEV), t(lv, DEV)
    want = codec.encode_batch(tq, tm, tl)
    kept = tuple(np.argwhere(m[3] > 0.5)[4])
    for where, what in ((("q", 3) + kept, 8.0), (("lv", 3, 0, 1, 2), 49.0)):
        qq, ll = q.copy(), lv.copy()
        (qq if where[0] == "q" else ll)[where[1:]] = what
        if where[0] == "q":
            qq[(4,) + kept] = 9.0  # a later bad latent does not change the message
        single = _raised(codec.encode, t(qq[3:4], DEV), t(m[3:4], DEV), t(ll[3:4], DEV))
        assert single is not None
        for _ in range(3):
            got = _raised(codec.encode_batch, t(qq, DEV), t(m, DEV), t(ll, DEV))
            assert got == single + " (latent 3)", (got, single)
        with pytest.raises(RuntimeError, match="not in the last encode"):
            codec._batch_stream_bytes(0, 0)
        assert codec.encode_batch(tq, tm, tl) == want, "a good batch right after a failed one"
    for args in ((tq[..., :-2], tm, tl), (tq, tm.double(), tl), (tq, tm, tl.cpu()), (tq, tm[:4], tl), (tq, tm, tl[:, :, :-1]),
                 (tq[:0], tm[:0], tl[:0])):
        with pytest.raises(RuntimeError):
            codec.encode_batch(*args)
    assert codec.encode_batch(tq, tm, tl) == want
    for k, sid in ((5, 0), (-1, 1), (0, 2)):
        with pytest.raises(RuntimeError):
            codec._batch_stream_bytes(k, sid)
    assert codec._batch_stream_bytes(4, 0) == want[4][1]
    codec.decode(*want[0])
    with pytest.raises(RuntimeError, match="not in the last encode"):
        codec._batch_stream_bytes(0, 0)


def test_two_codecs_on_two_threads():
    """two encode_batch calls of K = 4 at the same time, one per codec and thread, give the serial results"""
    pl = _pl()
    H, W = 32, 64
    q, m, lv = _latents(8, H, W, 2700)
    codecs = [pl.FusedCodec(_params("random"), H=H, W=W) for _ in range(2)]
    parts = [(t(q[4 * i:4 * i + 4], DEV), t(m[4 * i:4 * i + 4], DEV), t(lv[4 * i:4 * i + 4], DEV)) for i in range(2)]
    serial = [c.encode_batch(*p) for c, p in zip(codecs, parts)]
    got, errs = [None, None], []
    start = threading.Barrier(2)

    def run(i):
        try:
            start.wait()
            got[i] = codecs[i].encode_batch(*parts[i])
        except Exception as e:  # noqa: BLE001 -- reported below
            errs.append(e)

    threads = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errs, errs
    assert got == serial
    assert serial[0] == _singles(codecs[0], q[:4], m[:4], lv[:4])
