"""GPU: the batched rate estimate (FusedCodec.estimate_batch, lic360_codec_estimate_batch) against single-latent estimates bit for bit
and against the probe networks' float64 bits; the candidate levels and masks of levels_to_mask (lic360_imp_levels_to_mask) against
synthetic_latent and a numpy restatement, and through encode -> decode; and FusedCodec.encode_to_budget."""
import functools

import numpy as np
import pytest
import torch

import probe_nets as pn
from test_gpu_rate_estimate import _assert_estimate, _raised
from util import n, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SHAPES = [(8, 16), (10, 14), (6, 130), (64, 128)]


def _pl():
    import lic360_pipeline as pl
    return pl


@functools.lru_cache(maxsize=None)
def _params(kind):
    pl = _pl()
    return pl.make_codec_params(DEV, seed=1000) if kind == "random" else pn.to_torch(pn.probe_params(kind), DEV)


@functools.lru_cache(maxsize=None)
def _codec(kind, H, W):
    return _pl().FusedCodec(_params(kind), H=H, W=W)


def _latents(K, H, W, seed):
    qs, ms, ls = zip(*[synthetic_latent(seed + 17 * k, H=H, W=W) for k in range(K)])
    return np.concatenate(qs), np.concatenate(ms), np.concatenate(ls)


def _bits(x):
    return n(x).view(np.int32)


def _assert_batch_equals_singles(codec, q, m, lv, maps=True):
    K = q.shape[0]
    got = codec.estimate_batch(t(q, DEV), t(m, DEV), t(lv, DEV), maps=maps)
    assert len(got) == K
    for k, e in enumerate(got):
        one = codec.estimate(t(q[k:k + 1], DEV), t(m[k:k + 1], DEV), t(lv[k:k + 1], DEV))
        assert e["code_bits"] == one["code_bits"] and e["imp_bits"] == one["imp_bits"], (k, e["code_bits"], one["code_bits"])
        assert e["code_symbols"] == int((m[k] >= 0.5).sum()) and e["imp_symbols"] == lv[k].size, k
        if maps:
            for key in ("code_map", "imp_map"):
                assert e[key].shape == one[key].shape, key
                diff = np.argwhere(_bits(e[key]) != _bits(one[key]))
                assert len(diff) == 0, "latent %d %s: %d entries differ, first %s" % (k, key, len(diff), tuple(diff[0]))
        else:
            assert e["code_map"] is None and e["imp_map"] is None
    return got


@pytest.mark.parametrize("H,W", SHAPES)
@pytest.mark.parametrize("kind", ["random", "P"])
def test_batch_equals_singles_bit_for_bit(kind, H, W):
    q, m, lv = _latents(5, H, W, 1100 + H + W)
    codec = _codec(kind, H, W)
    _assert_batch_equals_singles(codec, q, m, lv)
    _assert_batch_equals_singles(codec, q, m, lv, maps=False)


@pytest.mark.parametrize("K,H,W", [(1, 10, 14), (16, 32, 64)])
def test_batch_equals_singles_k1_k16(K, H, W):
    q, m, lv = _latents(K, H, W, 1200)
    _assert_batch_equals_singles(_codec("random", H, W), q, m, lv)


@pytest.mark.parametrize("name", pn.PROBES)
def test_probe_networks_exact_bits_in_a_batch(name):
    """each batch entry is within 1 ulp of the float64 bits of the probe networks' exact tables"""
    H, W = 10, 14
    q, m, lv = _latents(3, H, W, 1300)
    got = _codec(name, H, W).estimate_batch(t(q, DEV), t(m, DEV), t(lv, DEV))
    params = pn.probe_params(name)
    for k, e in enumerate(got):
        tables = pn.expected_tables(params, q[k:k + 1], m[k:k + 1], lv[k:k + 1])
        _assert_estimate(e, *tables, m[k:k + 1], H, W)


def _same_batch(a, b):
    return all(x["code_bits"] == y["code_bits"] and x["imp_bits"] == y["imp_bits"] and x["code_symbols"] == y["code_symbols"]
               and torch.equal(x["code_map"], y["code_map"]) and torch.equal(x["imp_map"], y["imp_map"]) for x, y in zip(a, b))


def test_batch_is_deterministic_and_leaves_encode_alone():
    pl = _pl()
    H, W = 24, 72
    params = pl.make_codec_params(DEV, seed=1400)
    q, m, lv = _latents(4, H, W, 1401)
    tq, tm, tl = t(q, DEV), t(m, DEV), t(lv, DEV)
    codec = pl.FusedCodec(params, H=H, W=W)
    want = codec.encode(tq[:1], tm[:1], tl[:1])
    e1 = codec.estimate_batch(tq, tm, tl)
    assert _same_batch(e1, codec.estimate_batch(tq, tm, tl)), "second batch on the same codec"
    assert _same_batch(e1, pl.FusedCodec(params, H=H, W=W).estimate_batch(tq, tm, tl)), "batch on a second codec"
    got = codec.encode(tq[:1], tm[:1], tl[:1])
    assert got == want, "encode after a batch estimate"
    code, mup = codec.decode(*got)
    assert np.array_equal(n(mup), m[:1]) and np.array_equal(n(code), q[:1] * m[:1])
    codec.set_mode(2)
    assert _same_batch(e1, codec.estimate_batch(tq, tm, tl)), "batch in mode 2"
    # a smaller batch after a larger one: the grown buffers serve it unchanged
    assert _same_batch(e1[1:3], codec.estimate_batch(tq[1:3], tm[1:3], tl[1:3]))


def _np_levels_to_mask(lv, k, G=48):
    """numpy restatement: max(s - k, 0), channel c < 4 L of the 192-channel mask, then depth-to-width"""
    L = np.maximum(lv.astype(np.int64) - k, 0)[0, 0]
    h, w = L.shape
    c = np.arange(4 * G)[:, None, None]
    m192 = (c < 4 * L[None]).astype(np.float32)
    m = m192.reshape(G, 2, 2, h, w).transpose(0, 3, 1, 4, 2).reshape(1, G, 2 * h, 2 * w)
    return L.astype(np.float32)[None, None], m


def test_levels_to_mask_matches_synthetic_latent_and_numpy():
    pl = _pl()
    H, W = 12, 40
    q, mask, lv = synthetic_latent(1500, H=H, W=W)
    levels, masks = pl.levels_to_mask(t(lv, DEV), [0, 1, 7, 48])
    assert levels.shape == (4, 1, H // 2, W // 2) and masks.shape == (4, 48, H, W) and masks.device == torch.device(DEV)
    assert np.array_equal(n(levels[0:1]), lv) and np.array_equal(n(masks[0:1]), mask), "offset 0 is synthetic_latent's mask"
    for j, k in enumerate([0, 1, 7, 48]):
        wl, wm = _np_levels_to_mask(lv, k)
        assert np.array_equal(n(levels[j:j + 1]), wl), k
        assert np.array_equal(n(masks[j:j + 1]), wm), k
    assert n(masks[3]).sum() == 0 and n(levels[3]).sum() == 0
    # fractional levels: the symbol encode codes is their integer part
    lf = lv + 0.75
    lf[lf >= 49] = 48.5
    levels_f, masks_f = pl.levels_to_mask(t(lf, DEV), [3])
    wl, wm = _np_levels_to_mask(np.trunc(lf), 3)
    assert np.array_equal(n(levels_f), wl) and np.array_equal(n(masks_f), wm)


def test_derived_pair_decodes_to_its_mask():
    pl = _pl()
    H, W = 16, 48
    q, _, lv = synthetic_latent(1600, H=H, W=W)
    codec = _codec("random", H, W)
    levels, masks = pl.levels_to_mask(t(lv, DEV), [5])
    got = codec.encode(t(q, DEV), masks, levels)
    code, mup = codec.decode(*got)
    wm = n(masks)
    assert 0 < wm.sum() < wm.size
    assert np.array_equal(n(mup), wm), "the decoder's mask is the derived one"
    assert np.array_equal(n(code), q * wm), "the kept symbols are unchanged"


@functools.lru_cache(maxsize=None)
def _budget_case():
    pl = _pl()
    H, W = 16, 48
    q, mask, lv = synthetic_latent(1700, H=H, W=W)
    tq = t(q, DEV)
    codec = _codec("random", H, W)
    offsets = list(range(49))
    levels, masks = pl.levels_to_mask(t(lv, DEV), offsets)
    ests = codec.estimate_batch(tq.expand(49, -1, -1, -1), masks, levels, maps=False)
    bounds = {k: pl.budget_bound(e) for k, e in zip(offsets, ests)}
    return codec, q, mask, lv, bounds


def _check_budget(budget):
    pl = _pl()
    codec, q, mask, lv, all_bounds = _budget_case()
    r = codec.encode_to_budget(t(q, DEV), t(lv, DEV), budget)
    total = len(r["imp_bytes"]) + len(r["code_bytes"])
    assert total <= r["bound"] <= budget, (total, r["bound"], budget)
    assert r["bounds"] == {k: all_bounds[k] for k in r["bounds"]}, "bounds of the evaluated offsets"
    assert r["offset"] == min(k for k, b in r["bounds"].items() if b <= budget), "the smallest evaluated offset that fits"
    assert r["bound"] == all_bounds[r["offset"]]
    levels, masks = pl.levels_to_mask(t(lv, DEV), [r["offset"]])
    assert torch.equal(r["levels"], levels) and torch.equal(r["mask"], masks)
    assert (r["imp_bytes"], r["code_bytes"]) == codec.encode(t(q, DEV), masks, levels)
    code, mup = codec.decode(r["imp_bytes"], r["code_bytes"])
    assert np.array_equal(n(mup), n(masks)) and np.array_equal(n(code), q * n(masks))
    return r


def test_budget_at_offset_zero():
    codec, q, mask, lv, bounds = _budget_case()
    r = _check_budget(bounds[0])
    assert r["offset"] == 0 and sorted(r["bounds"]) == list(range(0, 49, 8))
    assert (r["imp_bytes"], r["code_bytes"]) == codec.encode(t(q, DEV), t(mask, DEV), t(lv, DEV))


def test_budget_inside_the_range():
    _, _, _, _, bounds = _budget_case()
    budget = (bounds[0] + bounds[48]) // 2
    r = _check_budget(budget)
    assert 0 < r["offset"] < 48 and len(r["bounds"]) == 14


def test_budget_at_the_ends_of_the_range():
    codec, q, mask, lv, bounds = _budget_case()
    assert bounds[48] < bounds[0]
    _check_budget(bounds[48] + 1)
    with pytest.raises(RuntimeError, match="no level offset"):
        codec.encode_to_budget(t(q, DEV), t(lv, DEV), bounds[48] - 1)


def test_errors_name_the_first_bad_latent():
    pl = _pl()
    H, W = 8, 16
    codec = _codec("random", H, W)
    q, m, lv = _latents(5, H, W, 1800)
    kept = tuple(np.argwhere(m[3] > 0.5)[4])
    for where, what in ((("q", 3) + kept, 8.0), (("lv", 3, 0, 1, 2), 49.0)):
        qq, ll = q.copy(), lv.copy()
        (qq if where[0] == "q" else ll)[where[1:]] = what
        if where[0] == "q":
            (qq)[(4,) + kept] = 9.0  # a later bad latent does not change the message
        single = _raised(codec.encode, t(qq[3:4], DEV), t(m[3:4], DEV), t(ll[3:4], DEV))
        assert single is not None
        got = _raised(codec.estimate_batch, t(qq, DEV), t(m, DEV), t(ll, DEV))
        assert got == single + " (latent 3)", (got, single)
    tq, tm, tl = t(q, DEV), t(m, DEV), t(lv, DEV)
    for args in ((tq[..., :-2], tm, tl), (tq, tm.double(), tl), (tq, tm, tl.cpu()), (tq, tm[:4], tl), (tq, tm, tl[:, :, :-1]),
                 (tq[:0], tm[:0], tl[:0])):
        with pytest.raises(RuntimeError):
            codec.estimate_batch(*args)
    with pytest.raises(RuntimeError, match="must not be negative"):
        pl.levels_to_mask(tl[:1], [0, -1])
    with pytest.raises(RuntimeError, match="at least 1"):
        pl.levels_to_mask(tl[:1], [])
    with pytest.raises(RuntimeError):
        pl.levels_to_mask(tl[:1].double(), [0])
    assert codec.estimate_batch(tq, tm, tl)[4]["code_bits"] > 0
