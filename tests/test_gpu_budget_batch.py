"""GPU: rate control of many latents.  FusedCodec.estimate_candidates (lic360_codec_estimate_candidates) against estimate_batch of the
materialised candidates, levels_to_mask_batch against levels_to_mask and numpy, encode_batch_to_budget per latent against
encode_to_budget and in its shared mode, BandCodec.encode_to_budget, and the errors."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from test_gpu_budget_protect import _np_protected, _random_protect
from util import n, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _pl():
    import lic360_pipeline as pl
    return pl


@functools.lru_cache(maxsize=None)
def _codec(H, W):
    pl = _pl()
    return pl.FusedCodec(pl.make_codec_params(DEV, seed=1000), H=H, W=W)


def _sources(K, H, W, seed):
    """K synthetic latents stacked: code (K,48,H,W) and importance levels (K,1,H/2,W/2) on the GPU"""
    qs, lvs = zip(*[(q, lv) for q, _, lv in (synthetic_latent(seed + k, H=H, W=W) for k in range(K))])
    return t(np.concatenate(qs), DEV), t(np.concatenate(lvs), DEV)


def _protects(K, h, w, seed):
    return torch.from_numpy(np.concatenate([_random_protect(h, w, seed + k) for k in range(K)])).to(DEV)


def _materialised(code, imp, pairs, protect):
    """the candidates' code, levels and masks as levels_to_mask builds them one source at a time"""
    pl = _pl()
    parts = [pl.levels_to_mask(imp[k:k + 1], [o], None if protect is None else protect[k:k + 1]) for k, o in pairs]
    idx = torch.tensor([k for k, _ in pairs], device=DEV)
    return code[idx].contiguous(), torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])


def _same_estimates(got, want):
    for j, (g, w) in enumerate(zip(got, want)):
        for key in ("code_bits", "imp_bits", "code_symbols", "imp_symbols"):
            assert g[key] == w[key], (j, key, g[key], w[key])


@pytest.mark.parametrize("with_protect", [False, True])
def test_estimate_candidates_equals_estimate_batch_of_the_materialised_candidates(with_protect):
    pl = _pl()
    H, W, K = 16, 32, 3
    codec = _codec(H, W)
    code, imp = _sources(K, H, W, 3000)
    protect = _protects(K, H // 2, W // 2, 3010) if with_protect else None
    top = 48 + (int(protect.max()) if with_protect else 0)
    # unsorted, a repeated pair, every source, offsets 0 and the top, and above 48 with a map: 37 candidates
    pairs = [(2, 5), (0, 0), (1, top), (0, 17), (2, 5), (1, 3), (0, top), (2, 0), (1, 48)]
    pairs += [(k, o) for o in range(top, 0, -3) for k in range(K)][:37 - len(pairs)]  # 48 pairs or more: 16+ offsets x 3
    assert len(pairs) == 37 and (not with_protect or max(o for _, o in pairs) > 48)
    got = codec.estimate_candidates(code, imp, [k for k, _ in pairs], [o for _, o in pairs], protect)
    mcode, levels, masks = _materialised(code, imp, pairs, protect)
    want = codec.estimate_batch(mcode, masks, levels, maps=False)
    _same_estimates(got, want)
    # in passes of at most 16 candidates (J not a multiple of it): the same numbers
    chunked = pl._chunked(lambda ps: codec.estimate_candidates(code, imp, [k for k, _ in ps], [o for _, o in ps], protect), pairs, 16)
    _same_estimates(chunked, want)
    # a repeated pair is estimated twice, alike
    assert got[0] == got[4]


def test_levels_to_mask_batch_matches_levels_to_mask_and_numpy():
    pl = _pl()
    H, W, K = 12, 40, 3
    _, imp = _sources(K, H, W, 3100)
    P = _protects(K, H // 2, W // 2, 3110)
    pairs = [(1, 60), (0, 0), (2, 33), (1, 0), (0, 96), (2, 49), (1, 60)] + [(j % K, j) for j in range(40)]
    lat, off = [k for k, _ in pairs], [o for _, o in pairs]
    for protect in (None, P):
        levels, masks = pl.levels_to_mask_batch(imp, lat, off, protect)
        assert levels.shape == (len(pairs), 1, H // 2, W // 2) and masks.shape == (len(pairs), 48, H, W)
        for j, (k, o) in enumerate(pairs):
            one = pl.levels_to_mask(imp[k:k + 1], [o], None if protect is None else protect[k:k + 1])
            assert torch.equal(levels[j:j + 1], one[0]) and torch.equal(masks[j:j + 1], one[1]), (j, k, o)
            Pk = np.zeros((1, 1, H // 2, W // 2), np.int32) if protect is None else n(protect[k:k + 1])
            wl, wm = _np_protected(n(imp[k:k + 1]), Pk, o)
            assert np.array_equal(n(levels[j:j + 1]), wl) and np.array_equal(n(masks[j:j + 1]), wm), (j, k, o)


def _budgets(codec, code, imp, protect):
    """four distinct budgets per latent: at offset 0's bound, halfway, just above the top offset's bound, and at a third"""
    top = [48 + (0 if protect is None else int(protect[k].max())) for k in range(code.shape[0])]
    pairs = [(k, o) for k in range(code.shape[0]) for o in (0, top[k])]
    ests = codec.estimate_candidates(code, imp, [k for k, _ in pairs], [o for _, o in pairs], protect)
    b = [_pl().budget_bound(e) for e in ests]
    ends = [(b[2 * k], b[2 * k + 1]) for k in range(code.shape[0])]
    shapes = [lambda b0, bz: b0, lambda b0, bz: (b0 + bz) // 2, lambda b0, bz: bz + 1, lambda b0, bz: bz + (b0 - bz) // 3]
    return [shapes[k % 4](*ends[k]) for k in range(code.shape[0])]


def _same_result(got, want):
    assert sorted(got) == sorted(want)
    for key in want:
        same = torch.equal(got[key], want[key]) if isinstance(want[key], torch.Tensor) else got[key] == want[key]
        assert same, key


@pytest.mark.parametrize("with_protect", [False, True])
def test_per_latent_mode_equals_encode_to_budget(with_protect):
    H, W, K = 16, 32, 4
    codec = _codec(H, W)
    code, imp = _sources(K, H, W, 3200)
    protect = None
    if with_protect:
        pl = _pl()
        lat = pl.latitude_protection(H // 2, W // 2, 16, DEV)
        protect = torch.cat([torch.zeros_like(lat), lat, _protects(1, H // 2, W // 2, 3210), torch.full_like(lat, 7)])
    budgets = _budgets(codec, code, imp, protect)
    assert len(set(budgets)) == K
    want = [codec.encode_to_budget(code[k:k + 1], imp[k:k + 1], budgets[k], None if protect is None else protect[k:k + 1])
            for k in range(K)]
    assert len({r["offset"] for r in want}) > 1
    for max_batch in (3, 16):
        got = codec.encode_batch_to_budget(code, imp, budgets, protect=protect, max_batch=max_batch)
        assert len(got) == K
        for k in range(K):
            _same_result(got[k], want[k])
    for k, r in enumerate(got):
        dcode, dmask = codec.decode(r["imp_bytes"], r["code_bytes"])
        assert torch.equal(dmask, r["mask"]) and torch.equal(dcode, code[k:k + 1] * r["mask"]), k
    # one int for every latent
    same = codec.encode_batch_to_budget(code, imp, max(budgets), protect=protect)
    for k in range(K):
        _same_result(same[k], codec.encode_to_budget(code[k:k + 1], imp[k:k + 1], max(budgets),
                                                     None if protect is None else protect[k:k + 1]))


def test_shared_mode():
    pl = _pl()
    H, W, K = 16, 32, 3
    codec = _codec(H, W)
    code, imp = _sources(K, H, W, 3300)
    ends = codec.estimate_candidates(code, imp, [0, 1, 2] * 2, [0] * 3 + [48] * 3)
    b0 = sum(pl.budget_bound(e) for e in ends[:3])
    bz = sum(pl.budget_bound(e) for e in ends[3:])
    checked_between = False
    for budget in (b0, (b0 + bz) // 2, bz + (b0 - bz) // 5, bz):
        r = codec.encode_batch_to_budget(code, imp, budget, shared=True, max_batch=5)
        res = r["results"]
        assert sum(len(x["imp_bytes"]) + len(x["code_bytes"]) for x in res) <= r["bound"] <= budget
        assert r["offset"] == min(o for o, b in r["bounds"].items() if b <= budget), "the smallest evaluated offset that fits"
        assert all(x["offset"] == r["offset"] for x in res)
        pairs = [(k, o) for o in sorted(r["bounds"]) for k in range(K)]
        ests = codec.estimate_candidates(code, imp, [k for k, _ in pairs], [o for _, o in pairs])
        for i, o in enumerate(sorted(r["bounds"])):
            per = [pl.budget_bound(e) for e in ests[i * K:(i + 1) * K]]
            assert r["bounds"][o] == sum(per), o
            assert [x["bounds"][o] for x in res] == per
        levels, masks = pl.levels_to_mask_batch(imp, range(K), [r["offset"]] * K)
        for k, x in enumerate(res):
            assert torch.equal(x["levels"], levels[k:k + 1]) and torch.equal(x["mask"], masks[k:k + 1])
            assert (x["imp_bytes"], x["code_bytes"]) == codec.encode(code[k:k + 1], masks[k:k + 1], levels[k:k + 1])
            dcode, dmask = codec.decode(x["imp_bytes"], x["code_bytes"])
            assert torch.equal(dmask, masks[k:k + 1]), k
        o, bd = r["offset"], r["bounds"]
        if o > 0 and o - 1 in bd and bd[o - 1] > bd[o] and all(bd[k] >= bd[o - 1] for k in bd if k < o):
            # a budget between the summed bounds of o - 1 and o takes o, the larger offset
            mid = (bd[o - 1] + bd[o]) // 2
            between = codec.encode_batch_to_budget(code, imp, mid, shared=True)
            assert between["offset"] == o and between["bounds"][o] <= mid < between["bounds"][o - 1]
            checked_between = True
    assert checked_between
    # K = 1 is encode_to_budget
    for budget in (b0 // 3, (b0 + bz) // 6):
        want = codec.encode_to_budget(code[1:2], imp[1:2], budget)
        got = codec.encode_batch_to_budget(code[1:2], imp[1:2], budget, shared=True)
        assert got["offset"] == want["offset"] and got["bound"] == want["bound"] and got["bounds"] == want["bounds"]
        _same_result(got["results"][0], want)


@pytest.mark.parametrize("with_protect", [False, True])
def test_band_codec_encode_to_budget(with_protect):
    pl = _pl()
    from lic360_shard import BandCodec, unpack_band_streams
    H, W, nb = 32, 64, 2
    params = pl.make_codec_params(DEV, seed=1000)
    band = BandCodec(lambda h, w: pl.FusedCodec(params, H=h, W=w), H, W, nb)
    q, _, lv = synthetic_latent(3400, H=H, W=W)
    code, imp = t(q, DEV), t(lv, DEV)
    protect = pl.latitude_protection(H // 2, W // 2, 24, DEV) if with_protect else None
    full = band.encode(code, t(synthetic_latent(3400, H=H, W=W)[1], DEV), imp)
    budget = len(full) * 2 // 3
    r = band.encode_to_budget(code, imp, budget, protect=protect)
    blob = r["container"]
    assert len(blob) <= r["bound"] <= budget
    assert r["offset"] == min(o for o, b in r["bounds"].items() if b <= budget)
    H2, W2, streams = unpack_band_streams(blob)
    assert (H2, W2, len(streams)) == (H, W, nb)
    bc = band.codecs[0]
    for b, (r0, r1) in enumerate(band.rows):
        rows = slice(r0 // 2, r1 // 2)
        levels, masks = pl.levels_to_mask(imp[:, :, rows].contiguous(), [r["offset"]],
                                          None if protect is None else protect[:, :, rows].contiguous())
        dcode, dmask = bc.decode(*streams[b])
        assert torch.equal(dmask, masks), b
        assert torch.equal(dcode, code[:, :, r0:r1] * masks), b
    dcode, dmask = band.decode(blob)
    assert dmask.shape == (1, 48, H, W)
    assert torch.equal(dmask, torch.cat([x["mask"] for x in r["results"]], dim=2))
    assert torch.equal(dcode, code * dmask)


def test_errors():
    pl = _pl()
    from lic360._lib import LIB
    H, W, K = 8, 16, 4
    codec = _codec(H, W)
    code, imp = _sources(K, H, W, 3500)
    big = 10 ** 6
    # no offset fits latent 2
    with pytest.raises(RuntimeError, match=r"^encode_to_budget: no level offset up to 48 fits 1 bytes .*\(latent 2\)$"):
        codec.encode_batch_to_budget(code, imp, [big, big, 1, 1])
    # a candidate encode would refuse: level 60 is out of range until an offset of 12 brings it to 48, a code symbol of 9 until
    # its cell's level is 0
    bad_imp, bad_code = imp.clone(), code.clone()
    bad_imp[1, 0, 2, 3] = 60
    lvl = 20
    bad_imp[3, 0, 0, 0] = lvl
    bad_code[3, 0, 0, 0] = 9
    pairs = [(1, 12), (3, lvl), (0, 0), (3, 0), (1, 0)]
    ok = codec.estimate_candidates(bad_code, bad_imp, [0, 1, 3], [0, 12, lvl])
    assert len(ok) == 3
    mcode, levels, masks = _materialised(bad_code, bad_imp, pairs[3:4], None)
    with pytest.raises(RuntimeError) as single:
        codec.estimate_batch(mcode, masks, levels, maps=False)
    with pytest.raises(RuntimeError) as batch:
        codec.estimate_candidates(bad_code, bad_imp, [k for k, _ in pairs], [o for _, o in pairs])
    assert str(batch.value) == str(single.value).replace("(latent 0)", "(candidate 3)")
    with pytest.raises(RuntimeError, match=r"importance level 49 out of range \(candidate 1\)$"):
        codec.estimate_candidates(bad_code, bad_imp, [1, 1], [12, 11])
    # shapes, dtypes, devices, budgets, max_batch
    for args in ((code.double(), imp), (code, imp.double()), (code.cpu(), imp), (code[:3], imp), (code[:, :, :-2], imp)):
        with pytest.raises(RuntimeError, match="FusedCodec"):
            codec.encode_batch_to_budget(*args, big)
    with pytest.raises(RuntimeError, match="3 budgets for 4 latents"):
        codec.encode_batch_to_budget(code, imp, [big] * 3)
    with pytest.raises(RuntimeError, match="one budget"):
        codec.encode_batch_to_budget(code, imp, [big] * 4, shared=True)
    for mb in (0, 2.5, None):
        with pytest.raises(RuntimeError, match="max_batch"):
            codec.encode_batch_to_budget(code, imp, big, max_batch=mb)
    good = torch.zeros((K, 1, H // 2, W // 2), dtype=torch.int32, device=DEV)
    high = good.clone()
    high[2, 0, 1, 1] = 49
    for bad in (good.float(), good[:3], good.cpu(), high):
        with pytest.raises(RuntimeError, match="protect"):
            codec.encode_batch_to_budget(code, imp, big, protect=bad)
        with pytest.raises(RuntimeError, match="protect"):
            pl.levels_to_mask_batch(imp, [0], [0], bad)
    # the C-ABI: a source outside [0, K), a negative offset
    c_int = ctypes.c_int
    totals, counts = (ctypes.c_double * 4)(), (ctypes.c_longlong * 4)()
    for lat, off, msg in (((0, 4), (0, 0), b"cand_latent"), ((0, -1), (0, 0), b"cand_latent"), ((0, 1), (0, -2), b"negative")):
        rc = LIB.lic360_codec_estimate_candidates(codec._h, K, code.data_ptr(), imp.data_ptr(), None, 2, (c_int * 2)(*lat),
                                                  (c_int * 2)(*off), totals, counts)
        assert rc != 0 and msg in LIB.lic360_last_error()
        lv_out = torch.empty((2, 1, H // 2, W // 2), device=DEV)
        m_out = torch.empty((2, 48, H, W), device=DEV)
        rc = LIB.lic360_imp_levels_to_mask_batch(imp.data_ptr(), K, H // 2, W // 2, None, 2, (c_int * 2)(*lat), (c_int * 2)(*off),
                                                 lv_out.data_ptr(), m_out.data_ptr(), None)
        assert rc != 0 and msg in LIB.lic360_last_error()
    with pytest.raises(RuntimeError, match="cand_latent"):
        pl.levels_to_mask_batch(imp, [K], [0])
    with pytest.raises(RuntimeError, match="negative"):
        codec.estimate_candidates(code, imp, [0], [-1])
    # band budgets across ranks
    from lic360_shard import BandCodec
    band = BandCodec(lambda h, w: codec, H, W, 2, world=2, rank=0)
    with pytest.raises(RuntimeError, match="world == 1"):
        band.encode_to_budget(code[:1], imp[:1], big)
