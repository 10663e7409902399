"""GPU: FusedCodec.encode_candidates (lic360_codec_encode_candidates) against encode_batch of the materialised candidates, its buffers,
accessors and errors, and TileCodec.encode_ladder: budget rungs against TileCodec.encode_to_budget, offset rungs against
TileCodec.encode, and mixed cuts (rungs_for_views + ladder_to_tiles) decoded by decode_tiles / decode_views."""
import functools

import numpy as np
import pytest
import torch

import probe_nets as pn
from test_gpu_budget_protect import _random_protect
from util import synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _pl():
    import lic360_pipeline as pl
    return pl


def _sh():
    import lic360_shard as sh
    return sh


@functools.lru_cache(maxsize=None)
def _params(kind):
    return _pl().make_codec_params(DEV, seed=4100) if kind == "random" else pn.to_torch(pn.probe_params(kind), DEV)


@functools.lru_cache(maxsize=None)
def _codec(kind, H, W):
    return _pl().FusedCodec(_params(kind), H=H, W=W)


def _sources(K, H, W, seed):
    """K synthetic latents stacked: code (K,48,H,W) and importance levels (K,1,H/2,W/2); source 1 (when K > 2) has every level 0 and
    source 2 (when K > 3) every level 48"""
    qs, lvs = zip(*[(q, lv) for q, _, lv in (synthetic_latent(seed + k, H=H, W=W) for k in range(K))])
    code, imp = t(np.concatenate(qs), DEV), t(np.concatenate(lvs), DEV)
    if K > 2:
        imp[1] = 0
    if K > 3:
        imp[2] = 48
    return code, imp


def _protects(K, h, w, seed):
    return torch.from_numpy(np.concatenate([_random_protect(h, w, seed + k) for k in range(K)])).to(DEV)


def _materialised(code, imp, pairs, protect):
    """the candidates' code, masks and levels, materialised by levels_to_mask_batch, in encode_batch's argument order"""
    lat, off = [k for k, _ in pairs], [o for _, o in pairs]
    levels, masks = _pl().levels_to_mask_batch(imp, lat, off, protect)
    return code[torch.tensor(lat, device=DEV)].contiguous(), masks, levels


def _split(pairs):
    return [k for k, _ in pairs], [o for _, o in pairs]


def _pairs37(K, top):
    """37 unsorted (source, offset) pairs with repeats, every source, offsets 0, 48 and the top"""
    pairs = [(2 % K, 5), (0, 0), (1 % K, top), (0, 17), (2 % K, 5), (1 % K, 3), (0, top), (K - 1, 0), (1 % K, 48)]
    pairs += [(k, o) for o in range(top, 0, -3) for k in range(K)][:37 - len(pairs)]
    assert len(pairs) == 37
    return pairs


@pytest.mark.parametrize("with_protect", [False, True])
@pytest.mark.parametrize("kind", ["random", "P"])
def test_encode_candidates_equals_encode_batch_of_the_materialised_candidates(kind, with_protect):
    H, W, K = 16, 32, 4
    codec = _codec(kind, H, W)
    code, imp = _sources(K, H, W, 4200)
    protect = _protects(K, H // 2, W // 2, 4210) if with_protect else None
    top = 48 + (int(protect.max()) if with_protect else 0)
    pairs = _pairs37(K, top)
    assert not with_protect or max(o for _, o in pairs) > 48
    got = codec.encode_candidates(code, imp, *_split(pairs), protect=protect)
    mcode, masks, levels = _materialised(code, imp, pairs, protect)
    want = codec.encode_batch(mcode, masks, levels)
    assert len(got) == 37
    for j in range(37):
        assert got[j] == want[j], (j, pairs[j])
    assert got[0] == got[4]  # a repeated pair
    # in passes of at most 16 candidates: the same streams
    passes = sum((codec.encode_candidates(code, imp, *_split(pairs[i:i + 16]), protect=protect) for i in range(0, 37, 16)), [])
    assert passes == got
    # every stream decodes to its candidate's mask and the source's code under it
    for j, (k, _) in enumerate(pairs):
        dcode, dmask = codec.decode(*got[j])
        assert torch.equal(dmask, masks[j:j + 1]), j
        assert torch.equal(dcode, code[k:k + 1] * masks[j:j + 1]), j


@pytest.mark.parametrize("H,W", [(8, 16), (32, 64), (64, 128)])
def test_encode_candidates_at_other_sizes(H, W):
    codec = _codec("random", H, W)
    K = 4
    code, imp = _sources(K, H, W, 4300 + H)
    for protect in (None, _protects(K, H // 2, W // 2, 4310 + H)):
        pairs = [(3, 2), (0, 0), (2, 0), (1, 0), (2, 30), (0, 11), (3, 60), (0, 11)]
        got = codec.encode_candidates(code, imp, *_split(pairs), protect=protect)
        mcode, masks, levels = _materialised(code, imp, pairs, protect)
        assert got == codec.encode_batch(mcode, masks, levels)
        dcode, dmask = codec.decode(*got[0])
        assert torch.equal(dmask, masks[:1]) and torch.equal(dcode, code[3:4] * masks[:1])


def test_buffers_grow_and_interleave_with_other_calls():
    from lic360._lib import LIB
    H, W = 16, 32
    codec = _pl().FusedCodec(_params("random"), H=H, W=W)  # a fresh codec: its buffers start at one latent
    code, imp = _sources(4, H, W, 4400)

    def check_candidates(pairs):
        got = codec.encode_candidates(code, imp, *_split(pairs))
        mcode, masks, levels = _materialised(code, imp, pairs, None)
        return got, (mcode, masks, levels)

    # after a larger estimate_candidates (the frames hold 40, the row buffers one)
    codec.estimate_candidates(code, imp, [j % 4 for j in range(40)], list(range(40)))
    small = [(1, 4), (0, 9), (3, 0)]
    got, (mcode, masks, levels) = check_candidates(small)
    assert got == codec.encode_batch(mcode, masks, levels)
    # around encode_batch calls of other K: each call's results are its own
    b5 = codec.encode_batch(*_materialised(code, imp, [(k % 4, 0) for k in range(5)], None))
    pairs = [(2, 7), (0, 1), (1, 0), (3, 48), (0, 33), (2, 12), (3, 3), (1, 20), (0, 0)]
    got, mats = check_candidates(pairs)
    # the batch accessors return candidate j's streams, and -1 past J
    for j, (a, b) in enumerate(got):
        assert LIB.lic360_codec_batch_stream_size(codec._h, j, 1) == len(a)
        assert LIB.lic360_codec_batch_stream_size(codec._h, j, 0) == len(b)
    assert LIB.lic360_codec_batch_stream_size(codec._h, len(pairs), 0) == -1
    assert LIB.lic360_codec_batch_stream_size(codec._h, -1, 0) == -1
    b2 = codec.encode_batch(*_materialised(code, imp, [(3, 0), (1, 5)], None))
    assert got == codec.encode_batch(*mats)
    assert b5 == codec.encode_batch(*_materialised(code, imp, [(k % 4, 0) for k in range(5)], None))
    assert b2 == codec.encode_batch(*_materialised(code, imp, [(3, 0), (1, 5)], None))
    assert LIB.lic360_codec_batch_stream_size(codec._h, 2, 0) == -1  # the last encode had two latents


def test_encode_candidates_errors():
    H, W, K = 8, 16, 4
    codec = _codec("random", H, W)
    code, imp = _sources(K, H, W, 4500)
    imp[1] = 20  # source 1 has non-zero levels here
    bad_imp, bad_code = imp.clone(), code.clone()
    bad_imp[0, 0, 2, 3] = 60  # out of range until an offset of 12 brings it to 48
    lvl = 20
    bad_imp[3, 0, 0, 0] = lvl
    bad_code[3, 0, 0, 0] = 9  # out of range while its cell's level is above 0
    # lowered enough, both sources encode: a masked-out bad symbol is never reported
    ok_pairs = [(0, 12), (3, lvl), (1, 0)]
    got = codec.encode_candidates(bad_code, bad_imp, *_split(ok_pairs))
    assert got == codec.encode_batch(*_materialised(bad_code, bad_imp, ok_pairs, None))
    # the lowest bad candidate's message, as encode gives it for that candidate alone, with the suffix
    for pairs, j in (([(1, 0), (0, 12), (3, 0), (0, 0)], 2), ([(0, 30), (0, 0), (3, 0)], 1)):
        mcode, masks, levels = _materialised(bad_code, bad_imp, pairs[j:j + 1], None)
        with pytest.raises(RuntimeError) as alone:
            codec.encode(mcode, masks, levels)
        with pytest.raises(RuntimeError) as batch:
            codec.encode_candidates(bad_code, bad_imp, *_split(pairs))
        assert str(batch.value) == str(alone.value) + " (candidate %d)" % j
    # within a candidate, the importance stream's error comes first
    both = bad_code.clone()
    both[0, 5, 1, 1] = 9
    mcode, masks, levels = _materialised(both, bad_imp, [(0, 0)], None)
    with pytest.raises(RuntimeError) as alone:
        codec.encode(mcode, masks, levels)
    with pytest.raises(RuntimeError) as batch:
        codec.encode_candidates(both, bad_imp, [1, 0], [0, 0])
    assert str(batch.value) == str(alone.value) + " (candidate 1)"
    with pytest.raises(RuntimeError) as imp_alone:
        codec.encode(mcode, torch.zeros_like(masks), levels)
    assert str(alone.value) == str(imp_alone.value)
    # a failed call leaves no streams
    from lic360._lib import LIB
    assert LIB.lic360_codec_batch_stream_size(codec._h, 0, 0) == -1
    # argument errors
    for lat, off, match in (([], [], "J must be at least 1"), ([0, 4], [0, 0], r"cand_latent must lie in \[0, K\)"),
                            ([0, -1], [0, 0], r"cand_latent must lie"), ([0, 1], [0, -2], "offsets must not be negative"),
                            ([0, 1], [0], "2 latents for 1 offsets")):
        with pytest.raises(RuntimeError, match=match):
            codec.encode_candidates(code, imp, lat, off)
    with pytest.raises(RuntimeError):
        codec.encode_candidates(code, imp, [0], [0], protect=torch.zeros((K, 1, 2, 2), dtype=torch.int32, device=DEV))
    with pytest.raises(RuntimeError):
        codec.encode_candidates(code[:, :, :4], imp, [0], [0])
    assert codec.encode_candidates(code, imp, [3], [0]) == codec.encode_batch(*_materialised(code, imp, [(3, 0)], None))


# ---- the ladder --------------------------------------------------------------------------------------------------------------------
def _maker(kind):
    return lambda h, w: _pl().FusedCodec(_params(kind), H=h, W=w)


def _image(H, W, seed):
    q, m, lv = synthetic_latent(seed, H=H, W=W)
    return t(q, DEV), t(m, DEV), t(lv, DEV)


def _rung_budgets(tc, code, imap, protect, R):
    """R container budgets spread between the bound of the all-zero levels and that of offset 0"""
    pl, sh = _pl(), _sh()
    T = len(tc.tiles)
    top = 48 + (0 if protect is None else int(protect.max()))
    codes, imaps = sh.split_tiles(code, tc.rows, tc.cols), sh.split_tiles(imap, tc.rows, tc.cols)
    prot = None if protect is None else sh.split_tiles(protect, tc.rows, tc.cols)
    ests = tc.codecs[0].estimate_candidates(codes, imaps, list(range(T)) * 2, [0] * T + [top] * T, prot)
    head = sh.tile_header_bytes(T)
    lo, hi = head + sum(map(pl.budget_bound, ests[T:])), head + sum(map(pl.budget_bound, ests[:T]))
    return [lo + (hi - lo) * (R - r) // R for r in range(R)]


@pytest.mark.parametrize("with_protect", [False, True])
@pytest.mark.parametrize("rows,cols", [(2, 2), (4, 4)])
def test_budget_rungs_equal_encode_to_budget(rows, cols, with_protect):
    sh = _sh()
    H, W = 32, 64
    code, _, imap = _image(H, W, 4600 + rows)
    protect = _pl().view_protection(H // 2, W // 2, [0.0], [0.0], 0.4, 20, device=DEV) if with_protect else None
    tc = sh.TileCodec(_maker("random"), H, W, rows, cols)
    budgets = _rung_budgets(tc, code, imap, protect, 4)
    r = tc.encode_ladder(code, imap, budgets=budgets, protect=protect, max_batch=7)
    assert sorted(r) == ["bounds", "ladder", "offsets", "sizes"]
    rr, cc, hh, ww, offsets, _ = sh.unpack_ladder_streams(r["ladder"])
    assert (rr, cc, hh, ww, offsets) == (rows, cols, H, W, r["offsets"])
    for k, b in enumerate(budgets):
        want = tc.encode_to_budget(code, imap, b, protect=protect)
        cut = sh.ladder_to_tiles(r["ladder"], k)
        assert cut == want["container"], k
        assert r["offsets"][k] == want["offset"] and r["bounds"][k] == want["bounds"], k
        assert r["sizes"][k] == len(cut) <= b
    assert r["offsets"][0] == 0 < r["offsets"][-1]
    # the default max_batch gives the same ladder
    assert tc.encode_ladder(code, imap, budgets=budgets, protect=protect)["ladder"] == r["ladder"]


@pytest.mark.parametrize("kind", ["random", "P"])
def test_offset_rungs_equal_encode_of_the_materialised_candidates(kind):
    pl, sh = _pl(), _sh()
    H, W = 32, 64
    code, _, imap = _image(H, W, 4700)
    tc = sh.TileCodec(_maker(kind), H, W, 2, 4)
    protect = pl.latitude_protection(H // 2, W // 2, 30, DEV)
    for prot, offsets in ((None, [0, 9, 9, 30]), (protect, [70, 0, 55])):
        r = tc.encode_ladder(code, imap, offsets=offsets, protect=prot, max_batch=5)
        assert r["offsets"] == offsets and r["bounds"] is None
        for k, o in enumerate(offsets):
            levels, masks = pl.levels_to_mask(imap, [o], prot)
            want = tc.encode(code, masks, levels)
            assert sh.ladder_to_tiles(r["ladder"], k) == want, (k, o)
            assert r["sizes"][k] == len(want)


def test_mixed_cut_decodes_each_tile_at_its_rung():
    pl, sh = _pl(), _sh()
    H, W = 32, 64
    code, _, imap = _image(H, W, 4800)
    tc = sh.TileCodec(_maker("random"), H, W, 4, 4, in_flight=2)
    offsets = [0, 14, 40]
    r = tc.encode_ladder(code, imap, offsets=offsets)
    view = ([0.0], [0.0], 0.5)
    rungs = tc.rungs_for_views(*view, inside=0, outside=2)
    need = tc.tiles_for_views(*view)
    assert rungs == [0 if k in need else 2 for k in range(16)] and 0 < len(need) < 16
    cut = sh.ladder_to_tiles(r["ladder"], rungs)
    assert len(cut) < r["sizes"][0]
    masks = [pl.levels_to_mask(imap, [o])[1] for o in offsets]
    want_mask = torch.zeros_like(masks[0])
    for k, (r0, r1, c0, c1) in enumerate(tc.tiles):
        want_mask[:, :, r0:r1, c0:c1] = masks[rungs[k]][:, :, r0:r1, c0:c1]
    dcode, dmask = tc.decode(cut)
    assert torch.equal(dmask, want_mask) and torch.equal(dcode, code * want_mask)
    vcode, vmask, dec = tc.decode_views(cut, *view)
    assert torch.equal(vmask, want_mask * dec) and torch.equal(vcode, code * want_mask * dec)
    tcode, tmask, dec2 = tc.decode_tiles(cut, [k for k in range(16) if k not in need][:3])
    assert torch.equal(tmask, want_mask * dec2) and torch.equal(tcode, code * want_mask * dec2)


def test_encode_ladder_errors():
    pl, sh = _pl(), _sh()
    H, W = 16, 32
    code, _, imap = _image(H, W, 4900)
    tc = sh.TileCodec(_maker("random"), H, W, 2, 2)
    for kw in ({}, {"budgets": [10 ** 6], "offsets": [0]}, {"offsets": []}, {"offsets": [0, -1]}, {"offsets": [0], "max_batch": 0},
               {"offsets": [0], "protect": torch.zeros((1, 1, 4, 4), dtype=torch.int32, device=DEV)}):
        with pytest.raises(RuntimeError):
            tc.encode_ladder(code, imap, **kw)
    with pytest.raises(RuntimeError):
        tc.encode_ladder(code[:, :, :8], imap[:, :, :4], offsets=[0])
    with pytest.raises(RuntimeError, match="needs world == 1"):
        sh.TileCodec(_maker("random"), H, W, 2, 2, world=2, rank=0).encode_ladder(code, imap, offsets=[0])
    # the lowest rung no offset fits, with encode_to_budget's message
    head = sh.tile_header_bytes(4)
    with pytest.raises(RuntimeError) as alone:
        tc.encode_to_budget(code, imap, head + 10)
    with pytest.raises(RuntimeError) as ladder:
        tc.encode_ladder(code, imap, budgets=[10 ** 6, head + 10, head + 5])
    assert str(ladder.value) == str(alone.value) + " (rung 1)"
