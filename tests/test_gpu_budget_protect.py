"""GPU: protection maps for rate control.  levels_to_mask with a map (lic360_imp_levels_to_mask_protected) against a numpy
restatement; FusedCodec.encode_to_budget with latitude and viewport maps; the footprint of viewport_protection against the view's
cone; the argument checks."""
import functools
import math

import numpy as np
import pytest
import torch

from test_gpu_estimate_batch import _np_levels_to_mask
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


def _np_protected(lv, P, k):
    """numpy restatement: level max(s - max(k - P, 0), 0) with P clamped to [0, 48], and the decoder's mask of it"""
    drop = np.maximum(k - np.clip(P, 0, 48), 0)
    L = np.maximum(np.trunc(lv).astype(np.int64) - drop, 0)
    return _np_levels_to_mask(L, 0)


def _random_protect(h, w, seed):
    P = np.random.default_rng(seed).integers(0, 49, size=(1, 1, h, w)).astype(np.int32)
    P[0, 0, 0, :3] = (0, 48, 17)
    return P


def test_protected_levels_match_numpy_and_the_semantics():
    pl = _pl()
    H, W = 12, 40
    q, mask, lv = synthetic_latent(2100, H=H, W=W)
    P = _random_protect(H // 2, W // 2, 2101)
    top = 48 + int(P.max())
    offsets = list(range(top + 1))  # 97 candidates: four launches of the kernel
    levels, masks = pl.levels_to_mask(t(lv, DEV), offsets, torch.from_numpy(P).to(DEV))
    assert levels.shape == (top + 1, 1, H // 2, W // 2) and masks.shape == (top + 1, 48, H, W)
    L, M = n(levels), n(masks)
    for k in (0, 1, 7, 48, top):
        wl, wm = _np_protected(lv, P, k)
        assert np.array_equal(L[k:k + 1], wl), k
        assert np.array_equal(M[k:k + 1], wm), k
    assert np.array_equal(L[0:1], lv) and np.array_equal(M[0:1], mask), "t = 0 is the input"
    assert L[top].sum() == 0 and M[top].sum() == 0, "t = 48 + max P lowers every level to 0"
    assert np.all(M[1:] <= M[:-1]) and np.all(L[1:] <= L[:-1]), "candidates are nested in t"
    # more protection never means a lower level among cells with the same symbol
    s, p = lv[0, 0].ravel(), P[0, 0].ravel()
    for k in range(top + 1):
        lk = L[k, 0].ravel()
        for sym in np.unique(s):
            idx = np.flatnonzero(s == sym)
            order = idx[np.argsort(p[idx], kind="stable")]
            assert np.all(np.diff(lk[order]) >= 0), (k, sym)


def test_zero_and_constant_maps_are_the_uniform_candidates():
    pl = _pl()
    H, W = 16, 48
    _, _, lv = synthetic_latent(2200, H=H, W=W)
    tl = t(lv, DEV)
    offsets = [0, 1, 5, 8, 31, 48, 60]
    want = pl.levels_to_mask(tl, offsets)
    for zero in (torch.zeros((1, 1, H // 2, W // 2), dtype=torch.int32, device=DEV),
                 torch.zeros((1, 1, H // 2, W // 2), dtype=torch.int64, device=DEV)):
        got = pl.levels_to_mask(tl, offsets, zero)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), "a zero map is protect=None bit for bit"
    for c in (1, 7, 48):
        const = torch.full((1, 1, H // 2, W // 2), c, dtype=torch.int32, device=DEV)
        got = pl.levels_to_mask(tl, offsets, const)
        uni = pl.levels_to_mask(tl, [max(k - c, 0) for k in offsets])
        assert torch.equal(got[0], uni[0]) and torch.equal(got[1], uni[1]), c


@functools.lru_cache(maxsize=None)
def _protected_case(kind):
    """a 16x48 latent, its protection map and the bounds of every candidate t = 0 .. 48 + max P, computed once"""
    pl = _pl()
    H, W = 16, 48
    q, mask, lv = synthetic_latent(2300, H=H, W=W)
    codec = _codec(H, W)
    if kind == "latitude":
        P = pl.latitude_protection(H // 2, W // 2, 16, DEV)
    elif kind == "front":
        P = pl.viewport_protection(H // 2, W // 2, [1], 48, device=DEV)
    else:
        P = torch.zeros((1, 1, H // 2, W // 2), dtype=torch.int32, device=DEV)
    assert kind == "zero" or int(P.min()) < int(P.max()), "a map that protects some cells more than others"
    offsets = list(range(48 + int(P.max()) + 1))
    levels, masks = pl.levels_to_mask(t(lv, DEV), offsets, P)
    ests = codec.estimate_batch(t(q, DEV).expand(len(offsets), -1, -1, -1), masks, levels, maps=False)
    return codec, q, lv, P, {k: pl.budget_bound(e) for k, e in zip(offsets, ests)}


def _check_protected_budget(kind, budget):
    pl = _pl()
    codec, q, lv, P, all_bounds = _protected_case(kind)
    r = codec.encode_to_budget(t(q, DEV), t(lv, DEV), budget, protect=P)
    total = len(r["imp_bytes"]) + len(r["code_bytes"])
    assert total <= r["bound"] <= budget, (total, r["bound"], budget)
    assert max(r["bounds"]) == 48 + int(P.max())
    assert r["bounds"] == {k: all_bounds[k] for k in r["bounds"]}, "bounds of the evaluated offsets"
    assert r["offset"] == min(k for k, b in r["bounds"].items() if b <= budget), "the smallest evaluated offset that fits"
    levels, masks = pl.levels_to_mask(t(lv, DEV), [r["offset"]], P)
    assert torch.equal(r["levels"], levels) and torch.equal(r["mask"], masks)
    assert (r["imp_bytes"], r["code_bytes"]) == codec.encode(t(q, DEV), masks, levels)
    code, mup = codec.decode(r["imp_bytes"], r["code_bytes"])
    assert np.array_equal(n(mup), n(masks)) and np.array_equal(n(code), q * n(masks))
    return r


@pytest.mark.parametrize("kind", ["latitude", "front"])
def test_protected_budget_encodes(kind):
    codec, q, lv, P, bounds = _protected_case(kind)
    top = 48 + int(P.max())
    assert bounds[top] < bounds[0]
    r = _check_protected_budget(kind, bounds[0])
    assert r["offset"] == 0
    r = _check_protected_budget(kind, (bounds[0] + bounds[top]) // 2)
    assert 0 < r["offset"] < top
    _check_protected_budget(kind, bounds[top] + 1)
    _check_protected_budget(kind, bounds[top])
    with pytest.raises(RuntimeError, match="no level offset up to %d" % top):
        codec.encode_to_budget(t(q, DEV), t(lv, DEV), min(bounds.values()) - 1, protect=P)


def test_zero_map_budget_is_the_uniform_budget():
    codec, q, lv, P, bounds = _protected_case("zero")
    for budget in (bounds[0], (bounds[0] + bounds[48]) // 2, bounds[48] + 1):
        want = codec.encode_to_budget(t(q, DEV), t(lv, DEV), budget)
        got = codec.encode_to_budget(t(q, DEV), t(lv, DEV), budget, protect=P)
        assert sorted(got) == sorted(want)
        for key in want:
            same = torch.equal(got[key], want[key]) if isinstance(want[key], torch.Tensor) else got[key] == want[key]
            assert same, (budget, key)


def _cell_angles(h, w, view):
    """angle between each cell centre and the direction of viewport `view`, from MultiProject's theta / phi list"""
    from lic360_operator._modules import VIEWPORT_PHIS, VIEWPORT_THETAS
    th, ph = VIEWPORT_THETAS[view] * math.pi, VIEWPORT_PHIS[view] * math.pi
    d = np.array([math.cos(ph) * math.cos(th), math.cos(ph) * math.sin(th), math.sin(ph)])
    lat = math.pi / 2 - math.pi * (np.arange(h) + 0.5) / h
    lon = -math.pi + 2 * math.pi * (np.arange(w) + 0.5) / w
    la, lo = np.meshgrid(lat, lon, indexing="ij")
    c = np.stack([np.cos(la) * np.cos(lo), np.cos(la) * np.sin(lo), np.sin(la)], -1)
    return np.arccos(np.clip(c @ d, -1.0, 1.0))


@pytest.mark.parametrize("h,w", [(16, 32), (32, 64), (64, 128)])
@pytest.mark.parametrize("view", [1, 2, 12])  # front, side, north pole
def test_viewport_footprint_is_the_views_cone(view, h, w):
    pl = _pl()
    fov = 0.6
    p = pl.viewport_protection(h, w, [view], 9, fov=fov, device=DEV)
    assert p.shape == (1, 1, h, w) and p.dtype == torch.int32 and p.device == torch.device(DEV)
    got = n(p)[0, 0]
    assert set(np.unique(got)) <= {0, 9}
    ang = _cell_angles(h, w, view)
    a = fov * math.pi / 2  # half-fov of the square viewport, both axes
    tol = math.hypot(2 * math.pi / w, math.pi / h)  # one cell's largest angular extent (a cell on the equator, corner to corner)
    inside = ang < a - tol
    assert inside.any() and np.all(got[inside] == 9), "cells inside the cone: %s" % np.argwhere(inside & (got == 0))[:5].tolist()
    outside = ang > math.atan(math.sqrt(2 * math.tan(a) ** 2)) + tol
    assert outside.any() and np.all(got[outside] == 0), "cells beyond the corners: %s" % np.argwhere(outside & (got > 0))[:5].tolist()


def test_viewport_maps_combine():
    pl = _pl()
    front = pl.viewport_protection(16, 32, [1], 48, device=DEV)
    both = pl.viewport_protection(16, 32, [1, 12], 48, device=DEV)
    north = pl.viewport_protection(16, 32, [12], 48, device=DEV)
    assert torch.equal(both, torch.maximum(front, north))
    lat = pl.latitude_protection(16, 32, 16, DEV)
    assert torch.equal(torch.maximum(front, lat), torch.where(front > 0, front, lat))
    for views, levels in (([], 48), ([14], 48), ([1], 49)):
        with pytest.raises(RuntimeError):
            pl.viewport_protection(16, 32, views, levels, device=DEV)
    with pytest.raises(RuntimeError, match="CUDA"):
        pl.viewport_protection(16, 32, [1], 48, device="cpu")


def test_bad_protect_maps_are_refused():
    pl = _pl()
    H, W = 8, 16
    q, _, lv = synthetic_latent(2400, H=H, W=W)
    tl, tq = t(lv, DEV), t(q, DEV)
    good = torch.zeros((1, 1, H // 2, W // 2), dtype=torch.int32, device=DEV)
    high, low = good.clone(), good.clone()
    high[0, 0, 1, 2], low[0, 0, 3, 1] = 49, -1
    for bad in (good.float(), good[:, :, :, :-1], good[0], good.cpu(), good.bool(), high, low):
        with pytest.raises(RuntimeError, match="protect"):
            pl.levels_to_mask(tl, [0, 3], bad)
        with pytest.raises(RuntimeError, match="protect"):
            _codec(H, W).encode_to_budget(tq, tl, 10 ** 6, protect=bad)
    assert _codec(H, W).encode_to_budget(tq, tl, 10 ** 6, protect=good)["offset"] == 0
