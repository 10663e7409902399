"""GPU: the view-footprint kernel (lic360_view_footprint) against the float64 numpy restatement, dense sampling and
viewport_protection, and TileCodec on FusedCodec: per-tile parity with single-tile encodes, view decodes, budgets and errors."""
import functools
import math

import numpy as np
import pytest
import torch

import probe_nets as pn
from test_tile_codec import footprint_np, sampled_cells
from util import n, synthetic_latent, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _pl():
    import lic360_pipeline as pl
    return pl


def _sh():
    import lic360_shard as sh
    return sh


def _views(seed, count):
    """random views as float32 values, the precision the kernel takes them in: any direction, fov in (0.05, 0.95)"""
    r = np.random.default_rng(seed)
    th = r.uniform(-1, 1, count).astype(np.float32)
    ph = r.uniform(-0.5, 0.5, count).astype(np.float32)
    fov = r.uniform(0.05, 0.95, count).astype(np.float32)
    extra = [(1.0, 0.0, 0.5), (-1.0, 0.1, 0.3), (0.0, 0.5, 0.4), (0.3, -0.42, 0.5), (0.25, 0.3, 0.35)]  # seam, poles
    th = np.concatenate([th, np.float32([e[0] for e in extra])])
    ph = np.concatenate([ph, np.float32([e[1] for e in extra])])
    fov = np.concatenate([fov, np.float32([e[2] for e in extra])])
    return [float(x) for x in th], [float(x) for x in ph], [float(x) for x in fov]


@pytest.mark.parametrize("h,w", [(8, 16), (16, 32), (32, 64), (64, 128), (128, 256)])
def test_footprint_equals_restatement(h, w):
    """equal to the restatement except where the field's boundary passes within 1e-9 rad of a cell: there the kernel's answer lies
    between the restatement's for the field shrunk and grown by 1e-9 rad"""
    th, ph, fov = _views(100 + h, 27)  # 32 views: two launches of the kernel
    got = n(_pl().view_footprint(h, w, th, ph, fov, DEV))
    assert got.shape == (len(th), 1, h, w) and got.dtype == np.int32
    eps = 2e-9 / math.pi  # 1e-9 rad of half-angle, in units of pi of fov
    for v in range(len(th)):
        lo = footprint_np(h, w, th[v], ph[v], fov[v] - eps)
        hi = footprint_np(h, w, th[v], ph[v], fov[v] + eps)
        g = got[v, 0]
        assert np.all(lo <= g) and np.all(g <= hi), "view %d (%r, %r, %r): %d cells below, %d above" % (
            v, th[v], ph[v], fov[v], int((lo > g).sum()), int((g > hi).sum()))
        assert np.array_equal(g, footprint_np(h, w, th[v], ph[v], fov[v])) or np.any(lo != hi)


@pytest.mark.parametrize("h,w", [(16, 32), (64, 128)])
def test_footprint_has_no_misses(h, w):
    th, ph, fov = _views(300 + h, 11)
    got = n(_pl().view_footprint(h, w, th, ph, fov, DEV))
    for v in range(len(th)):
        hit = sampled_cells(h, w, th[v], ph[v], fov[v], n=601)
        assert np.all(got[v, 0][hit] == 1), "view %d: %d sampled cells missing" % (v, int((got[v, 0][hit] == 0).sum()))


def _dilate1(x):
    """(1,1,h,w) 0/1 -> dilated by one cell, longitude wrapping"""
    wide = torch.nn.functional.pad(x.float(), (1, 1, 0, 0), mode="circular")
    return torch.nn.functional.max_pool2d(wide, 3, stride=1, padding=(1, 0)).to(torch.int32)


@pytest.mark.parametrize("h,w", [(16, 32), (32, 64), (64, 128)])
def test_footprint_within_viewport_protection(h, w):
    """MultiProject's 14 views: footprint <= viewport_protection <= footprint dilated by one cell, view by view"""
    from lic360_operator._modules import VIEWPORT_PHIS, VIEWPORT_THETAS
    pl = _pl()
    fp = pl.view_footprint(h, w, VIEWPORT_THETAS, VIEWPORT_PHIS, 0.6, DEV)
    for v in range(len(VIEWPORT_THETAS)):
        vp = pl.viewport_protection(h, w, [v], 1, fov=0.6, device=DEV)
        f = fp[v:v + 1]
        assert torch.all(f <= vp), "view %d: %d footprint cells outside viewport_protection" % (v, int((f > vp).sum()))
        d = _dilate1(f)
        assert torch.all(vp <= d), "view %d: %d protected cells beyond the dilated footprint" % (v, int((vp > d).sum()))


def test_view_protection_and_errors():
    pl = _pl()
    h, w = 16, 32
    th, ph = [0.9, 0.0], [0.0, 0.5]
    fp = pl.view_footprint(h, w, th, ph, 0.3, DEV)
    p0 = pl.view_protection(h, w, th, ph, 0.3, 20, device=DEV)
    assert p0.shape == (1, 1, h, w) and p0.dtype == torch.int32
    assert torch.equal(p0, fp.amax(dim=0, keepdim=True) * 20)
    p2 = pl.view_protection(h, w, th, ph, 0.3, 20, margin=2, device=DEV)
    want = fp.amax(dim=0, keepdim=True)
    for _ in range(2):
        want = _dilate1(want)
    assert torch.equal(p2, want * 20)
    assert p0[0, 0, 8, 0] == 20 and p0[0, 0, 8, w - 1] == 20  # theta 0.9 reaches across the seam
    assert torch.equal(pl.view_protection(h, w, [0.0], [0.0], 0.3, 1, margin=100, device=DEV), torch.ones((1, 1, h, w), dtype=torch.int32,
                                                                                                           device=DEV))
    for args in ((15, 32, [0.0], [0.0], 0.3), (16, 0, [0.0], [0.0], 0.3), (16, 32, [0.0], [0.0], 0.0), (16, 32, [0.0], [0.0], 1.0),
                 (16, 32, [float("nan")], [0.0], 0.3), (16, 32, [0.0], [float("inf")], 0.3), (16, 32, [], [], 0.3),
                 (16, 32, [0.0], [0.0, 0.1], 0.3), (16, 32, [0.0, 0.1], [0.0, 0.1], [0.3])):
        with pytest.raises(RuntimeError):
            pl.view_footprint(*args, device=DEV)
    with pytest.raises(RuntimeError, match="CUDA"):
        pl.view_footprint(16, 32, [0.0], [0.0], 0.3, device="cpu")
    for bad in (dict(levels=49), dict(margin=-1), dict(margin=1.5)):
        kw = dict(levels=8, margin=0)
        kw.update(bad)
        with pytest.raises(RuntimeError):
            pl.view_protection(16, 32, [0.0], [0.0], 0.3, kw["levels"], margin=kw["margin"], device=DEV)


# ---- TileCodec on the GPU --------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _params(kind):
    return _pl().make_codec_params(DEV, seed=2500) if kind == "random" else pn.to_torch(pn.probe_params(kind), DEV)


def _maker(kind):
    return lambda h, w: _pl().FusedCodec(_params(kind), H=h, W=w)


def _latent(H, W, seed):
    q, m, lv = synthetic_latent(seed, H=H, W=W)
    return t(q, DEV), t(m, DEV), t(lv, DEV)


@pytest.mark.parametrize("rows,cols", [(1, 1), (2, 2), (4, 4), (2, 4)])
@pytest.mark.parametrize("kind", ["random", "P"])
def test_tile_encode_parity_and_decode(kind, rows, cols):
    sh = _sh()
    H, W = 32, 64
    q, m, lv = _latent(H, W, 2600 + rows * 10 + cols)
    tc = sh.TileCodec(_maker(kind), H, W, rows, cols)
    blob = tc.encode(q, m, lv)
    _, _, _, _, streams = sh.unpack_tile_streams(blob)
    alone = tc.codecs[0]
    for k, (r0, r1, c0, c1) in enumerate(sh.tile_grid(H, W, rows, cols)):
        want = alone.encode(q[:, :, r0:r1, c0:c1].contiguous(), m[:, :, r0:r1, c0:c1].contiguous(),
                            lv[:, :, r0 // 2:r1 // 2, c0 // 2:c1 // 2].contiguous())
        assert streams[k] == want, "tile %d" % k
    code, mask = tc.decode(blob)
    assert torch.equal(mask, m) and torch.equal(code, q * m)


def _view_case():
    sh = _sh()
    H, W = 32, 64
    q, m, lv = _latent(H, W, 2700)
    return sh, H, W, q, m, lv


@pytest.mark.parametrize("in_flight", [1, 4])
def test_decode_views(in_flight):
    sh, H, W, q, m, lv = _view_case()
    tc = sh.TileCodec(_maker("random"), H, W, 4, 4, in_flight=in_flight)
    assert len(tc.codecs) == in_flight
    blob = tc.encode(q, m, lv)
    full_code, full_mask = tc.decode(blob)
    grid = sh.tile_grid(H, W, 4, 4)
    for views, margin in ((([0.0], [0.0], 0.5), 0), (([0.0], [0.5], 0.4), 0), (([1.0], [0.1], 0.3), 1), (([-0.5, 0.5], [0.25, -0.25], 0.3), 2)):
        tiles = tc.tiles_for_views(*views, margin=margin)
        fp = _pl().view_protection(H // 2, W // 2, *views, 1, margin=margin, device=DEV)
        want = [k for k, (r0, r1, c0, c1) in enumerate(grid) if fp[0, 0, r0 // 2:r1 // 2, c0 // 2:c1 // 2].any()]
        assert tiles == want and 0 < len(tiles) < 16
        code, mask, dec = tc.decode_views(blob, *views, margin=margin)
        marked = torch.zeros((1, 1, H, W), dtype=torch.int32, device=DEV)
        for k in tiles:
            r0, r1, c0, c1 = grid[k]
            marked[:, :, r0:r1, c0:c1] = 1
        assert torch.equal(dec, marked)
        assert torch.equal(code, full_code * dec) and torch.equal(mask, full_mask * dec)
    north = tc.tiles_for_views([0.0], [0.5], 0.25)  # reaches down to latitude 59.6 degrees, inside the top row of tiles (48 and up)
    assert north == [0, 1, 2, 3], north


def test_tile_budgets():
    sh, H, W, q, m, lv = _view_case()
    tc = sh.TileCodec(_maker("random"), H, W, 2, 4)
    full = tc.encode(q, m, lv)
    head = sh.tile_header_bytes(8)
    for budget in (len(full) // 2, len(full) // 4):
        r = tc.encode_to_budget(q, lv, budget)
        assert len(r["container"]) <= budget and r["bound"] <= budget and r["offset"] > 0
        code, mask = tc.decode(r["container"])
        for k, (r0, r1, c0, c1) in enumerate(sh.tile_grid(H, W, 2, 4)):
            x = r["results"][k]
            assert torch.equal(mask[:, :, r0:r1, c0:c1], x["mask"]), "tile %d" % k
            assert torch.equal(code[:, :, r0:r1, c0:c1], q[:, :, r0:r1, c0:c1] * x["mask"])
    front = tc.tiles_for_views([0.0], [0.0], 0.4)
    _, _, _, _, streams = sh.unpack_tile_streams(full)
    budgets = [len(a) + len(b) if k in front else (len(a) + len(b)) // 3 for k, (a, b) in enumerate(streams)]
    r = tc.encode_to_budget(q, lv, budgets, protect=_pl().view_protection(H // 2, W // 2, [0.0], [0.0], 0.4, 48, device=DEV))
    _, _, _, _, got = sh.unpack_tile_streams(r["container"])
    assert len(r["container"]) == head + sum(len(a) + len(b) for a, b in got)
    for k, (a, b) in enumerate(got):
        assert len(a) + len(b) <= budgets[k]
        assert r["offsets"][k] == r["results"][k]["offset"]
    code, mask = tc.decode(r["container"])
    for k, (r0, r1, c0, c1) in enumerate(sh.tile_grid(H, W, 2, 4)):
        assert torch.equal(mask[:, :, r0:r1, c0:c1], r["results"][k]["mask"])
    with pytest.raises(RuntimeError):
        tc.encode_to_budget(q, lv, budgets[:3])
    with pytest.raises(RuntimeError):
        tc.encode_to_budget(q, lv, head + 10)


def test_tile_codec_errors():
    sh, H, W, q, m, lv = _view_case()
    with pytest.raises(ValueError):
        sh.TileCodec(_maker("random"), H, W, 3, 4)
    tc = sh.TileCodec(_maker("random"), H, W, 2, 2)
    with pytest.raises(RuntimeError):
        tc.encode(q[:, :, :16], m[:, :, :16], lv[:, :, :8])
    with pytest.raises(RuntimeError):
        tc.encode_to_budget(q, lv, 10 ** 6, protect=torch.zeros((1, 1, 4, 4), dtype=torch.int32, device=DEV))
    blob = tc.encode(q, m, lv)
    for bad in (blob[:-1], b"L3B1" + blob[4:]):
        with pytest.raises(ValueError):
            tc.decode(bad)
    with pytest.raises(ValueError):
        sh.TileCodec(_maker("random"), H, W, 1, 2).decode(blob)
    with pytest.raises(ValueError):
        tc.decode_tiles(blob, [-1])
    with pytest.raises(RuntimeError):
        tc.decode_views(blob, [0.0], [0.0], 1.5)
    with pytest.raises(RuntimeError):
        sh.TileCodec(_maker("random"), H, W, 2, 2, world=2, rank=0).encode_to_budget(q, lv, 10 ** 6)
