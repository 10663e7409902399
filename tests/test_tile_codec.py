"""Tiled container and TileCodec (lic360_shard) on the CPU, and a float64 numpy restatement of the view-footprint predicate
(lic360_view_footprint) checked on hand-built cases.  The per-tile codec is the CPU rendition (oracle/cpu_codec.py), as in
tests/test_band_codec.py; tests/test_gpu_tile_codec.py runs the GPU codec and the footprint kernel against the restatement."""
import math
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_band_codec import _free_port
from util import synthetic_latent

H, W, ROWS, COLS = 8, 16, 2, 2


# ---- the footprint predicate, restated in numpy --------------------------------------------------------------------------------
def view_axes(theta, phi):
    """(f, r, u) of view (theta, phi) in units of pi: rotate about z by theta, then about the rotated y axis by -phi"""
    th, ph = theta * math.pi, phi * math.pi
    Rz = np.array([[math.cos(th), -math.sin(th), 0.0], [math.sin(th), math.cos(th), 0.0], [0.0, 0.0, 1.0]])
    a = Rz[:, 1]
    K = np.array([[0.0, -a[2], a[1]], [a[2], 0.0, -a[0]], [-a[1], a[0], 0.0]])
    R2 = np.eye(3) + math.sin(-ph) * K + (1 - math.cos(-ph)) * (K @ K)
    R = R2 @ Rz
    return R[:, 0], R[:, 1], R[:, 2]


def cell_bounds(h, w):
    """(lon0, lon1) per column and (lat0, lat1) per row of ProjectsOp's grid: x in [j-1/2, j+1/2], y in [i-1/2, i+1/2], clamped"""
    hx, hy = (w - 1) / 2.0, (h - 1) / 2.0
    j, i = np.arange(w, dtype=np.float64), np.arange(h, dtype=np.float64)
    lon0 = (np.maximum(j - 0.5, 0) - hx) / hx * math.pi
    lon1 = (np.minimum(j + 0.5, w - 1) - hx) / hx * math.pi
    lat1 = (hy - np.maximum(i - 0.5, 0)) / hy * (math.pi / 2)
    lat0 = (hy - np.minimum(i + 0.5, h - 1)) / hy * (math.pi / 2)
    return lon0, lon1, lat0, lat1


def _unit(lon, lat):
    return np.stack(np.broadcast_arrays(np.cos(lat) * np.cos(lon), np.cos(lat) * np.sin(lon), np.sin(lat)), -1)


def _lat(p):
    return np.arctan2(p[..., 2], np.hypot(p[..., 0], p[..., 1]))


def _lon_in(lon, lo, hi):
    c, hw = 0.5 * (lo + hi), 0.5 * (hi - lo)
    return np.abs(np.remainder(lon - c + math.pi, 2 * math.pi) - math.pi) <= hw


def footprint_parts(h, w, theta, phi, fov):
    f, r, u = view_axes(theta, phi)
    t = math.tan(fov * math.pi / 2)
    planes = np.stack([t * f - r, t * f + r, t * f - u, t * f + u])
    corners = np.stack([f - t * r - t * u, f + t * r - t * u, f + t * r + t * u, f - t * r + t * u])
    corners /= np.linalg.norm(corners, axis=1, keepdims=True)
    lon0, lon1, lat0, lat1 = cell_bounds(h, w)
    LO0, LA0 = np.meshgrid(lon0, lat0)
    LO1, LA1 = np.meshgrid(lon1, lat1)
    shape = (h, w)
    # 1. a cell corner in the field
    cc = np.stack([_unit(LO0, LA0), _unit(LO1, LA0), _unit(LO0, LA1), _unit(LO1, LA1)], -2)  # (h,w,4,3)
    corner_in = np.any(np.all(cc @ planes.T >= 0, -1), -1)
    # 2. a field corner in the cell
    field_in = np.zeros(shape, bool)
    for p in corners:
        la = _lat(p)
        rho = math.hypot(p[0], p[1])
        lon_ok = True if rho == 0 else _lon_in(math.atan2(p[1], p[0]), LO0, LO1)
        field_in |= (la >= LA0) & (la <= LA1) & lon_ok
    # 3. a field edge across a meridian or a parallel of the cell
    mer, par = np.zeros(shape, bool), np.zeros(shape, bool)
    for k in range(4):
        A, B = corners[k], corners[(k + 1) % 4]
        n = np.cross(A, B)

        def on_arc(p):
            return (np.cross(A, p) @ n >= 0) & (np.cross(p, B) @ n >= 0)

        for lon in (LO0, LO1):
            m = np.stack([-np.sin(lon), np.cos(lon), np.zeros_like(lon)], -1)
            q = np.cross(n, m)
            for s in (1.0, -1.0):
                p = s * q
                ok = p[..., 0] * np.cos(lon) + p[..., 1] * np.sin(lon) >= 0
                la = _lat(p)
                mer |= ok & (la >= LA0) & (la <= LA1) & on_arc(p)
        rho = math.hypot(n[0], n[1])
        if rho == 0:
            continue
        for lat in (LA0, LA1):
            s, c = np.sin(lat), np.cos(lat)
            along = -n[2] * s / rho
            disc = c * c - along * along
            perp = np.sqrt(np.maximum(disc, 0))
            for sg in (1.0, -1.0):
                tt = sg * perp
                p = np.stack([along * n[0] / rho - tt * n[1] / rho, along * n[1] / rho + tt * n[0] / rho, s], -1)
                ok = (disc >= 0) & (np.abs(lat) < math.pi / 2)
                par |= ok & _lon_in(np.arctan2(p[..., 1], p[..., 0]), LO0, LO1) & on_arc(p)
    return {"corner": corner_in, "field_corner": field_in, "meridian": mer, "parallel": par}


def footprint_np(h, w, theta, phi, fov):
    parts = footprint_parts(h, w, theta, phi, fov)
    return (parts["corner"] | parts["field_corner"] | parts["meridian"] | parts["parallel"]).astype(np.int32)


def sampled_cells(h, w, theta, phi, fov, n=401):
    """(h,w) bool: the cells hit by an n x n float64 sampling of the view's field, its boundary included"""
    f, r, u = view_axes(theta, phi)
    t = math.tan(fov * math.pi / 2)
    s = np.linspace(-t, t, n)
    a, b = np.meshgrid(s, s)
    d = f + a[..., None] * r + b[..., None] * u
    lon, lat = np.arctan2(d[..., 1], d[..., 0]), _lat(d)
    hx, hy = (w - 1) / 2.0, (h - 1) / 2.0
    j = np.clip(np.rint(lon / math.pi * hx + hx), 0, w - 1).astype(int)
    i = np.clip(np.rint(-2 * lat / math.pi * hy + hy), 0, h - 1).astype(int)
    out = np.zeros((h, w), bool)
    out[i, j] = True
    return out


def test_footprint_restatement_front_and_seam():
    h, w = 16, 32
    front = footprint_np(h, w, 0, 0, 0.5)
    assert np.array_equal(front, front[:, ::-1]) and np.array_equal(front, front[::-1])  # symmetric about lon 0 and the equator
    assert front[h // 2, w // 2] and not front[:, 0].any() and not front[0].any()
    back = footprint_np(h, w, 1, 0, 0.5)  # looks at the +-pi seam: both half columns, mirror images of each other
    assert back[h // 2, 0] and back[h // 2, w - 1] and np.array_equal(back, back[:, ::-1])
    assert not back[:, w // 2 - 2:w // 2 + 2].any()
    for th, ph, fov in ((0.3, 0.1, 0.4), (-0.7, -0.2, 0.3), (1.0, 0.05, 0.2)):
        fp = footprint_np(h, w, th, ph, fov)
        assert np.all(fp[sampled_cells(h, w, th, ph, fov)] == 1)


@pytest.mark.parametrize("phi,fov", [(0.5, 0.3), (0.4, 0.5), (-0.35, 0.5)])
def test_footprint_restatement_views_containing_a_pole(phi, fov):
    """a view that contains a pole touches every cell of that pole's row; the other pole's row stays clear"""
    h, w = 8, 16
    fp = footprint_np(h, w, 0.2, phi, fov)
    near, far = (0, h - 1) if phi > 0 else (h - 1, 0)
    assert fp[near].all() and not fp[far].any()
    assert np.all(fp[sampled_cells(h, w, 0.2, phi, fov)] == 1)


def test_footprint_restatement_view_below_a_pole():
    """a view that reaches high latitudes without the pole: part of the polar row only"""
    h, w = 8, 16
    fp = footprint_np(h, w, -0.5, 0.3, 0.35)
    assert fp[0].any() and not fp[0].all()
    assert np.all(fp[sampled_cells(h, w, -0.5, 0.3, 0.35)] == 1)


def test_footprint_restatement_parallel_only_crossing():
    """the field's top edge bulges into cell (5, 5) through the cell's lower parallel between its meridians: no corner of either lies
    in the other and no meridian is crossed, yet the cell is in the footprint, and a sample of the field lies in it"""
    h, w, th, ph, fov = 8, 16, -0.327, -0.013, 0.26
    parts = footprint_parts(h, w, th, ph, fov)
    assert parts["parallel"][5, 5] and not (parts["corner"][5, 5] or parts["field_corner"][5, 5] or parts["meridian"][5, 5])
    assert footprint_np(h, w, th, ph, fov)[5, 5] == 1
    assert sampled_cells(h, w, th, ph, fov, n=2001)[5, 5]


# ---- tile geometry and container ------------------------------------------------------------------------------------------------
def test_tile_geometry():
    import lic360_shard as sh
    assert sh.tile_grid(8, 16, 2, 2) == [(0, 4, 0, 8), (0, 4, 8, 16), (4, 8, 0, 8), (4, 8, 8, 16)]
    assert sh.tile_grid(256, 512, 4, 4)[5] == (64, 128, 128, 256)
    assert sh.tile_grid(8, 16, 1, 1) == [(0, 8, 0, 16)]
    for bad in ((8, 16, 0, 2), (8, 16, 2, 0), (8, 16, 3, 2), (8, 16, 8, 2), (8, 16, 2, 16), (12, 16, 4, 2), (0, 16, 1, 1)):
        with pytest.raises(ValueError):
            sh.tile_grid(*bad)
    x = torch.arange(2 * 8 * 16, dtype=torch.float32).reshape(1, 2, 8, 16)
    tiles = sh.split_tiles(x, 2, 4)
    assert tiles.shape == (8, 2, 4, 4)
    for k, (r0, r1, c0, c1) in enumerate(sh.tile_grid(8, 16, 2, 4)):
        assert torch.equal(tiles[k], x[0, :, r0:r1, c0:c1])


def test_tile_container():
    import lic360_shard as sh
    streams = [(b"ab", b"cde"), (b"", b"x"), (b"\x00" * 5, b""), (b"q", b"rs")]
    blob = sh.pack_tile_streams(2, 2, 8, 16, streams)
    assert blob[:4] == b"L3T1" and len(blob) == 20 + 8 * 4 + sum(len(a) + len(b) for a, b in streams)
    assert sh.unpack_tile_streams(blob) == (2, 2, 8, 16, streams)
    import struct
    bad_grid = blob[:4] + struct.pack("<IIII", 3, 2, 8, 16) + blob[20:]
    zero_grid = blob[:4] + struct.pack("<IIII", 0, 2, 8, 16) + blob[20:]
    huge_grid = blob[:4] + struct.pack("<IIII", 4, 8, 8, 16) + blob[20:]  # a valid grid whose header the blob cannot hold
    for broken in (blob[:-1], blob + b"z", b"XXXX" + blob[4:], sh.pack_band_streams(8, 16, streams), blob[:10], blob[:30],
                   bad_grid, zero_grid, huge_grid):
        with pytest.raises(ValueError):
            sh.unpack_tile_streams(broken)
    with pytest.raises(ValueError):
        sh.pack_tile_streams(2, 2, 8, 16, streams[:3])
    with pytest.raises(RuntimeError):
        sh.exchange_streams({0: (b"", b"")}, 2, "tile")


# ---- TileCodec with the CPU rendition -------------------------------------------------------------------------------------------
class _CpuTile(object):
    """CpuCodec behind FusedCodec's encode / decode signatures, on torch CPU tensors"""

    def __init__(self, h, w):
        import lic360_codec_ops as ops
        from oracle import cpu_codec
        params = {'code': ops.make_entropy_params(48, 4, 3, 3, 7, 'cpu'), 'imp': ops.make_entropy_params(1, 144, 49, None, 8, 'cpu')}
        self.h, self.w = h, w
        self.cd = cpu_codec.CpuCodec(cpu_codec.params_to_numpy(params))

    def encode(self, code, mask, imap):
        return self.cd.encode(*(np.ascontiguousarray(x.numpy()) for x in (code, mask, imap)))

    def decode(self, bi, bc):
        code, mask = self.cd.decode(bi, bc, self.h // 2, self.w // 2)
        return torch.from_numpy(np.ascontiguousarray(code)), torch.from_numpy(np.ascontiguousarray(mask))


def _inputs():
    q, mask, lv = synthetic_latent(654, H=H, W=W)
    return torch.from_numpy(q), torch.from_numpy(mask), torch.from_numpy(lv)


def test_tile_codec_single_process():
    """each tile's streams are the codec's for that tile as an image of its own; decode gives the image, decode_tiles the chosen
    tiles and zeros elsewhere"""
    import lic360_shard as sh
    q, mask, lv = _inputs()
    tc = sh.TileCodec(_CpuTile, H, W, ROWS, COLS, in_flight=2)
    blob = tc.encode(q, mask, lv)
    rows, cols, h, w, streams = sh.unpack_tile_streams(blob)
    assert (rows, cols, h, w, len(streams)) == (ROWS, COLS, H, W, ROWS * COLS)
    grid = sh.tile_grid(H, W, ROWS, COLS)
    for k, (r0, r1, c0, c1) in enumerate(grid):
        alone = _CpuTile(r1 - r0, c1 - c0).encode(q[:, :, r0:r1, c0:c1], mask[:, :, r0:r1, c0:c1], lv[:, :, r0 // 2:r1 // 2, c0 // 2:c1 // 2])
        assert streams[k] == alone
    code, m = tc.decode(blob)
    assert torch.equal(code, q * mask) and torch.equal(m, mask)
    for chosen in ([1], [0, 3], [2, 2, 1], []):
        c, mk, dec = tc.decode_tiles(blob, chosen)
        want = torch.zeros((1, 1, H, W), dtype=torch.int32)
        for k in set(chosen):
            r0, r1, c0, c1 = grid[k]
            want[:, :, r0:r1, c0:c1] = 1
        assert dec.dtype == torch.int32 and torch.equal(dec, want)
        assert torch.equal(c, code * want) and torch.equal(mk, m * want)
    with pytest.raises(ValueError):
        tc.decode_tiles(blob, [4])
    with pytest.raises(ValueError):
        sh.TileCodec(_CpuTile, H, W, 1, 2).decode(blob)  # another grid
    with pytest.raises(RuntimeError):
        tc.encode(q[:, :, :4], mask[:, :, :4], lv[:, :, :2])


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import lic360_shard as sh
        q, mask, lv = _inputs()
        tc = sh.TileCodec(_CpuTile, H, W, ROWS, COLS, world=world, rank=rank)
        blob = tc.encode(q, mask, lv)
        code, m = tc.decode(blob)
        c, mk, dec = tc.decode_tiles(blob, [1, 2])
        part = bool(torch.equal(c, q * mask * dec) and torch.equal(mk, mask * dec) and int(dec.sum()) == 2 * (H // ROWS) * (W // COLS))
        out.put((rank, tc.mine, blob, bool(torch.equal(code, q * mask) and torch.equal(m, mask)), part))
    finally:
        dist.destroy_process_group()


def test_tile_codec_two_ranks_gloo():
    """world_size 2: tiles dealt round-robin; both ranks hold the single-process container, the image, and any subset of tiles"""
    import lic360_shard as sh
    q, mask, lv = _inputs()
    ref_blob = sh.TileCodec(_CpuTile, H, W, ROWS, COLS).encode(q, mask, lv)
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(out.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert [r[1] for r in res] == [[0, 2], [1, 3]]
    assert all(r[2] == ref_blob and r[3] and r[4] for r in res)
