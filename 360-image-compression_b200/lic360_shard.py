"""Image-level sharding of the codec path across the GPUs of one box (SURVEY.md s8e: every image has its own two
bitstreams, coder state and wavefront, so the path partitions by image with NO data-path collective).

One process per GPU (torchrun / mp.spawn, like the reference's trainers, train/trainDDP_IMP_ENT.py:105-108); the only
cross-rank traffic is bookkeeping: the max-over-ranks step time and the gathered stream sizes.  Used by bench.py
(NCCL on the GPU box) and covered by a world_size-2 gloo test on CPU (tests/test_shard_gloo.py).
"""
import torch
import torch.distributed as dist


def rank_images(n_images, world, rank):
    """Indices of the images rank `rank` codes: contiguous blocks, remainder to the first ranks (16 images over
    1/2/4/8 GPUs -> 16/8/4/2 per GPU, BASELINE.json configs[2])."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("rank_images: bad world/rank %r/%r" % (world, rank))
    base, rem = divmod(int(n_images), world)
    start = rank * base + min(rank, rem)
    return list(range(start, start + base + (1 if rank < rem else 0)))


def max_over_ranks(value, device="cpu"):
    """Step time as the driver wants it: the slowest rank's."""
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_stream_sizes(local, n_images, device="cpu"):
    """local: {image index: (imp_bytes, code_bytes)} of this rank -> the full table on every rank.
    Each image must be reported by exactly one rank (checked)."""
    tab = torch.zeros((n_images, 3), dtype=torch.int64, device=device)
    for i, (a, b) in local.items():
        tab[i, 0] = int(a)
        tab[i, 1] = int(b)
        tab[i, 2] = 1
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(tab, op=dist.ReduceOp.SUM)
    owners = tab[:, 2].tolist()
    if any(o != 1 for o in owners):
        raise RuntimeError("gather_stream_sizes: images coded by %s ranks (expected exactly one each)" % owners)
    return [(int(a), int(b)) for a, b, _ in tab.tolist()]


# ---------------------------------------------------------------------------------------------------------------------
# Latitude bands of ONE image (BASELINE.json configs[3], SURVEY.md s8e option 3).
#
# Inside one image the wavefront is strictly sequential and the reference's bitstream is ONE arithmetic-coded stream per
# network, so a single image does not shard in the reference's format ("replicas only").  What does shard is a FORMAT
# EXTENSION: the latent is cut into `nbands` horizontal (latitude) bands and every band is coded as an independent
# sub-image with its own two bitstreams -- the context of a band's first rows is the zero padding an image border has.
# Every band is exactly what the reference produces when the band is handed to it as an image of its own (that is the
# parity statement, per band); the total size differs from the single-stream size by the context lost at the band edges.
# Bands are dealt to the ranks round-robin; the codec path has no collective, the ranks only exchange the finished byte
# strings (encode) and the decoded rows (decode) -- assembly, not coding.
# ---------------------------------------------------------------------------------------------------------------------
import struct

BAND_MAGIC = b"L3B1"


def band_rows(H, nbands):
    """Row ranges [r0, r1) of the bands of an H-row latent.  Rows come in pairs (one importance row covers two latent
    rows), so H / nbands must be an even integer."""
    if nbands < 1 or H % nbands or (H // nbands) % 2:
        raise ValueError("band_rows: %d rows do not split into %d bands of an even number of rows" % (H, nbands))
    hb = H // nbands
    return [(b * hb, (b + 1) * hb) for b in range(nbands)]


def rank_bands(nbands, world, rank):
    """Bands (or tiles) of rank `rank`: round-robin, so that neighbouring parts (similar content, similar cost) land on different GPUs."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("rank_bands: bad world/rank %r/%r" % (world, rank))
    return list(range(rank, nbands, world))


def split_bands(code, mask, imap, nbands):
    """(1,C,H,W) code and mask, (1,1,H/2,W/2) importance levels -> per band (code_b, mask_b, imap_b), contiguous copies."""
    H = code.shape[2]
    out = []
    for r0, r1 in band_rows(H, nbands):
        out.append((code[:, :, r0:r1].contiguous(), mask[:, :, r0:r1].contiguous(), imap[:, :, r0 // 2:r1 // 2].contiguous()))
    return out


def pack_band_streams(H, W, streams):
    """streams: [(imp_bytes, code_bytes)] in band order -> one container: magic, nbands, H, W, the 2*nbands lengths, the payloads."""
    head = BAND_MAGIC + struct.pack("<III", len(streams), H, W)
    head += b"".join(struct.pack("<II", len(a), len(b)) for a, b in streams)
    return head + b"".join(a + b for a, b in streams)


def unpack_band_streams(blob):
    """-> (H, W, [(imp_bytes, code_bytes)]); raises ValueError on a malformed container."""
    if len(blob) < 16 or blob[:4] != BAND_MAGIC:
        raise ValueError("unpack_band_streams: not a band container")
    nb, H, W = struct.unpack_from("<III", blob, 4)
    off = 16 + 8 * nb
    if nb < 1 or len(blob) < off:
        raise ValueError("unpack_band_streams: truncated header")
    lens = [struct.unpack_from("<II", blob, 16 + 8 * b) for b in range(nb)]
    if off + sum(a + b for a, b in lens) != len(blob):
        raise ValueError("unpack_band_streams: payload size does not match the header")
    out = []
    for a, b in lens:
        out.append((bytes(blob[off:off + a]), bytes(blob[off + a:off + a + b])))
        off += a + b
    return H, W, out


def exchange_streams(local, nparts, kind="band"):
    """local: {part: (imp_bytes, code_bytes)} of this rank -> the full list on every rank (bookkeeping traffic only)."""
    table = dict(local)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        parts = [None] * dist.get_world_size()
        dist.all_gather_object(parts, local)
        table = {}
        for p in parts:
            for k, v in p.items():
                if k in table:
                    raise RuntimeError("exchange_%s_streams: %s %d coded by two ranks" % (kind, kind, k))
                table[k] = v
    if sorted(table) != list(range(nparts)):
        raise RuntimeError("exchange_%s_streams: %ss %s of %d present" % (kind, kind, sorted(table), nparts))
    return [table[b] for b in range(nparts)]


def exchange_band_streams(local, nbands):
    return exchange_streams(local, nbands, "band")


class _PartCodec(object):
    """What BandCodec and TileCodec share: the parts dealt round-robin to the ranks (rank_bands), `in_flight` codecs of the part size
    with one worker thread each, and the exchange of decoded parts between ranks."""

    def __init__(self, make_codec, part_hw, nparts, world, rank, in_flight):
        self.world, self.rank = world, rank
        self.mine = rank_bands(nparts, world, rank)
        self.codecs = [make_codec(*part_hw) for _ in range(max(1, min(in_flight, len(self.mine))))]

    def _map(self, fn, items):
        """fn(codec, item) over this rank's items, one worker thread per codec (each codec = one part in flight)."""
        if len(self.codecs) == 1 or len(items) <= 1:
            return [fn(self.codecs[0], it) for it in items]
        import threading
        out, errs, lock, nxt = [None] * len(items), [], threading.Lock(), [0]

        def worker(cd):
            while True:
                with lock:
                    i = nxt[0]
                    nxt[0] += 1
                if i >= len(items):
                    return
                try:
                    out[i] = fn(cd, items[i])
                except Exception as e:  # noqa: BLE001 -- re-raised below
                    errs.append(e)
                    return

        th = [threading.Thread(target=worker, args=(cd,)) for cd in self.codecs[:len(items)]]
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        return out

    def _gather(self, local):
        """{part: (code_p, mask_p)} decoded by this rank -> the parts decoded by every rank (assembly, not coding)."""
        if not (self.world > 1 and dist.is_available() and dist.is_initialized()):
            return local
        parts = [None] * self.world
        dist.all_gather_object(parts, {b: (c.cpu(), m.cpu()) if hasattr(c, "cpu") else (c, m) for b, (c, m) in local.items()})
        table = {}
        for p in parts:
            table.update(p)
        return table


class BandCodec(_PartCodec):
    """One image as `nbands` independently coded latitude bands, dealt round-robin to the ranks of the process group (or all on
    this process without one).  `make_codec(h, w)` builds the per-band codec (FusedCodec on a GPU box; the tests pass the CPU
    rendition): anything with encode(code, mask, imap) -> (imp_bytes, code_bytes) and decode(imp_bytes, code_bytes) -> (code, mask)."""

    def __init__(self, make_codec, H, W, nbands, world=1, rank=0, in_flight=1):
        self.H, self.W, self.nbands = H, W, nbands
        self.rows = band_rows(H, nbands)
        _PartCodec.__init__(self, make_codec, (H // nbands, W), nbands, world, rank, in_flight)

    def encode_local(self, code, mask, imap):
        """Codes this rank's bands of the full-size inputs -> {band: (imp_bytes, code_bytes)}."""
        bands = split_bands(code, mask, imap, self.nbands)
        res = self._map(lambda cd, b: cd.encode(*bands[b]), self.mine)
        return dict(zip(self.mine, res))

    def encode(self, code, mask, imap):
        """-> the container (identical on every rank)."""
        return pack_band_streams(self.H, self.W, exchange_streams(self.encode_local(code, mask, imap), self.nbands))

    def encode_to_budget(self, code, imap, max_bytes, protect=None):
        """The container in at most max_bytes bytes, its header (16 + 8 * nbands bytes) included: the bands, split as split_bands
        splits them (protect rows too), are coded by one FusedCodec of the band size in its shared budget mode
        (FusedCodec.encode_batch_to_budget(..., shared=True)), so every band is lowered by the same level offset.  code (1,48,H,W),
        imap (1,1,H/2,W/2), protect None or an integer (1,1,H/2,W/2) map.  decode reads the container as any other.  world == 1
        only: the bands' bounds are not gathered across ranks.
        -> {'container': bytes, 'offset': the shared offset, 'bound': the container's bound at it, 'bounds': {offset: container
        bound} of every offset evaluated, 'results': the per-band dicts of encode_batch_to_budget}"""
        if self.world != 1:
            raise RuntimeError("BandCodec.encode_to_budget: needs world == 1 (got %d); the bands' bounds are not gathered across ranks"
                               % self.world)
        hi = self.H // 2
        if tuple(code.shape) != (1, code.shape[1], self.H, self.W) or tuple(imap.shape) != (1, 1, hi, self.W // 2):
            raise RuntimeError("BandCodec.encode_to_budget: expected a (1,C,%d,%d) latent and a (1,1,%d,%d) importance map"
                               % (self.H, self.W, hi, self.W // 2))
        if protect is not None and (not isinstance(protect, torch.Tensor) or tuple(protect.shape) != tuple(imap.shape)):
            raise RuntimeError("BandCodec.encode_to_budget: protect must be a (1,1,%d,%d) integer tensor, like the importance map"
                               % (hi, self.W // 2))
        head = 16 + 8 * self.nbands
        codes = torch.cat([code[:, :, r0:r1] for r0, r1 in self.rows])
        imaps = torch.cat([imap[:, :, r0 // 2:r1 // 2] for r0, r1 in self.rows])
        prot = None if protect is None else torch.cat([protect[:, :, r0 // 2:r1 // 2] for r0, r1 in self.rows])
        r = self.codecs[0].encode_batch_to_budget(codes, imaps, int(max_bytes) - head, protect=prot, shared=True)
        blob = pack_band_streams(self.H, self.W, [(x["imp_bytes"], x["code_bytes"]) for x in r["results"]])
        return {"container": blob, "offset": r["offset"], "bound": r["bound"] + head,
                "bounds": {t: b + head for t, b in r["bounds"].items()}, "results": r["results"]}

    def decode_local(self, blob):
        """Decodes this rank's bands -> {band: (code_b, mask_b)}."""
        H, W, streams = unpack_band_streams(blob)
        if (H, W, len(streams)) != (self.H, self.W, self.nbands):
            raise ValueError("BandCodec.decode: container is %dx%d in %d bands, codec is %dx%d in %d" % (H, W, len(streams), self.H, self.W, self.nbands))
        res = self._map(lambda cd, b: cd.decode(*streams[b]), self.mine)
        return dict(zip(self.mine, res))

    def decode(self, blob, like=None):
        """-> (code, mask) of the whole image on every rank (the decoded bands are exchanged: assembly, not coding)."""
        local = self.decode_local(blob)
        table = self._gather(local)
        cat = torch.cat if isinstance(next(iter(table.values()))[0], torch.Tensor) else None
        if cat is None:
            import numpy as np
            return (np.concatenate([table[b][0] for b in range(self.nbands)], axis=2),
                    np.concatenate([table[b][1] for b in range(self.nbands)], axis=2))
        dev = like.device if like is not None else next(iter(local.values()))[0].device
        return (torch.cat([table[b][0].to(dev) for b in range(self.nbands)], dim=2),
                torch.cat([table[b][1].to(dev) for b in range(self.nbands)], dim=2))


# ---------------------------------------------------------------------------------------------------------------------
# Tiles of ONE image: random access for viewers.
#
# A viewer shows one viewport of a 360-degree image, yet a single stream (or a latitude band) must be decoded whole.  The same
# format extension as the bands, in two dimensions: the latent is cut into rows x cols tiles of equal size and every tile is coded
# as an independent sub-image with its own two bitstreams (zero context at the tile's edges, as at the image's).  Each tile is
# exactly what the codec produces for that tile as an image of its own (the parity statement, per tile); a viewer decodes only the
# tiles its view touches (TileCodec.decode_views, with the exact footprint of lic360_pipeline.view_footprint).  Equal tiles make the
# whole image one batch for FusedCodec.encode_batch and its budget searches.
# ---------------------------------------------------------------------------------------------------------------------
TILE_MAGIC = b"L3T1"


def tile_grid(H, W, rows, cols):
    """[(r0, r1, c0, c1)] of the rows x cols tiles of an H x W latent, row-major.  One importance cell covers 2 x 2 latent cells, so
    the tiles, H / rows by W / cols, must have an even positive number of rows and columns."""
    if rows < 1 or cols < 1 or H < 1 or W < 1 or H % rows or W % cols or (H // rows) % 2 or (W // cols) % 2:
        raise ValueError("tile_grid: a %dx%d latent does not split into %dx%d tiles of an even number of rows and columns"
                         % (H, W, rows, cols))
    ht, wt = H // rows, W // cols
    return [(r * ht, (r + 1) * ht, c * wt, (c + 1) * wt) for r in range(rows) for c in range(cols)]


def pack_tile_streams(rows, cols, H, W, streams):
    """streams: [(imp_bytes, code_bytes)] in tile order -> one container: magic, rows, cols, H, W, the 2 * rows * cols lengths, the
    payloads."""
    tile_grid(H, W, rows, cols)
    if len(streams) != rows * cols:
        raise ValueError("pack_tile_streams: %d stream pairs for %dx%d tiles" % (len(streams), rows, cols))
    head = TILE_MAGIC + struct.pack("<IIII", rows, cols, H, W)
    head += b"".join(struct.pack("<II", len(a), len(b)) for a, b in streams)
    return head + b"".join(a + b for a, b in streams)


def tile_header_bytes(ntiles):
    return 20 + 8 * ntiles


def unpack_tile_streams(blob):
    """-> (rows, cols, H, W, [(imp_bytes, code_bytes)]); raises ValueError on a malformed container."""
    if len(blob) < 20 or blob[:4] != TILE_MAGIC:
        raise ValueError("unpack_tile_streams: not a tile container")
    rows, cols, H, W = struct.unpack_from("<IIII", blob, 4)
    tile_grid(H, W, rows, cols)  # ValueError when the grid does not divide the latent
    n = rows * cols
    off = tile_header_bytes(n)
    if len(blob) < off:
        raise ValueError("unpack_tile_streams: truncated header")
    lens = [struct.unpack_from("<II", blob, 20 + 8 * k) for k in range(n)]
    if off + sum(a + b for a, b in lens) != len(blob):
        raise ValueError("unpack_tile_streams: payload size does not match the header")
    out = []
    for a, b in lens:
        out.append((bytes(blob[off:off + a]), bytes(blob[off + a:off + a + b])))
        off += a + b
    return rows, cols, H, W, out


# A quality ladder of a tiled image: every tile coded at R rates (rungs), so that a server can cut, per viewer, an ordinary tile
# container that sends the tiles in view from a high rung and the rest from a low one (ladder_to_tiles).  Rung r of tile k is an
# ordinary stream pair, coded with the rung's level offset.
LADDER_MAGIC = b"L3L1"


def ladder_header_bytes(nrungs, ntiles):
    return 24 + 4 * nrungs + 8 * nrungs * ntiles


def pack_ladder_streams(rows, cols, H, W, offsets, rungs):
    """offsets: the R rungs' level offsets; rungs: R lists of rows * cols (imp_bytes, code_bytes) in tile order -> one container: magic,
    rows, cols, H, W, R, the R offsets, the R * rows * cols stream-length pairs rung-major, the payloads in the same order."""
    tile_grid(H, W, rows, cols)
    T, R = rows * cols, len(rungs)
    if R < 1 or len(offsets) != R:
        raise ValueError("pack_ladder_streams: %d offsets for %d rungs (need at least one rung)" % (len(offsets), R))
    if any(isinstance(t, bool) or not isinstance(t, int) or not 0 <= t < 2 ** 32 for t in offsets):
        raise ValueError("pack_ladder_streams: offsets must be non-negative ints (got %r)" % (list(offsets),))
    if any(len(r) != T for r in rungs):
        raise ValueError("pack_ladder_streams: rungs of %s stream pairs for %dx%d tiles" % ([len(r) for r in rungs], rows, cols))
    head = LADDER_MAGIC + struct.pack("<IIIII", rows, cols, H, W, R) + struct.pack("<%dI" % R, *offsets)
    head += b"".join(struct.pack("<II", len(a), len(b)) for r in rungs for a, b in r)
    return head + b"".join(a + b for r in rungs for a, b in r)


def unpack_ladder_streams(blob):
    """-> (rows, cols, H, W, offsets, rungs), rungs[r][k] = (imp_bytes, code_bytes) of tile k at rung r; raises ValueError on a
    malformed container."""
    if len(blob) < 24 or blob[:4] != LADDER_MAGIC:
        raise ValueError("unpack_ladder_streams: not a ladder container")
    rows, cols, H, W, R = struct.unpack_from("<IIIII", blob, 4)
    tile_grid(H, W, rows, cols)  # ValueError when the grid does not divide the latent
    T = rows * cols
    if R < 1:
        raise ValueError("unpack_ladder_streams: a ladder needs at least one rung")
    off = ladder_header_bytes(R, T)
    if len(blob) < off:
        raise ValueError("unpack_ladder_streams: truncated header")
    offsets = list(struct.unpack_from("<%dI" % R, blob, 24))
    lens = struct.unpack_from("<%dI" % (2 * R * T), blob, 24 + 4 * R)
    if off + sum(lens) != len(blob):
        raise ValueError("unpack_ladder_streams: payload size does not match the header")
    rungs = []
    for r in range(R):
        rung = []
        for k in range(T):
            a, b = lens[2 * (r * T + k)], lens[2 * (r * T + k) + 1]
            rung.append((bytes(blob[off:off + a]), bytes(blob[off + a:off + a + b])))
            off += a + b
        rungs.append(rung)
    return rows, cols, H, W, offsets, rungs


def ladder_to_tiles(blob, rungs):
    """Cuts a tile container from a ladder: tile k from rung rungs[k] (rungs: one rung index for every tile, or a list of rows * cols
    indices, e.g. TileCodec.rungs_for_views).  The result is an ordinary L3T1 container, equal to pack_tile_streams of the chosen
    streams, which TileCodec.decode / decode_tiles / decode_views read as any other.  ValueError on a malformed ladder, a wrongly
    sized list or a rung outside [0, R)."""
    rows, cols, H, W, offsets, ladder = unpack_ladder_streams(blob)
    T, R = rows * cols, len(offsets)
    if isinstance(rungs, int) and not isinstance(rungs, bool):
        rungs = [rungs] * T
    if not isinstance(rungs, (list, tuple)) or len(rungs) != T:
        raise ValueError("ladder_to_tiles: need one rung index or a list of %d (got %r)" % (T, rungs))
    if any(isinstance(r, bool) or not isinstance(r, int) or not 0 <= r < R for r in rungs):
        raise ValueError("ladder_to_tiles: rung indices must be ints in [0, %d) (got %r)" % (R, rungs))
    return pack_tile_streams(rows, cols, H, W, [ladder[r][k] for k, r in enumerate(rungs)])


def split_tiles(x, rows, cols):
    """(1,C,h,w) -> (rows*cols, C, h/rows, w/cols): the tiles in row-major order, one contiguous batch"""
    _, C, h, w = x.shape
    return x.reshape(C, rows, h // rows, cols, w // cols).permute(1, 3, 0, 2, 4).reshape(rows * cols, C, h // rows, w // cols)


class TileCodec(_PartCodec):
    """One image as rows x cols independently coded tiles, dealt round-robin to the ranks of the process group (or all on this
    process without one), decodable tile by tile.  `make_codec(h_t, w_t)` builds the per-tile codec: FusedCodec on a GPU, whose
    encode_batch codes all of a rank's tiles in one pass; anything with BandCodec's encode / decode methods is coded tile by tile.
    `in_flight` codecs decode tiles concurrently, one worker thread each."""

    def __init__(self, make_codec, H, W, rows, cols, world=1, rank=0, in_flight=1):
        self.H, self.W, self.rows, self.cols = H, W, rows, cols
        self.tiles = tile_grid(H, W, rows, cols)
        self.ht, self.wt = H // rows, W // cols
        _PartCodec.__init__(self, make_codec, (self.ht, self.wt), rows * cols, world, rank, in_flight)
        self.device = getattr(self.codecs[0], "dev", torch.device("cpu"))

    def _check(self, code, imap, who):
        hi, wi = self.H // 2, self.W // 2
        if (code.dim() != 4 or tuple(code.shape) != (1, code.shape[1], self.H, self.W) or imap.dim() != 4
                or tuple(imap.shape) != (1, 1, hi, wi)):
            raise RuntimeError("TileCodec.%s: expected a (1,C,%d,%d) latent and a (1,1,%d,%d) importance map" % (who, self.H, self.W, hi, wi))

    def encode_local(self, code, mask, imap):
        """Codes this rank's tiles of the full-size inputs -> {tile: (imp_bytes, code_bytes)}."""
        self._check(code, imap, "encode")
        if not self.mine:
            return {}
        codes, masks, imaps = (split_tiles(x, self.rows, self.cols)[self.mine] for x in (code, mask, imap))
        if hasattr(self.codecs[0], "encode_batch"):
            res = self.codecs[0].encode_batch(codes, masks, imaps)
        else:
            res = self._map(lambda cd, k: cd.encode(codes[k:k + 1], masks[k:k + 1], imaps[k:k + 1]), list(range(len(self.mine))))
        return dict(zip(self.mine, res))

    def encode(self, code, mask, imap):
        """code, mask (1,48,H,W), imap (1,1,H/2,W/2) -> the container (identical on every rank)."""
        streams = exchange_streams(self.encode_local(code, mask, imap), len(self.tiles), "tile")
        return pack_tile_streams(self.rows, self.cols, self.H, self.W, streams)

    def encode_to_budget(self, code, imap, max_bytes, protect=None):
        """The container within a byte budget, by FusedCodec.encode_batch_to_budget on the tiles (protect split as the importance map).

        max_bytes an int: the whole container, its header (20 + 8 * rows * cols bytes) included, with one level offset shared by all
        tiles (shared mode).  -> {'container', 'offset', 'bound': the container's bound at the offset, 'bounds': {offset: container
        bound} of every offset evaluated, 'results': the per-tile dicts}.
        max_bytes a list of rows * cols ints: each tile's two streams within its own budget (per-latent mode), e.g. more bytes for the
        tiles a viewer is likely to see.  -> {'container', 'offsets': per tile, 'results': the per-tile dicts}.
        world == 1 only: the tiles' bounds are not gathered across ranks."""
        if self.world != 1:
            raise RuntimeError("TileCodec.encode_to_budget: needs world == 1 (got %d); the tiles' bounds are not gathered across ranks"
                               % self.world)
        self._check(code, imap, "encode_to_budget")
        if protect is not None and (not isinstance(protect, torch.Tensor) or tuple(protect.shape) != tuple(imap.shape)):
            raise RuntimeError("TileCodec.encode_to_budget: protect must be a (1,1,%d,%d) integer tensor, like the importance map"
                               % (self.H // 2, self.W // 2))
        T = len(self.tiles)
        codes, imaps = split_tiles(code, self.rows, self.cols), split_tiles(imap, self.rows, self.cols)
        prot = None if protect is None else split_tiles(protect, self.rows, self.cols)
        cd = self.codecs[0]
        if isinstance(max_bytes, (list, tuple)):
            if len(max_bytes) != T:
                raise RuntimeError("TileCodec.encode_to_budget: %d budgets for %d tiles" % (len(max_bytes), T))
            res = cd.encode_batch_to_budget(codes, imaps, [int(b) for b in max_bytes], protect=prot)
            blob = pack_tile_streams(self.rows, self.cols, self.H, self.W, [(x["imp_bytes"], x["code_bytes"]) for x in res])
            return {"container": blob, "offsets": [x["offset"] for x in res], "results": res}
        head = tile_header_bytes(T)
        r = cd.encode_batch_to_budget(codes, imaps, int(max_bytes) - head, protect=prot, shared=True)
        blob = pack_tile_streams(self.rows, self.cols, self.H, self.W, [(x["imp_bytes"], x["code_bytes"]) for x in r["results"]])
        return {"container": blob, "offset": r["offset"], "bound": r["bound"] + head,
                "bounds": {t: b + head for t, b in r["bounds"].items()}, "results": r["results"]}

    def encode_ladder(self, code, imap, budgets=None, offsets=None, protect=None, max_batch=16):
        """Every tile at R rates in one ladder container (pack_ladder_streams), from which ladder_to_tiles cuts ordinary tile containers.
        Give exactly one of:
          budgets: R container budgets in bytes, header included.  Rung r is encode_to_budget(code, imap, budgets[r], protect)'s
            shared mode, one offset for all tiles, found for all rungs by one select_shared_offsets over estimate_candidates, so the
            stage-1 estimates are shared and no (tile, offset) pair is estimated twice; ladder_to_tiles(ladder, r) equals that call's
            container byte for byte.
          offsets: R fixed level offsets, no search; rung r is encode() of the tiles lowered by offsets[r] (levels_to_mask).
        Each distinct (tile, offset) pair is coded once by FusedCodec.encode_candidates, at most max_batch per pass (it bounds the
        encoder buffers and does not change the result).  code (1,48,H,W), imap (1,1,H/2,W/2), protect None or an integer (1,1,H/2,W/2)
        map, split as encode_to_budget splits it.
        -> {'ladder': bytes, 'offsets': per rung, 'bounds': per rung encode_to_budget's {offset: container bound} (None with offsets),
        'sizes': bytes of each rung's cut}.  RuntimeError, with nothing returned, when no offset fits a budget (encode_to_budget's
        message followed by ' (rung r)') or a cut exceeds its budget.  world == 1 only."""
        if self.world != 1:
            raise RuntimeError("TileCodec.encode_ladder: needs world == 1 (got %d); the tiles' bounds are not gathered across ranks"
                               % self.world)
        self._check(code, imap, "encode_ladder")
        if protect is not None and (not isinstance(protect, torch.Tensor) or tuple(protect.shape) != tuple(imap.shape)):
            raise RuntimeError("TileCodec.encode_ladder: protect must be a (1,1,%d,%d) integer tensor, like the importance map"
                               % (self.H // 2, self.W // 2))
        if (budgets is None) == (offsets is None):
            raise RuntimeError("TileCodec.encode_ladder: give exactly one of budgets and offsets")
        rungs = [int(x) for x in (budgets if offsets is None else offsets)]
        if not rungs:
            raise RuntimeError("TileCodec.encode_ladder: a ladder needs at least one rung")
        if isinstance(max_batch, bool) or not isinstance(max_batch, int) or max_batch < 1:
            raise RuntimeError("TileCodec.encode_ladder: max_batch must be a positive int (got %r)" % (max_batch,))
        import lic360_pipeline as pl
        T, head = len(self.tiles), tile_header_bytes(len(self.tiles))
        codes, imaps = split_tiles(code, self.rows, self.cols), split_tiles(imap, self.rows, self.cols)
        prot = None if protect is None else split_tiles(protect, self.rows, self.cols)
        cd = self.codecs[0]
        bounds = None
        if offsets is None:
            top = 48 if prot is None else 48 + int(prot.max())

            def estimate(pairs):
                return cd.estimate_candidates(codes, imaps, [k for k, _ in pairs], [t for _, t in pairs], prot)

            picks = pl.select_shared_offsets(estimate, [b - head for b in rungs], T, top, max_batch)
            offs = [o for o, _, _ in picks]
            bounds = [{t: b + head for t, b in own.items()} for _, own, _ in picks]
        else:
            offs = rungs
            if any(t < 0 for t in offs):
                raise RuntimeError("TileCodec.encode_ladder: offsets must not be negative (got %r)" % (offs,))
        pairs = [(k, t) for t in sorted(set(offs)) for k in range(T)]
        coded = {}
        for i in range(0, len(pairs), max_batch):
            part = pairs[i:i + max_batch]
            coded.update(zip(part, cd.encode_candidates(codes, imaps, [k for k, _ in part], [t for _, t in part], prot)))
        streams = [[coded[(k, t)] for k in range(T)] for t in offs]
        sizes = [head + sum(len(a) + len(b) for a, b in s) for s in streams]
        if budgets is not None:
            for r, (size, budget) in enumerate(zip(sizes, rungs)):
                if size > budget:
                    raise RuntimeError("TileCodec.encode_ladder: rung %d (offset %d) encoded to %d bytes, above its bound of %d and the "
                                       "budget of %d bytes" % (r, offs[r], size, bounds[r][offs[r]], budget))
        return {"ladder": pack_ladder_streams(self.rows, self.cols, self.H, self.W, offs, streams), "offsets": offs, "bounds": bounds,
                "sizes": sizes}

    def rungs_for_views(self, thetas, phis, fov, inside, outside, margin=0):
        """Rung indices for ladder_to_tiles: `inside` for the tiles the views need (tiles_for_views), `outside` for the others."""
        need = set(self.tiles_for_views(thetas, phis, fov, margin))
        return [inside if k in need else outside for k in range(len(self.tiles))]

    def tiles_for_views(self, thetas, phis, fov, margin=0):
        """Sorted indices of the tiles that hold a cell of the views' footprints (lic360_pipeline.view_protection on the importance
        grid, dilated by `margin` cells), by a max over each tile on the codec's device."""
        import lic360_pipeline as pl
        fp = pl.view_protection(self.H // 2, self.W // 2, thetas, phis, fov, 1, margin, self.device)
        hit = split_tiles(fp, self.rows, self.cols).amax(dim=(1, 2, 3))
        return [int(k) for k in torch.nonzero(hit).flatten().tolist()]

    def decode_tiles(self, blob, tiles):
        """Decodes only `tiles` (indices into tile_grid's order), this rank's share of them on up to in_flight codecs at once, and
        assembles them on every rank -> (code, mask, decoded): code and mask (1,48,H,W), zero outside the decoded tiles (mask 0: not
        coded), decoded (1,1,H,W) int32, 1 on the latent cells decoded."""
        rows, cols, H, W, streams = unpack_tile_streams(blob)
        if (rows, cols, H, W) != (self.rows, self.cols, self.H, self.W):
            raise ValueError("TileCodec.decode: container is %dx%d in %dx%d tiles, codec is %dx%d in %dx%d"
                             % (H, W, rows, cols, self.H, self.W, self.rows, self.cols))
        want = sorted(set(int(k) for k in tiles))
        if want and not (0 <= want[0] and want[-1] < len(self.tiles)):
            raise ValueError("TileCodec.decode_tiles: tile indices must lie in [0, %d) (got %s)" % (len(self.tiles), want))
        mine = [k for k in want if k in set(self.mine)]
        local = dict(zip(mine, self._map(lambda cd, k: cd.decode(*streams[k]), mine)))
        table = self._gather(local)
        dev = self.device
        code = torch.zeros((1, 48, H, W), dtype=torch.float32, device=dev)
        mask = torch.zeros((1, 48, H, W), dtype=torch.float32, device=dev)
        decoded = torch.zeros((1, 1, H, W), dtype=torch.int32, device=dev)
        for k in want:
            r0, r1, c0, c1 = self.tiles[k]
            c, m = table[k]
            code[:, :, r0:r1, c0:c1] = torch.as_tensor(c).to(dev)
            mask[:, :, r0:r1, c0:c1] = torch.as_tensor(m).to(dev)
            decoded[:, :, r0:r1, c0:c1] = 1
        return code, mask, decoded

    def decode_views(self, blob, thetas, phis, fov, margin=0):
        """decode_tiles of the tiles the views need (tiles_for_views) -> (code, mask, decoded)."""
        return self.decode_tiles(blob, self.tiles_for_views(thetas, phis, fov, margin))

    def decode(self, blob):
        """-> (code, mask) of the whole image on every rank."""
        code, mask, _ = self.decode_tiles(blob, range(len(self.tiles)))
        return code, mask
