"""Tiled coding on cuda:0: what a viewer pays to see one view of a 360-degree image, against decoding the single stream.

A 256x512 latent (a 2048x4096 image) from synthetic_latent with seeded parameters (make_codec_params), as one stream and as 4x4 tiles
of 64x128 (lic360_shard.TileCodec).  After a warm-up of every arm, each repetition runs the arms of a group in rotating order, with a
host clock around calls that end in a device synchronise; medians and 10th / 90th percentiles are recorded.

  decode : the single-stream decode, TileCodec.decode of all 16 tiles, and decode_views of the front view (0, 0), the (0, 0.25) view
           and the north-pole view (0, 0.5), fov 0.5, at in_flight 1, 2, 4 and 6, with the tiles each view needs
  encode : the single-stream encode against TileCodec.encode (one encode_batch of the 16 tiles)
  bytes  : the container against the single stream (random-init weights: not representative of trained weights)
  footprint: view_footprint of one view and of MultiProject's 14 views on the 128x256 importance grid, against viewport_protection
           of the same views

The GPU name and power limit are read in the same run.  Prints one JSON line and writes it to OUT/tile_view_timing.json.

    python tools/tile_view_timing.py --out DIR [--reps 7] [--warmup 2]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "360-image-compression_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import lic360_pipeline as pl  # noqa: E402
import lic360_shard as sh  # noqa: E402
from estimate_batch_timing import stats  # noqa: E402
from estimate_timing import gpu_card  # noqa: E402
from util import synthetic_latent, t  # noqa: E402

H, W, ROWS, COLS, FOV = 256, 512, 4, 4, 0.5
VIEWS = {"front": (0.0, 0.0), "up_0.25": (0.0, 0.25), "north_pole": (0.0, 0.5)}
IN_FLIGHT = (1, 2, 4, 6)


def timed(arms, reps, warmup):
    """arms: {name: fn}; ms per call of each, in rotating order"""
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    names = list(arms)
    times = {k: [] for k in names}
    for i in range(reps):
        k = i % len(names)
        for name in names[k:] + names[:k]:
            t0 = time.perf_counter()
            arms[name]()
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
    return {k: stats(v) for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for tile_view_timing.json")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tile_view_timing: needs a CUDA device")
    dev = "cuda:0"
    line = dict(gpu_card())
    line.update({"latent": [H, W], "image": [8 * H, 8 * W], "tiles": [ROWS, COLS], "tile": [H // ROWS, W // COLS], "fov": FOV,
                 "reps": a.reps})
    params = pl.make_codec_params(dev, seed=a.seed)
    qn, mn, lvn = synthetic_latent(a.seed + 1, H=H, W=W)
    q, m, lv = t(qn, dev), t(mn, dev), t(lvn, dev)

    single = pl.FusedCodec(params, H=H, W=W)
    tiled = {k: sh.TileCodec(lambda h, w: pl.FusedCodec(params, H=h, W=w), H, W, ROWS, COLS, in_flight=k) for k in IN_FLIGHT}
    one = tiled[1]
    streams = single.encode(q, m, lv)
    blob = one.encode(q, m, lv)
    assert blob == tiled[6].encode(q, m, lv)
    code, mask = one.decode(blob)
    assert torch.equal(mask, m) and torch.equal(code, q * m)
    line["bytes"] = {"single_stream": len(streams[0]) + len(streams[1]), "container": len(blob),
                     "container_header": sh.tile_header_bytes(ROWS * COLS),
                     "overhead_pct": 100.0 * (len(blob) / (len(streams[0]) + len(streams[1])) - 1),
                     "note": "random-init weights: not representative of trained weights"}

    line["encode_ms"] = timed({"single_stream": lambda: single.encode(q, m, lv), "tiles_encode_batch": lambda: one.encode(q, m, lv)},
                              a.reps, a.warmup)

    arms = {"single_stream": lambda: single.decode(*streams), "tiles_all": lambda: one.decode(blob)}
    line["view_tiles"] = {}
    for name, (th, ph) in VIEWS.items():
        line["view_tiles"][name] = one.tiles_for_views([th], [ph], FOV)
        for k in IN_FLIGHT:
            arms["%s_in_flight_%d" % (name, k)] = (lambda k=k, th=th, ph=ph: tiled[k].decode_views(blob, [th], [ph], FOV))
    line["decode_ms"] = timed(arms, a.reps, a.warmup)

    from lic360_operator._modules import VIEWPORT_PHIS, VIEWPORT_THETAS
    h, w = H // 2, W // 2
    line["footprint_grid"] = [h, w]
    line["footprint_ms"] = timed({
        "view_footprint_1": lambda: pl.view_footprint(h, w, [0.0], [0.0], 0.6, dev),
        "view_footprint_14": lambda: pl.view_footprint(h, w, VIEWPORT_THETAS, VIEWPORT_PHIS, 0.6, dev),
        "viewport_protection_1": lambda: pl.viewport_protection(h, w, [1], 48, fov=0.6, device=dev),
        "viewport_protection_14": lambda: pl.viewport_protection(h, w, list(range(14)), 48, fov=0.6, device=dev),
    }, max(a.reps, 20), a.warmup)
    s = json.dumps(line)
    print(s)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "tile_view_timing.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
