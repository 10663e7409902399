"""Tiled quality ladders on cuda:0: TileCodec.encode_ladder against R separate TileCodec.encode_to_budget calls.

A 256x512 latent (a 2048x4096 image) from synthetic_latent with seeded random-init parameters (make_codec_params), in 4x4 tiles of
64x128.  The rungs are R = 3 and R = 4 container budgets spread evenly between the bound of the all-zero levels (offset 48) and the
bound of offset 0, the top rung at offset 0's bound.

  time     : encode_ladder(budgets) against R encode_to_budget calls, after one warm-up of each, alternating the arms in rotating order
             within each repetition; host clock around calls that end in a device synchronise; medians and 10th / 90th percentiles
  estimates: the (tile, offset) candidates each arm estimates
  memory   : peak torch allocation above the inputs (torch.cuda.max_memory_allocated) and the growth of the codec's own buffers
             (device memory taken outside torch's allocator) on a fresh TileCodec, for encode_ladder with its search, for its encode
             alone (offsets given), for the same ladder built with levels_to_mask_batch + encode_batch (materialised candidates), and
             for the R encode_to_budget calls
  cut      : bytes of the front view's cut (tiles in view from the top rung, the others from the bottom rung) against the top rung

Every arm's containers are checked equal first.  The GPU name and power limit are read in the same run.  Prints one JSON line and
writes it to OUT/tile_ladder_timing.json.

    python tools/tile_ladder_timing.py --out DIR [--reps 5] [--warmup 1]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "360-image-compression_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import lic360_pipeline as pl  # noqa: E402
import lic360_shard as sh  # noqa: E402
from estimate_timing import gpu_card  # noqa: E402
from tile_view_timing import timed  # noqa: E402
from util import synthetic_latent, t  # noqa: E402

H, W, ROWS, COLS, FOV, MAX_BATCH = 256, 512, 4, 4, 0.5, 16
T = ROWS * COLS


def budgets(tc, code, imap, R):
    """R container budgets from the bound of offset 0 (top rung) down towards that of offset 48 (all levels 0)"""
    codes, imaps = sh.split_tiles(code, ROWS, COLS), sh.split_tiles(imap, ROWS, COLS)
    ests = tc.codecs[0].estimate_candidates(codes, imaps, list(range(T)) * 2, [0] * T + [48] * T)
    head = sh.tile_header_bytes(T)
    lo, hi = head + sum(map(pl.budget_bound, ests[T:])), head + sum(map(pl.budget_bound, ests[:T]))
    return [lo + (hi - lo) * (R - r) // R for r in range(R)]


def materialised_ladder(tc, code, imap, offsets):
    """the ladder encode_ladder(offsets=...) builds, from materialised candidates: levels_to_mask_batch + encode_batch per pass"""
    codes, imaps = sh.split_tiles(code, ROWS, COLS), sh.split_tiles(imap, ROWS, COLS)
    pairs = [(k, o) for o in sorted(set(offsets)) for k in range(T)]
    coded = {}
    for i in range(0, len(pairs), MAX_BATCH):
        part = pairs[i:i + MAX_BATCH]
        lat, off = [k for k, _ in part], [o for _, o in part]
        levels, masks = pl.levels_to_mask_batch(imaps, lat, off)
        coded.update(zip(part, tc.codecs[0].encode_batch(codes[torch.tensor(lat, device=code.device)], masks, levels)))
    return sh.pack_ladder_streams(ROWS, COLS, H, W, list(offsets), [[coded[(k, o)] for k in range(T)] for o in offsets])


def counted(tc):
    """counts the candidates the tile codec's FusedCodec estimates (every budget search goes through _candidates)"""
    cd, n = tc.codecs[0], [0]
    inner = cd._candidates

    def wrap(code, imp, protect, pairs):
        n[0] += len(pairs)
        return inner(code, imp, protect, pairs)

    cd._candidates = wrap
    return n


def memory(make, fn):
    """peak torch allocation above what was allocated before, and growth of the device memory taken outside torch, for fn(tc) on
    a fresh TileCodec"""
    tc = make()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0, res0, alloc0 = torch.cuda.mem_get_info()[0], torch.cuda.memory_reserved(), torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn(tc)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - alloc0
    codec = (free0 - torch.cuda.mem_get_info()[0]) - (torch.cuda.memory_reserved() - res0)
    del tc
    return {"torch_peak_mb": peak / 2 ** 20, "codec_growth_mb": codec / 2 ** 20}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for tile_ladder_timing.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tile_ladder_timing: needs a CUDA device")
    dev = "cuda:0"
    line = dict(gpu_card())
    line.update({"latent": [H, W], "image": [8 * H, 8 * W], "tiles": [ROWS, COLS], "tile": [H // ROWS, W // COLS], "max_batch": MAX_BATCH,
                 "reps": a.reps, "weights": "random-init (make_codec_params): byte counts are not representative of trained weights"})
    params = pl.make_codec_params(dev, seed=a.seed)
    qn, _, lvn = synthetic_latent(a.seed + 1, H=H, W=W)
    code, imap = t(qn, dev), t(lvn, dev)

    def make():
        return sh.TileCodec(lambda h, w: pl.FusedCodec(params, H=h, W=w), H, W, ROWS, COLS)

    tc = make()
    n_est = counted(tc)
    line["rungs"] = {}
    for R in (3, 4):
        bud = budgets(tc, code, imap, R)
        n_est[0] = 0
        lad = tc.encode_ladder(code, imap, budgets=bud, max_batch=MAX_BATCH)
        ladder_estimates = n_est[0]
        n_est[0] = 0
        sep = [tc.encode_to_budget(code, imap, b) for b in bud]
        separate_estimates = n_est[0]
        for r in range(R):
            assert sh.ladder_to_tiles(lad["ladder"], r) == sep[r]["container"], r
        offsets = lad["offsets"]
        assert materialised_ladder(tc, code, imap, offsets) == lad["ladder"]
        rungs = tc.rungs_for_views([0.0], [0.0], FOV, inside=0, outside=R - 1)
        cut = sh.ladder_to_tiles(lad["ladder"], rungs)
        entry = {"budgets": bud, "offsets": offsets, "sizes": lad["sizes"], "ladder_bytes": len(lad["ladder"]),
                 "candidate_estimates": {"encode_ladder": ladder_estimates, "separate_encode_to_budget": separate_estimates},
                 "front_view_cut": {"fov": FOV, "tiles_in_view": sum(1 for x in rungs if x == 0), "bytes": len(cut),
                                    "top_rung_bytes": lad["sizes"][0], "ratio": len(cut) / lad["sizes"][0]}}
        entry["time_ms"] = timed({"encode_ladder": lambda: tc.encode_ladder(code, imap, budgets=bud, max_batch=MAX_BATCH),
                                  "separate_encode_to_budget": lambda: [tc.encode_to_budget(code, imap, b) for b in bud]},
                                 a.reps, a.warmup)
        entry["memory"] = {
            "encode_ladder": memory(make, lambda c: c.encode_ladder(code, imap, budgets=bud, max_batch=MAX_BATCH)),
            "encode_ladder_offsets_only": memory(make, lambda c: c.encode_ladder(code, imap, offsets=offsets, max_batch=MAX_BATCH)),
            "materialised_levels_to_mask_batch_encode_batch": memory(make, lambda c: materialised_ladder(c, code, imap, offsets)),
            "separate_encode_to_budget": memory(make, lambda c: [c.encode_to_budget(code, imap, b) for b in bud]),
        }
        line["rungs"][str(R)] = entry
    s = json.dumps(line)
    print(s)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "tile_ladder_timing.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
