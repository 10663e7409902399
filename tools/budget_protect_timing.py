"""FusedCodec.encode_to_budget without a protection map, with latitude_protection (levels 16) and with the front viewport's
viewport_protection (levels 48), on cuda:0.

Latents of 64x128 and 128x256 (images of 512x1024 and 1024x2048), seeded parameters (make_codec_params) and synthetic_latent.  The
budget is halfway between the byte bounds of candidate 0 (the latent as it is) and of the all-zero candidate.  After a warm-up of
every mode, each repetition times the three modes in rotating order, with a host clock around calls that end in a device
synchronise.  For each mode it records the median and 10th / 90th percentiles, the offsets evaluated, and, from an `estimate` of the
chosen candidate, the share of the code stream's bits and of its coded symbols that fall in the region the map protects (cells with
P >= max P / 2), next to the same shares of the uniform encode at the same budget.  The GPU name and power limit are read in the same
run.  Prints one JSON line and writes it to OUT/budget_protect_timing.json.

    python tools/budget_protect_timing.py --out DIR [--reps 30] [--warmup 3]
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
import torch.nn.functional as F  # noqa: E402

import lic360_pipeline as pl  # noqa: E402
from estimate_batch_timing import stats  # noqa: E402
from estimate_timing import gpu_card  # noqa: E402
from util import synthetic_latent, t  # noqa: E402

SIZES = [(64, 128), (128, 256)]


def per_cell(x):
    """(1,48,H,W) -> (h,w): the sum over a cell's 48 channels and 2x2 positions"""
    return F.avg_pool2d(x.sum(1, keepdim=True), 2, divisor_override=1)[0, 0]


def shares(codec, q, r, region):
    est = codec.estimate(q, r["mask"], r["levels"])
    bits, coded = per_cell(est["code_map"]), per_cell(r["mask"])
    return {"code_bits_share": float(bits[region].sum() / bits.sum()), "coded_symbols_share": float(coded[region].sum() / coded.sum())}


def run_size(H, W, reps, warmup, seed):
    dev = "cuda:0"
    h, w = H // 2, W // 2
    codec = pl.FusedCodec(pl.make_codec_params(dev, seed=seed), H=H, W=W)
    qn, _, lvn = synthetic_latent(seed + 1, H=H, W=W)
    q, lv = t(qn, dev), t(lvn, dev)
    levels, masks = pl.levels_to_mask(lv, [0, 48])
    ends = codec.estimate_batch(q.expand(2, -1, -1, -1), masks, levels, maps=False)
    b0, bz = pl.budget_bound(ends[0]), pl.budget_bound(ends[1])
    budget = (b0 + bz) // 2
    maps = {"uniform": None, "latitude16": pl.latitude_protection(h, w, 16, dev),
            "front_viewport48": pl.viewport_protection(h, w, [1], 48, device=dev)}
    out = {}
    arms = {name: (lambda name=name, P=P: out.__setitem__(name, codec.encode_to_budget(q, lv, budget, protect=P)))
            for name, P in maps.items()}
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    names = list(arms)
    times = {k: [] for k in names}
    for i in range(reps):
        for name in names[i % 3:] + names[:i % 3]:
            t0 = time.perf_counter()
            arms[name]()
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
    res = {"latent": [H, W], "image": [8 * H, 8 * W], "reps": reps, "max_bytes": budget, "bound_offset0": b0,
           "bound_all_zero": bz, "modes": {}}
    for name, P in maps.items():
        r = out[name]
        m = {"ms": stats(times[name]), "offset": r["offset"], "candidates_evaluated": len(r["bounds"]),
             "offsets": sorted(r["bounds"]),
             "bytes": len(r["imp_bytes"]) + len(r["code_bytes"]), "bound": r["bound"]}
        if P is not None:
            region = P[0, 0] >= (int(P.max()) + 1) // 2
            m["protected_cells"] = int(region.sum())
            m["region_share_of_cells"] = float(region.float().mean())
            m["protected"] = shares(codec, q, r, region)
            m["uniform_same_budget"] = shares(codec, q, out["uniform"], region)
        res["modes"][name] = m
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for budget_protect_timing.json")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("budget_protect_timing: needs a CUDA device")
    line = dict(gpu_card())
    line["sizes"] = [run_size(H, W, a.reps, a.warmup, a.seed) for H, W in SIZES]
    s = json.dumps(line)
    print(s)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "budget_protect_timing.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
