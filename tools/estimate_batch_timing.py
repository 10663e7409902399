"""K separate FusedCodec.estimate calls against one estimate_batch of K latents, and encode_to_budget against encode, on cuda:0.

Latents of 32x64, 64x128 and 128x256 (images of 256x512 to 1024x2048), K in {1, 4, 8, 16}, seeded parameters (make_codec_params)
and K different latents (synthetic_latent).  After a warm-up of every call, each repetition times both arms in alternating order,
with a host clock around calls that end in a device synchronise.  encode_to_budget runs at a budget halfway between the byte bounds
of offsets 0 and 48 (FusedCodec.encode_to_budget: two estimate_batch calls of 7 latents and one encode).  Prints one JSON line with
the medians and 10th / 90th percentiles and the batch speed-up (separate / batch); the GPU name and power limit are read in the
same run.  The line is also written to OUT/estimate_batch_timing.json.

    python tools/estimate_batch_timing.py --out DIR [--reps 30] [--warmup 3]
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

import lic360_pipeline as pl  # noqa: E402
from estimate_timing import gpu_card, pct  # noqa: E402
from util import synthetic_latent, t  # noqa: E402

SIZES = [(32, 64), (64, 128), (128, 256)]
KS = [1, 4, 8, 16]


def stats(v):
    return {"median": pct(v, 50), "p10": pct(v, 10), "p90": pct(v, 90)}


def alternate(arms, reps, warmup):
    """arms: {name: fn}; ms per call of each, in alternating order"""
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    names = list(arms)
    times = {k: [] for k in names}
    for i in range(reps):
        for name in (names if i % 2 == 0 else names[::-1]):
            t0 = time.perf_counter()
            arms[name]()
            torch.cuda.synchronize()
            times[name].append((time.perf_counter() - t0) * 1e3)
    return times


def run_size(H, W, reps, warmup, seed):
    dev = "cuda:0"
    codec = pl.FusedCodec(pl.make_codec_params(dev, seed=seed), H=H, W=W)
    lat = [synthetic_latent(seed + 1 + k, H=H, W=W) for k in range(max(KS))]
    q, m, lv = (t(np.concatenate([x[i] for x in lat]), dev) for i in range(3))
    res = {"latent": [H, W], "image": [8 * H, 8 * W], "reps": reps, "batch": []}
    for K in KS:
        def separate(K=K):
            return [codec.estimate(q[k:k + 1], m[k:k + 1], lv[k:k + 1]) for k in range(K)]

        def batch(K=K):
            return codec.estimate_batch(q[:K], m[:K], lv[:K])

        times = alternate({"separate": separate, "batch": batch}, reps, warmup)
        ms = {k: stats(v) for k, v in times.items()}
        res["batch"].append({"K": K, "separate_ms": ms["separate"], "batch_ms": ms["batch"],
                             "speedup": ms["separate"]["median"] / ms["batch"]["median"]})
    levels, masks = pl.levels_to_mask(lv[:1], [0, 48])
    ends = codec.estimate_batch(q[:1].expand(2, -1, -1, -1), masks, levels, maps=False)
    b0, b48 = pl.budget_bound(ends[0]), pl.budget_bound(ends[1])
    budget = (b0 + b48) // 2
    out = {}

    def encode():
        out["encode"] = codec.encode(q[:1], m[:1], lv[:1])

    def to_budget():
        out["budget"] = codec.encode_to_budget(q[:1], lv[:1], budget)

    times = alternate({"encode": encode, "encode_to_budget": to_budget}, reps, warmup)
    r = out["budget"]
    res["budget"] = {"max_bytes": budget, "bound_offset0": b0, "bound_offset48": b48, "offset": r["offset"],
                     "bytes": len(r["imp_bytes"]) + len(r["code_bytes"]), "bound": r["bound"],
                     "encode_bytes_offset0": sum(len(s) for s in out["encode"]),
                     "encode_ms": stats(times["encode"]), "encode_to_budget_ms": stats(times["encode_to_budget"])}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for estimate_batch_timing.json")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("estimate_batch_timing: needs a CUDA device")
    line = dict(gpu_card())
    line["sizes"] = [run_size(H, W, a.reps, a.warmup, a.seed) for H, W in SIZES]
    s = json.dumps(line)
    print(s)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "estimate_batch_timing.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
