"""Encode vs rate estimate of one latent through FusedCodec on cuda:0, at the latents of a 512x1024 and a 1024x2048 image.

Seeded parameters (make_codec_params) and latent (synthetic_latent).  After a warm-up of both calls, each repetition times one
encode and one estimate, in alternating order, with a host clock around a call that ends in a device synchronise.  Prints one
JSON line: per size the median and the 10th / 90th percentile of both, the split of the last call of each (last_timing), and the
two bit totals beside the two stream lengths; the GPU name and power limit are read in the same run.  The line is also written
to OUT/estimate_timing.json.

    python tools/estimate_timing.py --out DIR [--reps 50] [--warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "360-image-compression_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import lic360_pipeline as pl  # noqa: E402
from util import synthetic_latent, t  # noqa: E402

SIZES = [(64, 128), (128, 256)]


def gpu_card():
    """name and power limit of cuda:0 as nvidia-smi reports them (a query only)"""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True,
                         check=True).stdout.strip().splitlines()
    name, power = [s.strip() for s in out[1].split(",")]
    return {"gpu": name, "power_limit": power}


def pct(xs, q):
    return float(np.percentile(np.asarray(xs), q))


def run_size(H, W, reps, warmup, seed):
    dev = "cuda:0"
    q, mask, lv = synthetic_latent(seed, H=H, W=W)
    tq, tm, tl = t(q, dev), t(mask, dev), t(lv, dev)
    codec = pl.FusedCodec(pl.make_codec_params(dev, seed=seed), H=H, W=W)
    for _ in range(warmup):
        codec.encode(tq, tm, tl)
        codec.estimate(tq, tm, tl)
    torch.cuda.synchronize()
    times = {"encode": [], "estimate": []}
    split = {}
    streams = est = None
    for i in range(reps):
        for which in (("encode", "estimate") if i % 2 == 0 else ("estimate", "encode")):
            t0 = time.perf_counter()
            if which == "encode":
                streams = codec.encode(tq, tm, tl)
            else:
                est = codec.estimate(tq, tm, tl)
            torch.cuda.synchronize()
            times[which].append((time.perf_counter() - t0) * 1e3)
            split[which] = codec.last_timing()
    res = {"latent": [H, W], "image": [8 * H, 8 * W], "reps": reps}
    for k, v in times.items():
        res[k + "_ms"] = {"median": pct(v, 50), "p10": pct(v, 10), "p90": pct(v, 90), "min": min(v)}
    res["encode_last_split_ms"] = {k: split["encode"][k] for k in ("total_ms", "host_coder_ms", "gpu_wait_ms")}
    res["estimate_last_split_ms"] = {k: split["estimate"][k] for k in ("total_ms", "gpu_wait_ms")}
    n_code = int((mask >= 0.5).sum())
    res["streams"] = {
        "code": {"bytes": len(streams[1]), "ideal_bits": est["code_bits"], "coded_symbols": n_code,
                 "8len_minus_bits": 8 * len(streams[1]) - est["code_bits"]},
        "imp": {"bytes": len(streams[0]), "ideal_bits": est["imp_bits"], "coded_symbols": (H // 2) * (W // 2),
                "8len_minus_bits": 8 * len(streams[0]) - est["imp_bits"]},
    }
    res["estimated_bpp"] = (est["code_bits"] + est["imp_bits"]) / (64.0 * H * W)
    res["encoded_bpp"] = 8.0 * (len(streams[0]) + len(streams[1])) / (64.0 * H * W)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for estimate_timing.json")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("estimate_timing: needs a CUDA device")
    line = dict(gpu_card())
    line["sizes"] = [run_size(H, W, a.reps, a.warmup, a.seed) for H, W in SIZES]
    s = json.dumps(line)
    print(s)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "estimate_timing.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
