"""K separate FusedCodec.encode calls against one encode_batch of K latents, on cuda:0.

Latents of 32x64, 64x128 and 128x256 (images of 256x512 to 1024x2048), K in {1, 4, 8, 16}, seeded parameters (make_codec_params)
and K different latents (synthetic_latent).  After a warm-up of every call, each repetition times both arms in alternating order,
with a host clock around calls that end in a device synchronise; both arms must return the same bytes.  Prints one JSON line with
the medians and 10th / 90th percentiles, the batch speed-up (separate / batch) and the batch's own split (lic360_codec_last_timing:
host-coding phase and GPU wait); the GPU name and power limit are read in the same run, with the host's CPU count (the batch codes
its streams on min(K, CPUs, 16) threads).  The line is also written to OUT/encode_batch_timing.json.

    python tools/encode_batch_timing.py --out DIR [--reps 30] [--warmup 3]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "360-image-compression_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import lic360_pipeline as pl  # noqa: E402
from estimate_batch_timing import alternate, stats  # noqa: E402
from estimate_timing import gpu_card  # noqa: E402
from util import synthetic_latent, t  # noqa: E402

SIZES = [(32, 64), (64, 128), (128, 256)]
KS = [1, 4, 8, 16]


def run_size(H, W, reps, warmup, seed):
    dev = "cuda:0"
    codec = pl.FusedCodec(pl.make_codec_params(dev, seed=seed), H=H, W=W)
    lat = [synthetic_latent(seed + 1 + k, H=H, W=W) for k in range(max(KS))]
    q, m, lv = (t(np.concatenate([x[i] for x in lat]), dev) for i in range(3))
    res = {"latent": [H, W], "image": [8 * H, 8 * W], "reps": reps, "batch": []}
    for K in KS:
        out, split = {}, {"host_coding_ms": [], "gpu_wait_ms": []}

        def separate(K=K):
            out["separate"] = [codec.encode(q[k:k + 1], m[k:k + 1], lv[k:k + 1]) for k in range(K)]

        def batch(K=K):
            out["batch"] = codec.encode_batch(q[:K], m[:K], lv[:K])
            tm = codec.last_timing()
            split["host_coding_ms"].append(tm["host_coder_ms"])
            split["gpu_wait_ms"].append(tm["gpu_wait_ms"])

        times = alternate({"separate": separate, "batch": batch}, reps, warmup)
        if out["separate"] != out["batch"]:
            sys.exit("encode_batch_timing: %dx%d K=%d: batch and separate encodes differ" % (H, W, K))
        ms = {k: stats(v) for k, v in times.items()}
        # alternate() calls each arm `warmup` times before its timed repetitions: keep the split of the timed calls only
        res["batch"].append({"K": K, "separate_ms": ms["separate"], "batch_ms": ms["batch"],
                             "speedup": ms["separate"]["median"] / ms["batch"]["median"],
                             "batch_host_coding_ms": stats(split["host_coding_ms"][warmup:]),
                             "batch_gpu_wait_ms": stats(split["gpu_wait_ms"][warmup:]),
                             "bytes": sum(len(a) + len(b) for a, b in out["batch"])})
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for encode_batch_timing.json")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("encode_batch_timing: needs a CUDA device")
    line = dict(gpu_card())
    line["host_cpus"] = os.cpu_count()
    line["host_cpus_usable"] = len(os.sched_getaffinity(0))
    line["sizes"] = [run_size(H, W, a.reps, a.warmup, a.seed) for H, W in SIZES]
    s = json.dumps(line)
    print(s)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "encode_batch_timing.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
