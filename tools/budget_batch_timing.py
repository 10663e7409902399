"""K separate FusedCodec.encode_to_budget calls against one encode_batch_to_budget of K latents, on cuda:0: per latent without a
protection map and with latitude_protection (levels 16), plus the shared mode (one offset for all K latents).

Latents of 32x64 and 64x128 (images of 256x512 and 512x1024), seeded parameters (make_codec_params) and synthetic_latent, K = 1, 4
and 16.  Latent k's budget is a fraction between the byte bounds of its candidate 0 and its all-zero candidate, the fraction
running from 0.2 to 0.8 over the K latents; the shared budget is the sum of the per-latent budgets.  After a warm-up of every arm,
each repetition times the arms in rotating order, with a host clock around calls that end in a device synchronise, and records the
median and 10th / 90th percentiles; the per-latent arms also check that both paths return the same offsets and bytes.

Memory, per arm, on a codec of its own created for the measurement: the peak of torch.cuda.max_memory_allocated during one call
(the tensors the path allocates through torch: candidate levels and masks, the code copies), and the growth of the device's used
memory over the call minus the growth of torch's reserved memory, which is what the codec's own buffers (encoder frames, partials,
row buffers) grew by.  The GPU name and power limit are read in the same run.  Prints one JSON line and writes it to
OUT/budget_batch_timing.json.

    python tools/budget_batch_timing.py --out DIR [--reps 15] [--warmup 2]
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
from estimate_batch_timing import stats  # noqa: E402
from estimate_timing import gpu_card  # noqa: E402
from util import synthetic_latent, t  # noqa: E402

SIZES = [(32, 64), (64, 128)]
KS = [1, 4, 16]


def arms_of(codec, q, lv, budgets, P):
    """the timed calls of one K: name -> fn returning what it computed"""
    K = q.shape[0]

    def loop(protect):
        return [codec.encode_to_budget(q[k:k + 1], lv[k:k + 1], budgets[k], None if protect is None else protect[k:k + 1])
                for k in range(K)]

    return {
        "loop_uniform": lambda: loop(None),
        "batch_uniform": lambda: codec.encode_batch_to_budget(q, lv, budgets),
        "loop_latitude16": lambda: loop(P),
        "batch_latitude16": lambda: codec.encode_batch_to_budget(q, lv, budgets, protect=P),
        "shared_uniform": lambda: codec.encode_batch_to_budget(q, lv, sum(budgets), shared=True),
    }


def memory_of(params, H, W, fn_of):
    """peak torch allocation and codec buffer growth of one call of an arm on a fresh codec"""
    codec = pl.FusedCodec(params, H=H, W=W)
    fn = fn_of(codec)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base_alloc, base_res = torch.cuda.memory_allocated(), torch.cuda.memory_reserved()
    free0, _ = torch.cuda.mem_get_info()
    fn()
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    out = {"torch_peak_bytes": int(torch.cuda.max_memory_allocated() - base_alloc),
           "codec_buffers_bytes": int((free0 - free1) - (torch.cuda.memory_reserved() - base_res))}
    del codec
    return out


def run_size(H, W, reps, warmup, seed):
    dev = "cuda:0"
    h, w = H // 2, W // 2
    params = pl.make_codec_params(dev, seed=seed)
    codec = pl.FusedCodec(params, H=H, W=W)
    lat = [synthetic_latent(seed + 1 + k, H=H, W=W) for k in range(max(KS))]
    q_all = t(np.concatenate([x[0] for x in lat]), dev)
    lv_all = t(np.concatenate([x[2] for x in lat]), dev)
    P_all = pl.latitude_protection(h, w, 16, dev).expand(max(KS), -1, -1, -1).contiguous()
    ends = codec.estimate_candidates(q_all, lv_all, [k for k in range(max(KS)) for _ in (0, 1)], [0, 48] * max(KS))
    res = {"latent": [H, W], "image": [8 * H, 8 * W], "reps": reps, "batch": []}
    for K in KS:
        q, lv, P = q_all[:K], lv_all[:K], P_all[:K]
        fr = [0.2 + 0.6 * k / max(K - 1, 1) for k in range(K)]
        budgets = [int(pl.budget_bound(ends[2 * k + 1]) + f * (pl.budget_bound(ends[2 * k]) - pl.budget_bound(ends[2 * k + 1])))
                   for k, f in enumerate(fr)]
        arms = arms_of(codec, q, lv, budgets, P)
        out = {}
        for _ in range(warmup):
            for name, fn in arms.items():
                out[name] = fn()
        torch.cuda.synchronize()
        names = list(arms)
        times = {k: [] for k in names}
        for i in range(reps):
            for name in names[i % len(names):] + names[:i % len(names)]:
                t0 = time.perf_counter()
                arms[name]()
                torch.cuda.synchronize()
                times[name].append((time.perf_counter() - t0) * 1e3)
        for mode in ("uniform", "latitude16"):
            a, b = out["loop_" + mode], out["batch_" + mode]
            assert [(r["offset"], r["imp_bytes"], r["code_bytes"]) for r in a] == \
                   [(r["offset"], r["imp_bytes"], r["code_bytes"]) for r in b], (H, W, K, mode)
        entry = {"K": K, "budgets": budgets, "ms": {name: stats(v) for name, v in times.items()},
                 "offsets": {"uniform": [r["offset"] for r in out["batch_uniform"]],
                             "latitude16": [r["offset"] for r in out["batch_latitude16"]],
                             "shared": out["shared_uniform"]["offset"]},
                 "candidates_evaluated": {"uniform": sum(len(r["bounds"]) for r in out["batch_uniform"]),
                                          "latitude16": sum(len(r["bounds"]) for r in out["batch_latitude16"]),
                                          "shared": K * len(out["shared_uniform"]["bounds"])},
                 "shared_bytes": sum(len(r["imp_bytes"]) + len(r["code_bytes"]) for r in out["shared_uniform"]["results"]),
                 "shared_budget": sum(budgets)}
        entry["speedup"] = {m: entry["ms"]["loop_" + m]["median"] / entry["ms"]["batch_" + m]["median"] for m in ("uniform", "latitude16")}
        entry["memory"] = {name: memory_of(params, H, W, lambda cd, name=name: arms_of(cd, q, lv, budgets, P)[name])
                           for name in ("loop_uniform", "batch_uniform")}
        res["batch"].append(entry)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for budget_batch_timing.json")
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=2024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("budget_batch_timing: needs a CUDA device")
    line = dict(gpu_card())
    line["host_cpus"] = os.cpu_count()
    line["sizes"] = [run_size(H, W, a.reps, a.warmup, a.seed) for H, W in SIZES]
    s = json.dumps(line)
    print(s)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "budget_batch_timing.json"), "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
