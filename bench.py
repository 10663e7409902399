#!/usr/bin/env python
"""bench.py -- ERP Mpx/s, entropy encode+decode of the LIC360 context-model path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
  (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step returned to its caller as float32 .npy files:
imp_stream.npy and code_stream.npy (the two bitstreams, one value per byte), code.npy and mask.npy (the decoded latent and its
importance mask).  The inputs are seeded, so two builds run with the same arguments can be compared array for array.

A step = one pass of the hot path over one synthetic 512x1024 ERP image per GPU (BASELINE.json configs[1], batch 1):
importance stream + code stream ENCODE to the two bitstreams, then DECODE back to the latent, through the fused native
codec (360-image-compression_b200/csrc/codec.cu).  Every rank codes its own image (independent bitstreams, no
collective on the codec path, SURVEY.md s8e), so scaling is weak: value = N * 0.524288 Mpx * K / max-over-ranks time.

`value`  : inputs resident in HBM, outputs left in HBM.
`e2e`    : the same call with the latent in pinned HOST memory: H2D of (code, mask, importance levels) and D2H of the
           decoded (code, mask) inside the timed region.
`roofline`: the dominant kernel by time, wf_chain4_kernel (the code-stream decode critical path; latency-bound, with its latency
           model); `roofline_data_mover`: wf_old4_kernel (old terms of all 12 context-conv layers of a wavefront step, TMA-fed), the
           kernel that moves the data; both timed with CUDA events on the codec stream in one extra serialized decode.
           `flop_view`: algorithmic GFLOP / time against the fp32 and tensor peaks, encode and decode.
`cpu_baseline` / `--impl reference`: the CPU rendition (oracle/: OpenMP restatement of the conv/table ops + the
           reference's own host arithmetic coder when oracle/_ref is built) of the SAME 512x1024 image, all host threads.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "360-image-compression_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle", "_ref")):
    if p not in sys.path:
        sys.path.insert(0, p)

MPX = 512 * 1024 / 1e6
H, W, G = 64, 128, 48  # code latent of a 512x1024 image


def synthetic_latent(seed, h=H, w=W):
    from util import synthetic_latent as mk
    return mk(seed, H=h, W=w)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, threading.Event(), []

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag.is_set():
            try:
                out = subprocess.check_output(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"], timeout=5).decode().strip()
                self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ algorithmic work
def old_kernel_algorithmic_bytes():
    """Algorithmic bytes of one launch of the dominant kernel, wf_old_kernel (old terms of all 12 layers x 3 nets of one
    code-stream wavefront step), averaged over the 238 steps of a decode (DESIGN.md s5): the non-zero old-term weights
    of the output groups present in the slab (read once), the activations of wavefronts <= p-2 that carry a non-zero
    weight for at least one slab output (read once), and the P sums (16 B per slab position, layer and net, written once)."""
    import numpy as np
    npos = np.zeros(H + W - 1, np.int64)
    for d in range(H + W - 1):
        npos[d] = min(d, H - 1) - max(0, d - W + 1) + 1
    layers = [(1, 4)] + [(4, 4)] * 10 + [(4, 3)]
    nsteps = H + W + G - 2
    total = 0
    for cin, cout in layers:
        nnz_g = np.zeros(G, np.int64)  # old-term weights of output group g: taps (kh,kw) x input groups <= g + 2 - s
        for g in range(G):
            for s in range(9):
                ntap = min(s, 8 - s) + 1
                nnz_g[g] += ntap * max(0, min(G, g + 3 - s)) * cin * cout
        for psum in range(nsteps):
            la, lb = max(0, psum - G + 1), min(psum, H + W - 2)
            wbytes = 4 * 3 * sum(int(nnz_g[psum - d]) for d in range(la, lb + 1))
            obytes = 16 * 3 * int(npos[la:lb + 1].sum())
            ibytes = 0
            for e in range(max(0, la - 4), min(H + W - 2, lb + 4) + 1):
                ibytes += 4 * 3 * cin * int(npos[e]) * max(0, min(G, psum - 1 - e))
            total += wbytes + obytes + ibytes
    return total / nsteps, nsteps


def chain_kernel_algorithmic_bytes():
    """Algorithmic bytes of one launch of wf_chain4_kernel (code stream: the 12-layer chain of same-wavefront terms of a step with
    bias / PReLU / TileAdd fused, the CDF rows of the step, and the previous-wavefront terms of the next step), averaged over
    the 238 steps.  Every byte is counted once: P and R sums read, the step's activations written in both frame layouts and read
    once by the layer above, the residual, the same-wavefront / previous-wavefront weights of the output groups present, rows."""
    import numpy as np
    npos = np.zeros(H + W - 1, np.int64)
    for d in range(H + W - 1):
        npos[d] = min(d, H - 1) - max(0, d - W + 1) + 1
    nsteps = H + W + G - 2

    def slab(p):
        if p >= nsteps:
            return 0, 0
        la, lb = max(0, p - G + 1), min(p, H + W - 2)
        return int(npos[la:lb + 1].sum()), lb - la + 1

    total = 0
    for p in range(nsteps):
        L, Dg = slab(p)
        L1, Dg1 = slab(p + 1)
        per_net = 12 * L * (16 + 16 + 16 + 32) + 5 * L * 16 + 11 * Dg * 1600 + Dg * 400 + 12 * Dg * 32
        rows = L * (36 + 16)
        rtail = 11 * (L1 * (16 + 16) + Dg1 * 1600)
        total += 3 * (per_net + rtail) + rows
    return total / nsteps


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_arm(steps, warmup, sample_hw=(H, W)):
    """CPU rendition of the same workload: one (8*h)x(8*w)-pixel ERP image worth of latent (default: the full 512x1024 image of
    configs[1], ~20 s per step on the GPU box's host cores), all host threads."""
    import numpy as np
    import torch
    from oracle import cpu_codec
    import lic360_codec_ops as ops
    h, w = sample_hw
    q, mask, lv = synthetic_latent(2024, h, w)
    params = {'code': ops.make_entropy_params(48, 4, 3, 3, 2024, 'cpu'), 'imp': ops.make_entropy_params(1, 144, 49, None, 2025, 'cpu')}
    codec = cpu_codec.CpuCodecFast(cpu_codec.params_to_numpy(params))  # channel-last SIMD dot products, same streams (oracle/cpu_codec.py)
    px = (8 * h) * (8 * w) / 1e6
    times = []
    for _ in range(warmup + steps):
        t0 = time.time()
        bi, bc = codec.encode(q, mask, lv)
        code, m = codec.decode(bi, bc, h // 2, w // 2)
        times.append(time.time() - t0)
        assert np.array_equal(code, q * mask) and np.array_equal(m, mask)
    t = sum(times[warmup:]) / steps
    from oracle import oracle as O
    return {"value": px / t, "unit": "Mpx/s", "cores": os.cpu_count(), "kind": "port", "steps_timed": steps,
            "sample": "%dx%d-pixel ERP latent (1,48,%d,%d)+(1,1,%d,%d), encode+decode, OpenMP channel-last fp32 conv + oracle tables + %s host coder, %.1f s/step"
                      % (8 * h, 8 * w, h, w, h // 2, w // 2, "reference" if O.have_ref_coder() else "restated", t)}, t, (bi, bc, code, m)


def workload_config(h=H, w=W):
    """`config` of the JSON line, identical for both arms (the reference arm times the same workload on the host cores)"""
    return {"workload": "configs[1]: 512x1024 ERP entropy encode+decode (importance + code stream), batch 1 per GPU, model-idx-3 shape, seeded random-init weights"
                        + ("" if (h, w) == (H, W) else " -- REDUCED sample, latent %dx%d" % (h, w)),
            "latent": [1, 48, h, w], "images_per_gpu_per_step": 1, "l2": "256 MB buffer written between iterations (L2 flush)",
            "parallelism": "image-sharded, no collective"}


def emit(line, real_stdout):
    """the ONE JSON line of the contract, on the real stdout (everything else -- NCCL banners included -- goes to stderr)"""
    os.write(real_stdout, (json.dumps(line) + "\n").encode())


def dump_outputs(dst, imp_stream, code_stream, code, mask):
    """the last timed step's results as float32 arrays: bitstreams one value per byte, decoded code and mask as returned"""
    import numpy as np
    os.makedirs(dst, exist_ok=True)
    arrays = {"imp_stream": np.frombuffer(imp_stream, np.uint8), "code_stream": np.frombuffer(code_stream, np.uint8),
              "code": np.asarray(code), "mask": np.asarray(mask)}
    for name, a in arrays.items():
        np.save(os.path.join(dst, name + ".npy"), a.astype(np.float32))


def main():
    # keep stdout clean: libraries (NCCL prints its version banner to stdout) write to fd 1, which now points at stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-ext", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        # reference arm: the CPU implementation of the path on the host cores; rank 0 alone runs it
        if rank != 0:
            return
        # torchrun exports OMP_NUM_THREADS=1 to every worker unless the user set it; this arm is meant to use all host threads
        # (the variable has to be right before libgomp / torch are loaded, which happens inside cpu_arm)
        if world > 1 or "TORCHELASTIC_RUN_ID" in os.environ:
            if os.environ.get("OMP_NUM_THREADS", "1") == "1":
                os.environ["OMP_NUM_THREADS"] = str(os.cpu_count())
        os.environ.setdefault("OMP_WAIT_POLICY", "passive")  # ~3000 short parallel regions per image: do not burn the cores between them
        # the SAME config and the same K / W as the b200 arm: one full 512x1024 image per step (about 20 s of CPU work per step on the
        # box's host cores; LIC360_BENCH_REF_SAMPLE=h,w shrinks the latent for a quick look, and says so in `config`)
        steps, ref_warm = args.steps, max(0, args.warmup)
        hw = tuple(int(v) for v in os.environ.get("LIC360_BENCH_REF_SAMPLE", "%d,%d" % (H, W)).split(","))
        cb, t, outs = cpu_arm(steps, ref_warm, hw)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, *outs)
        line = {"impl": "reference", "metric": "ERP Mpx/s encode+decode (entropy path, model-idx 3 shape)", "value": cb["value"], "unit": "Mpx/s",
                "n_gpus": args.gpus, "steps": cb["steps_timed"], "warmup": ref_warm, "ms_per_step": t * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(*hw),
                "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line, real_stdout)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (there is no CPU path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import lic360
    import lic360_pipeline as pl
    import lic360_shard as sh

    q, mask, lv = synthetic_latent(2024 + rank)
    params = pl.make_codec_params(dev, seed=2024)
    codec = pl.FusedCodec(params, H=H, W=W, gid=local_rank)
    host = [torch.from_numpy(a).pin_memory() for a in (q, mask, lv)]
    tq, tm, tl = [h.to(dev) for h in host]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(steps, e2e):
        nbytes, timing = None, {"enc": [], "dec": []}
        for _ in range(steps):
            flush.zero_()  # L2 flush between iterations
            if e2e:
                a, b, c = [h.to(dev, non_blocking=True) for h in host]
            else:
                a, b, c = tq, tm, tl
            bi, bc = codec.encode(a, b, c)
            timing["enc"].append(codec.last_timing())
            code, mup = codec.decode(bi, bc)
            timing["dec"].append(codec.last_timing())
            if e2e:
                code_h, mask_h = code.cpu(), mup.cpu()
            nbytes = (len(bi), len(bc))
        return nbytes, timing, (code, mup, bi, bc)

    def timed(steps, e2e):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lic360.launch_count()
        e0.record()
        nbytes, timing, outs = run(steps, e2e)
        e1.record()
        barrier()
        ms = sh.max_over_ranks(e0.elapsed_time(e1), dev)  # device time of the slowest rank
        return ms, nbytes, timing, outs, lic360.launch_count() - l0

    run(warmup, False)
    # decode mode of the one-image-at-a-time figures: 0 = graph replay per wavefront step, 2 = low latency (one persistent code-stream
    # chain kernel per decode, include/lic360_b200.h).  "auto": time both after the warm-up, keep the faster one -- if mode 2 is exact.
    decode_mode, mode_note = 0, "graph replay per step"
    want = os.environ.get("LIC360_BENCH_DECODE_MODE", "auto")
    if want in ("auto", "2"):
        med, why = {0: float("inf"), 2: float("inf")}, ""
        try:
            bi_, bc_ = codec.encode(tq, tm, tl)
            for m in (0, 2):
                codec.set_mode(m)
                ts = []
                for _ in range(4):
                    torch.cuda.synchronize()
                    t0 = time.time()
                    c_, m_ = codec.decode(bi_, bc_)
                    torch.cuda.synchronize()
                    ts.append(time.time() - t0)
                    if not (bool(torch.equal(c_, tq * tm)) and bool(torch.equal(m_, tm))):
                        raise RuntimeError("mode %d did not decode exactly" % m)
                med[m] = sorted(ts)[1] * 1e3
        except Exception as e:  # the default mode always works
            med[2], why = float("inf"), " (low-latency mode unavailable: %r)" % (e,)
        # every rank takes the same decision (collectives outside the try block: all ranks get here)
        m0, m2 = sh.max_over_ranks(med[0], dev), sh.max_over_ranks(med[2], dev)
        if m2 != float("inf") and (want == "2" or m2 < m0):
            decode_mode, mode_note = 2, "low latency: one persistent code-stream chain kernel per decode"
        mode_note += " (probe, slowest rank: %.2f ms graph replay, %.2f ms low latency)%s" % (m0, m2, why)
    codec.set_mode(decode_mode)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, nbytes, timing, outs, launches = timed(args.steps, False)
    if sampler:
        sampler.stop_flag.set()
        sampler.join()
    ok = bool(torch.equal(outs[0], tq * tm)) and bool(torch.equal(outs[1], tm))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs[2], outs[3], outs[0].cpu().numpy(), outs[1].cpu().numpy())
    run(1, True)
    ms_e2e, _, _, _, _ = timed(args.steps, True)

    # ---- secondary figures: several images in flight per GPU (one codec + its host threads each), so that the host arithmetic coder
    # of one image overlaps the GPU steps of another (INTEGRATION.md s3).  A queue of images is drained by `nfly` workers per rank.
    def in_flight(codecs, images, repeat):
        """images: list of (code, mask, levels) device tensors; every worker pulls the next image index until repeat * len(images)
        images are coded; returns (ms of the slowest rank, all round trips exact)"""
        import itertools
        counter, lock = itertools.count(), threading.Lock()
        total, res = repeat * len(images), [True] * len(codecs)

        def worker(k, cd):
            while True:
                with lock:
                    i = next(counter)
                if i >= total:
                    break
                a, b, c = images[i % len(images)]
                code, mup = cd.decode(*cd.encode(a, b, c))
                res[k] = res[k] and bool(torch.equal(code, a * b)) and bool(torch.equal(mup, b))

        barrier()
        t0 = time.time()
        th = [threading.Thread(target=worker, args=(k, cd)) for k, cd in enumerate(codecs)]
        for t_ in th:
            t_.start()
        for t_ in th:
            t_.join()
        torch.cuda.synchronize()
        return sh.max_over_ranks((time.time() - t0) * 1e3, dev), all(res)

    codec.set_mode(0)  # several images in flight: every decode keeps the SMs only while it computes
    piped_ms = None
    try:
        # each image in flight has 2 polling host threads (importance + code stream): 4 per GPU alone on the box, 2 when N ranks share it
        nfly = max(2, int(os.environ.get("LIC360_BENCH_IN_FLIGHT", "4" if world == 1 else "2")))
        codecs = [codec] + [pl.FusedCodec(params, H=H, W=W, gid=local_rank) for _ in range(nfly - 1)]
        for cd in codecs:
            cd.decode(*cd.encode(tq, tm, tl))
        piped_ms, piped_ok = in_flight(codecs, [(tq, tm, tl)], nfly * args.steps)
        del codecs
    except Exception as e:  # secondary figure only
        piped_ms, piped_ok = None, repr(e)

    # ---- configs[2]: LIC3602K shape, 16 images of 1024x2048 (latent 128x256) sharded by image over the ranks (16 / N per GPU), queue
    # drained by up to 4 (N = 1) or 2 (N > 1) codecs per GPU; no collective on the codec path
    cfg3 = None
    try:
        if os.environ.get("LIC360_BENCH_NO_CONFIG3"):
            raise RuntimeError("disabled by LIC360_BENCH_NO_CONFIG3")
        n_img = max(1, 16 // world)
        nfly3 = min(n_img, 4 if world == 1 else 2)
        imgs3 = []
        for i in range(n_img):
            a, b, c = synthetic_latent(3000 + 16 * rank + i, 128, 256)
            imgs3.append(tuple(torch.from_numpy(v).to(dev) for v in (a, b, c)))
        codecs3 = [pl.FusedCodec(params, H=128, W=256, gid=local_rank) for _ in range(nfly3)]
        for cd in codecs3:
            cd.decode(*cd.encode(*imgs3[0]))
        ms3, ok3 = in_flight(codecs3, imgs3, 1)
        cfg3 = {"value": world * n_img * (1024 * 2048 / 1e6) / (ms3 / 1e3), "unit": "Mpx/s", "images": world * n_img, "images_per_gpu": n_img,
                "in_flight_per_gpu": nfly3, "image": [1024, 2048], "latent": [1, 48, 128, 256], "ms_total": ms3, "round_trip_exact": ok3,
                "timing": "host wall clock around all worker threads, max over ranks",
                "note": "configs[2]: batch of 16 LIC3602K-shape images sharded by image, encode + decode of both streams of every image"}
        del codecs3, imgs3
    except Exception as e:  # secondary figure only
        cfg3 = {"unavailable": repr(e)}

    # ---- configs[3]: ONE 2048x4096 image (latent 256x512), decode stress.  Inside an image the wavefront and the arithmetic-coded
    # stream are sequential, so the reference's format does not shard (single stream: one GPU, see DESIGN.md s6); the latitude-band
    # FORMAT EXTENSION does (lic360_shard.BandCodec: 8 independently coded bands of 32 latent rows, dealt round-robin to the ranks).
    cfg4 = None
    try:
        if os.environ.get("LIC360_BENCH_NO_CONFIG4"):
            raise RuntimeError("disabled by LIC360_BENCH_NO_CONFIG4")
        H4, W4, NB4 = 256, 512, 8
        a4, b4, c4 = [torch.from_numpy(v).to(dev) for v in synthetic_latent(4000, H4, W4)]  # the same image on every rank
        bands = sh.BandCodec(lambda h, w: pl.FusedCodec(params, H=h, W=w, gid=local_rank), H4, W4, NB4, world=world, rank=rank,
                             in_flight=4 if world == 1 else 2)
        blob4 = bands.encode(a4, b4, c4)
        bands.decode_local(blob4)  # warm-up
        barrier()
        t0 = time.time()
        local4 = bands.decode_local(blob4)
        torch.cuda.synchronize()
        ms4 = sh.max_over_ranks((time.time() - t0) * 1e3, dev)
        ok4 = all(bool(torch.equal(cb, (a4 * b4)[:, :, r0:r1])) and bool(torch.equal(mb, b4[:, :, r0:r1]))
                  for bnd, (cb, mb) in local4.items() for r0, r1 in [bands.rows[bnd]])
        cfg4 = {"value": (2048 * 4096 / 1e6) / (ms4 / 1e3), "unit": "Mpx/s (decode only)", "image": [2048, 4096], "latent": [1, 48, H4, W4],
                "bands": NB4, "bands_per_gpu": len(bands.mine), "in_flight_per_gpu": len(bands.codecs), "decode_ms": ms4,
                "container_bytes": len(blob4), "round_trip_exact": ok4, "timing": "host wall clock around this rank's bands, max over ranks",
                "note": "configs[3]: one 2048x4096 image as 8 independently coded latitude bands (format extension: per band the bytes are what "
                        "the codec emits for the band as an image of its own); the single-stream decode of the same image takes 218 ms on one GPU"}
        del bands, local4
    except Exception as e:  # secondary figure only
        cfg4 = {"unavailable": repr(e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * MPX * args.steps / (ms / 1e3)
    e2e_value = world * MPX * args.steps / (ms_e2e / 1e3)
    mean = lambda k, xs: sum(x[k] for x in xs) / len(xs)
    # ---- roofline of the dominant kernel: one more decode with the same kernels launched one by one on the codec stream
    # and CUDA events between them (lic360_codec_set_mode(1)); wf_old_kernel launches once per wavefront step
    codec.set_mode(1)
    codec.decode(*codec.encode(tq, tm, tl))
    kt, kt_imp = codec.kernel_times(0), codec.kernel_times(1)
    codec.set_mode(0)
    alg_bytes, n_old = old_kernel_algorithmic_bytes()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    prof = {}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "old_kernel_summary.json")))
    except Exception:
        pass
    old_launch_us = kt["old_ms"] / max(kt["steps"], 1) * 1e3
    achieved = alg_bytes / (old_launch_us * 1e-6) / 1e9
    # FLOP view (SURVEY.md s8d: 2 x non-zero MACs): 253.9 GFLOP code stream + 13.2 GFLOP importance stream per image and direction
    gflop = 253.9 + 13.2
    fp32_peak = 148 * 128 * 2 * (peaks.get("sm_max_mhz", 1965.0) * 1e6) / 1e12        # TFLOP/s, FFMA on every lane at max clock
    enc_ms, dec_ms = mean("total_ms", timing["enc"]), mean("total_ms", timing["dec"])
    enc_gpu_ms = enc_ms - mean("host_coder_ms", timing["enc"])
    flop_view = {"algorithmic_gflop_per_image_per_direction": gflop, "fp32_peak_tflops": fp32_peak,
                 "tensor_peaks_tflops": {"bf16_dense_measured": peaks.get("bf16_tflops_sustained"), "tf32_mma_sync_measured": 276.0},
                 "encode": {"ms": enc_ms, "gpu_ms": enc_gpu_ms, "tflops_over_gpu_ms": gflop / enc_gpu_ms, "frac_fp32_peak": gflop / enc_gpu_ms / fp32_peak},
                 "decode": {"ms": dec_ms, "tflops": gflop / dec_ms, "frac_fp32_peak": gflop / dec_ms / fp32_peak},
                 "note": "the context conv runs as IEEE fp32 FMA (fma.rn.f32x2) on the CUDA cores; tools/mma_probe.cu measured mma.sync TF32 at 276 TFLOP/s "
                         "on this GPU, i.e. 92 TFLOP/s for the 3-way split that the 1e-5 tier needs (1.2x the fp32 peak) -- see DESIGN.md s3"}
    chain_us = kt["chain_ms"] / max(kt["steps"], 1) * 1e3
    chain_bytes = chain_kernel_algorithmic_bytes()
    chain_gbs = chain_bytes / (chain_us * 1e-6) / 1e9
    # the dominant kernel BY TIME is the code-stream chain (the decode critical path); it runs on 24 SMs and is latency-bound
    roofline_chain = {"bound": "hbm", "kernel": "wf_chain4_kernel (code stream: 12-layer chain of same-wavefront terms of one wavefront step, 3 clusters x 8 CTAs, "
                                               "CDF rows and next-step previous-wavefront terms fused)",
                      "achieved": chain_gbs, "peak": peak, "unit": "GB/s", "frac": chain_gbs / peak, "traffic": prof.get("chain4_dram_bytes_per_launch"),
                      "algorithmic_bytes_per_launch": chain_bytes, "avg_launch_us": chain_us, "launches_per_decode": n_old,
                      "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)",
                      "latency_model": {"layers": 12, "cluster_barrier_us": 0.75, "dependent_item_us": 2.5, "weight_staging_and_prefetch_us": 1.1,
                                        "floor_us": 12 * (0.75 + 2.5), "measured_chain_us_in_pipeline": 51.0,
                                        "note": "per-layer phases measured with LIC360_WF_TRACE=1 (DESIGN.md s4.1); the launch time here also contains the fused CDF rows "
                                                "(21 erff per symbol) and the previous-wavefront terms of the next step"},
                      "note": "latency-bound kernel on 24 of 148 SMs: the bandwidth fraction is reported because the contract asks for it, the latency model is what bounds it"}
    roofline = {"bound": "hbm", "kernel": "wf_old4_kernel (TMA-fed old-term context conv of all 12 layers x 3 nets of a wavefront step, code stream; four positions per lane, two diagonals per warp)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": prof.get("dram_bytes_per_launch"),
                "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_us": old_launch_us, "launches_per_decode": n_old,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)",
                "traffic_note": prof.get("note"), "traffic_step_algorithmic_bytes": prof.get("algorithmic_bytes_this_step"),
                "kernel_ms_per_decode": {"code": kt, "importance": kt_imp},
                "shares_under_ncu": prof.get("shares_of_summed_gpu_time_under_ncu"),
                "note": "avg launch = CUDA-event time around every old-term kernel launch (wf_old4_kernel) of one serialized decode on the codec stream (DESIGN.md s5). "
                        "the old-term kernel is the kernel that moves the data and occupies the whole GPU; the chain kernels (chain_ms: 24 resp. 16 SMs, "
                        "cluster barriers, incl. the fused CDF rows and next-step R terms) are latency-bound and have no bandwidth roofline"}
    line = {"metric": "ERP Mpx/s encode+decode (entropy path, model-idx 3 shape)", "value": value, "unit": "Mpx/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": dict(workload_config(), decode_mode=decode_mode, decode_mode_note=mode_note),
            "e2e": {"value": e2e_value, "unit": "Mpx/s", "h2d_bytes_per_step": int(sum(h.numel() * 4 for h in host)),
                    "d2h_bytes_per_step": int(2 * tq.numel() * 4), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches), "roofline": roofline_chain, "roofline_data_mover": roofline, "flop_view": flop_view,
            "breakdown_ms": {"encode": mean("total_ms", timing["enc"]), "encode_host_coder": mean("host_coder_ms", timing["enc"]),
                             "decode": mean("total_ms", timing["dec"]), "decode_host_coder": mean("host_coder_ms", timing["dec"]),
                             "decode_importance_stream": mean("imp_stream_ms", timing["dec"]), "decode_waiting_for_gpu": mean("gpu_wait_ms", timing["dec"])},
            "bitstream": {"imp_bytes": nbytes[0], "code_bytes": nbytes[1], "bpp": (nbytes[0] + nbytes[1]) * 8 / (512 * 1024), "round_trip_exact": ok}}
    if piped_ms:
        line["images_in_flight"] = {"value": world * nfly * args.steps * MPX / (piped_ms / 1e3), "unit": "Mpx/s", "images_in_flight_per_gpu": nfly,
                                        "round_trip_exact": piped_ok, "timing": "host wall clock around all worker threads, max over ranks",
                                        "note": "secondary figure; `value` and `e2e` are one image at a time"}
    line["config3_1024x2048_batch16"] = cfg3
    line["config4_2048x4096_bands"] = cfg4
    if sampler:
        line["clocks"] = sampler.summary()
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_arm(1, 0)[0]
        except Exception as e:  # the CPU arm is a reported baseline; never let it take the bench line down
            line["cpu_baseline"] = {"value": None, "unit": "Mpx/s", "cores": os.cpu_count(), "kind": "port", "sample": "failed: %r" % (e,)}
    if world == 1 and not args.no_ref_ext:
        # reported baseline A (BASELINE.md s4): the unmodified reference CUDA extension rebuilt for sm_100, same loops
        try:
            import lic360_ref
            ref = pl.PerOpCodec(lic360_ref, params, gid=local_rank)
            ref.encode(tq, tm, tl)
            torch.cuda.synchronize()
            t0 = time.time()
            rbi, rbc = ref.encode(tq, tm, tl)
            rc, rm = ref.decode(rbi, rbc, H // 2, W // 2)
            torch.cuda.synchronize()
            t1 = time.time()
            line["reference_cuda_ext"] = {"value": MPX / (t1 - t0), "unit": "Mpx/s", "ms_per_step": (t1 - t0) * 1e3, "imp_bytes": len(rbi), "code_bytes": len(rbc),
                                          "identical_bytes_to_b200": (rbi, rbc) == tuple(codec.encode(tq, tm, tl)), "round_trip_exact": bool(torch.equal(rc, tq * tm)),
                                          "note": "oracle/_ref/lic360_ref*.so driven by the per-op loops of lic360_demo.py; reported, not the target"}
        except Exception as e:
            line["reference_cuda_ext"] = {"unavailable": repr(e)}
    emit(line, real_stdout)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
