"""Records outputs of the UNMODIFIED reference CUDA extension (oracle/_ref/lic360_ref*.so, built for sm_100 by
oracle/Makefile.ref) on the B200 box for every case of tests/op_cases.py:

    python tests/golden/make_golden.py                # writes golden_out/ops_golden_*.npz
    cp golden_out/ops_golden_*.npz tests/golden/        # committed fixture

Bit-exact-tier arrays larger than 16K elements are stored as their SHA-256 only; float-tier arrays larger than that are
stored as a fixed strided subsample of 8192 elements (`<key>#sub`: flat[::size // 8192][:8192]) -- the full arrays are
covered by the live comparison in tests/test_gpu_ops.py::test_vs_reference_extension.  The arrays are split over as many
shards as keep each file below 1 MB (tests/util.py:ops_golden reads them back as one mapping).
"""
import hashlib
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.dirname(HERE), ROOT, os.path.join(ROOT, "360-image-compression_b200"), os.path.join(ROOT, "oracle", "_ref")):
    sys.path.insert(0, p)

import torch  # noqa: E402
import lic360_ref  # noqa: E402
from op_cases import CASES  # noqa: E402

assert torch.cuda.is_available()
out = {}
for case in CASES:
    try:
        res = case.run(lic360_ref, "cuda:0")
        torch.cuda.synchronize()
    except Exception as e:  # keep going: a reference op that cannot run is reported, not fatal
        print("REFERENCE FAILED on %s: %r" % (case.name, e))
        continue
    for k, v in res.items():
        if k in case.skip_ref:
            continue
        exactish = k in case.exact or k in case.libm
        if v.size <= 16384:
            out["%s/%s" % (case.name, k)] = v
        elif exactish:
            out["%s/%s#sha256" % (case.name, k)] = np.array(hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest())
        else:
            out["%s/%s#sub" % (case.name, k)] = np.ascontiguousarray(v).reshape(-1)[::v.size // 8192][:8192].copy()
    print("recorded", case.name, sorted(res))
dst = os.path.join(ROOT, "golden_out")
os.makedirs(dst, exist_ok=True)
shards, size = [{}], 0
for k, v in out.items():
    z = len(zlib.compress(np.ascontiguousarray(v).tobytes())) + 512
    if size + z > 900 * 1024 and shards[-1]:
        shards.append({})
        size = 0
    shards[-1][k], size = v, size + z
for i, s in enumerate(shards, 1):
    np.savez_compressed(os.path.join(dst, "ops_golden_%d.npz" % i), **s)
print("wrote", len(out), "arrays to", len(shards), "shards under", dst)
