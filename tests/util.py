"""Shared helpers for the parity tests."""
import functools
import glob
import hashlib
import os

import numpy as np
import torch

OPS_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ops_golden_*.npz")


@functools.lru_cache(maxsize=None)
def ops_golden():
    """Outputs of the reference extension for every op case, recorded on a B200 by tests/golden/make_golden.py:
    {"<case>/<key>[#sha256|#sub]": array}, stored in shards (tests/golden/ops_golden_*.npz) that each stay below 1 MB."""
    out = {}
    for f in sorted(glob.glob(OPS_GOLDEN)):
        with np.load(f) as z:
            out.update({k: z[k] for k in z.files})
    return out


def rng(seed):
    return np.random.default_rng(seed)


def t(a, dev="cuda:0"):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def n(x):
    return x.detach().to("cpu").numpy()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def rel_err(a, b):
    """norm-wise relative error max|a-b| / max|b| (the float tier is stated as 1e-5 relative)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


def conv_weights(r, nsets, cout, cin, scale=None):
    fan_in = cin * 25
    s = scale if scale is not None else (2.0 / fan_in) ** 0.5
    shape = (nsets, cout, cin, 5, 5) if nsets else (cout, cin, 5, 5)
    w = (r.standard_normal(shape) * s).astype(np.float32)
    bshape = (nsets, cout) if nsets else (cout,)
    b = (r.standard_normal(bshape) * 0.1).astype(np.float32)
    a = (0.25 + 0.1 * r.standard_normal(bshape)).astype(np.float32)
    return w, b, a


def random_tables(r, rows, ncode, total=65536):
    """strictly increasing integer CDF rows with a skewed distribution"""
    w = r.random((rows, ncode)) ** 3 + 1e-3
    cdf = np.cumsum(w / w.sum(1, keepdims=True), 1)
    tab = np.zeros((rows, ncode + 1), np.int64)
    tab[:, 1:] = np.round(cdf * total)
    for i in range(ncode):
        tab[:, i + 1] = np.maximum(tab[:, i + 1], tab[:, i] + 1)
    over = tab[:, -1] - total
    tab[:, -1] = total
    for i in range(ncode - 1, 0, -1):  # keep strict monotonicity from the top
        tab[:, i] = np.minimum(tab[:, i], tab[:, i + 1] - 1)
    assert (np.diff(tab, axis=1) > 0).all()
    return tab.astype(np.int32)


def synthetic_latent(seed, H=64, W=128, G=48, levels=48):
    """Config-1 style synthetic code-stream latent (SURVEY.md s8d): symbols q in {0..7} from a discretised Laplace
    around 3.5, importance levels smooth in latitude -> channel mask c < 4*L expanded and depth-to-width shuffled."""
    r = rng(seed)
    q = np.clip(np.round(r.laplace(3.5, 1.2, (1, G, H, W))), 0, 7).astype(np.float32)
    lat = np.cos((np.arange(H // 2) + 0.5) / (H // 2) * np.pi - np.pi / 2)  # (H/2,)
    lv = np.clip(np.round(levels * (0.25 + 0.6 * lat[:, None] + 0.1 * r.standard_normal((H // 2, W // 2)))), 0, levels)
    c = np.arange(4 * G)[None, :, None, None]
    mask192 = (c < 4 * lv[None, None]).astype(np.float32)  # (1,192,H/2,W/2)
    # depth-to-width (dtow_cuda.cu:38-56) in numpy
    m = mask192.reshape(1, G, 2, 2, H // 2, W // 2).transpose(0, 1, 4, 2, 5, 3).reshape(1, G, H, W)
    return q, np.ascontiguousarray(m), lv.astype(np.float32)[None, None]
