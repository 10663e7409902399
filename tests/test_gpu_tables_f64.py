"""GPU: the CDF table kernels (EntropyGmmTableOp.forward / forward_batch, EntropyTableOp) against the float64 statement of
their formulas (ref64.py), at row counts that cover one row, a partial CTA, whole CTAs and a large grid, on random inputs
and on the adversarial rows of test_ref64.py."""
import numpy as np
import pytest
import torch

import ref64
from test_ref64 import adversarial_gmm, adversarial_logits
from util import n, rng, t

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROWS = [1, 31, 4096, 400003]


def _gmm_rows(rows, seed):
    """adversarial rows first (cycled), then random mixtures whose bins are mostly clear of the fix-up"""
    r = rng(seed)
    w = (r.standard_normal((rows, 3)) * 2).astype(np.float32)
    d = (np.abs(r.standard_normal((rows, 3))) * 1.5 + 0.3).astype(np.float32)
    m = (r.standard_normal((rows, 3)) * 2.5).astype(np.float32)
    aw, ad, am = adversarial_gmm()
    k = min(rows, 3 * len(aw)) if rows > 1 else 0
    sel = np.arange(k) % len(aw)
    w[:k], d[:k], m[:k] = aw[sel], ad[sel], am[sel]
    if rows == 1:
        w[0], d[0], m[0] = aw[3], ad[3], am[3]
    return w, d, m


def _check(T_kernel, T64, mg, x, gmm, rows):
    assert T_kernel.shape == T64.shape
    bad = ref64.check_table_properties(T_kernel)
    assert len(bad) == 0, ("invalid kernel rows", bad[:5], T_kernel[bad[:3]])
    ok, how = ref64.compare(T_kernel, T64, mg, x, gmm)
    first = np.nonzero(~ok)[0]
    assert ok.all(), ("%d rows differ from the float64 tables; first %d: kernel %s float64 %s" %
                      (len(first), first[0], T_kernel[first[0]], T64[first[0]]))
    # the uncompared rows (an ambiguous bin next to the fix-up) stay a small share
    assert (how == 2).sum() <= max(1, 0.15 * rows), np.bincount(how, minlength=3)


@pytest.mark.parametrize("rows", ROWS)
def test_gmm_table_forward_against_float64(rows):
    import lic360
    w, d, m = _gmm_rows(rows, 1000 + rows)
    tw, td, tm = [t(v.reshape(1, 3, 1, rows), DEV) for v in (w, d, m)]
    op = lic360.EntropyGmmTableOp(8, 3.5, 3, 65536, 1e-6, 0, False)
    out = n(op.forward(tw, td, tm, torch.tensor([rows], dtype=torch.int32))[0])
    T64, mg, x = ref64.gmm_table64(w, d, m)
    _check(out.astype(np.int64), T64, mg, x, True, rows)
    # the op leaves the softmax weights and the clamped deltas in place of its inputs
    dd = np.where(d < 0, np.float32(1e-6), d + np.float32(1e-6))
    assert np.array_equal(n(td).reshape(rows, 3), dd)
    assert np.abs(n(tw).reshape(rows, 3).sum(1) - 1).max() < 1e-6


@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("rows", ROWS)
def test_gmm_table_forward_batch_against_float64(rows, B):
    import lic360
    w, d, m = _gmm_rows(rows, 2000 + rows + B)
    per = (rows + B - 1) // B + 5                 # tile-buffer capacity above the row count: rows stop at tnum
    buf = np.full((3 * B, 3, 1, per), np.nan, np.float32)
    stride = 3 * B * per
    flat = buf.reshape(-1)
    for k, v in enumerate((w, d, m)):
        flat[k * stride:k * stride + rows * 3] = v.reshape(-1)
    op = lic360.EntropyGmmTableOp(8, 3.5, 3, 65536, 1e-6, 0, False)
    out = n(op.forward_batch(t(buf, DEV), torch.tensor([rows], dtype=torch.int32))[0])
    assert out.shape == (B * per, 9)
    T64, mg, x = ref64.gmm_table64(w, d, m)
    _check(out[:rows].astype(np.int64), T64, mg, x, True, rows)


@pytest.mark.parametrize("nlog", [49, 5, 64])
@pytest.mark.parametrize("rows", ROWS)
def test_entropy_table_against_float64(rows, nlog):
    import lic360
    r = rng(3000 + rows + nlog)
    x = (r.standard_normal((rows, nlog)) * (0.6 if nlog > 8 else 2)).astype(np.float32)
    adv = adversarial_logits(nlog)
    k = min(rows, 3 * len(adv)) if rows > 1 else 0
    x[:k] = adv[np.arange(k) % len(adv)]
    if rows == 1:
        x[0] = adv[0]
    op = lic360.EntropyTableOp(nlog, 65536, 0, False)
    out = n(op.forward(t(x.reshape(1, nlog, 1, rows), DEV), torch.tensor([rows], dtype=torch.int32))[0])
    T64, mg, val = ref64.entropy_table64(x)
    _check(out.astype(np.int64), T64, mg, val, False, rows)
