"""Float64 statement of the two CDF table formulas, with the rounding margin of every bin.

gmm_table64     -- EntropyGmmTable (entropy_gmm_table_cuda.cu:29-107): softmax of the mixture logits, delta clamp,
                   T[pt] = int(total * sum_i w_i * Phi((v_pt - m_i) / d_i) + 0.5), then the GMM fix-up.
entropy_table64 -- EntropyTable (entropy_table_cuda.cu:24-96): softmax, a_i = int(total * p_i + 0.5),
                   T[i+1] = min(T[i] + a_i, total), T[w] = total, then the EntropyTable fix-up.

Both start from the fp32 values the kernels start from (the fp32 inputs, s2 = float(1/sqrt(2)), the bin edge
v = float(pt - 1 - bias) + 0.5 rounded to float, beta = float(1e-6)) and carry everything after that in float64.

Margin: for every rounded value x = total * p + 0.5 (a bin of the GMM table, a per-symbol count of the softmax table)
the distance of x from the nearest integer, in counts.  Where it is at least MARGIN = 0.1, every correct fp32
evaluation of the formula rounds to the float64 integer.  The fp32 error budget of one GMM bin (ng = 3):
  - the erff argument s2 * (v - m) / d takes four roundings (the clamp d + beta, the difference, the product, the
    division): at most 4u relative (u = 2^-24); Phi moves by at most |a| e^(-a^2) / sqrt(pi) <= 0.25 times the relative
    argument error, so 65536 * 0.25 * 4u = 0.004 counts;
  - erff is within 2 ulp and the fmaf 0.5 + 0.5 e rounds once: below 2e-7 absolute, 0.013 counts per component;
  - the softmax weights (expf, the fp32 sum, the division): below 5u relative, 0.02 counts;
  - the fp32 accumulation of three products into ps <= 1: below 3u, 0.012 counts.
That is about 0.05 counts, so 0.1 leaves a factor of two.  total * ps is exact (a power of two times a float).
The softmax table's counts see the same few ulp (expf, x - max, total / psum, the product: below 0.02 counts) plus
the fp32 running sum of the 49 exponentials, whose rounding grows with the number of terms: its bound,
u * sum_k S_k / S_w (S_k the partial sums in index order), times the count, is subtracted from the margin, so the
same MARGIN applies to both tables.  Everything after the rounding (prefix sums, clipping, fix-up) is integer
arithmetic that fp32 represents exactly below 2^24.
A row with any bin inside the margin is left out of the exact row comparison (compare() says what is still checked
there); the callers count such rows.
"""
import numpy as np
from scipy.special import erfc

MARGIN = 0.1
_U = 2.0 ** -24


def _dist(x):
    f = x - np.floor(x)
    return np.minimum(f, 1.0 - f)


def fixup64(o, gmm_rule):
    """The strictly-increasing fix-up of fixup_row (tables_dev.cuh) on integer rows (rows, n + 1), in place.
    gmm_rule: bump where T[i+1] <= T[i] (T[i] already raised, T[i+1] not yet); otherwise where T[i+1] + bias <= T[i]."""
    rows, nt = o.shape
    bias = np.zeros(rows, np.int64)
    mval = np.zeros(rows, np.int64)
    midx = np.zeros(rows, np.int64)
    for i in range(nt - 1):
        bump = (o[:, i + 1] <= o[:, i]) if gmm_rule else (o[:, i + 1] + bias <= o[:, i])
        bias += bump
        o[:, i + 1] += bias
        d = o[:, i + 1] - o[:, i]
        upd = d > mval
        mval = np.where(upd, d, mval)
        midx = np.where(upd, i, midx)
    for i in range(nt - 1):
        sel = (bias > 0) & (i >= midx)
        o[sel, i + 1] -= bias[sel]
    return o


def gmm_table64(w, d, m, nstep=8, bias=3.5, total=65536, beta=1e-6):
    """w, d, m: (rows, ng) mixture logits, deltas, means.  Returns (table int64 (rows, nstep + 1), margin (rows, nstep - 1)
    of the interior bins 1..nstep-1, their unrounded values total * ps + 0.5)."""
    w, d, m = [np.asarray(a, np.float32).astype(np.float64) for a in (w, d, m)]
    e = np.exp(w - w.max(1, keepdims=True))
    p = e / e.sum(1, keepdims=True)
    b32 = np.float64(np.float32(beta))
    dd = np.where(d < 0, b32, d + b32)
    s2 = np.float64(np.float32(1.0 / np.sqrt(2.0)))
    pts = np.arange(1, nstep)
    v = (np.float32(pts - 1) - np.float32(bias) + np.float32(0.5)).astype(np.float32).astype(np.float64)
    a = s2 * (v[None, :, None] - m[:, None, :]) / dd[:, None, :]        # (rows, nstep - 1, ng)
    ps = (p[:, None, :] * 0.5 * erfc(-a)).sum(2)
    x = total * ps + 0.5
    T = np.zeros((w.shape[0], nstep + 1), np.int64)
    T[:, 1:nstep] = np.floor(x)
    T[:, nstep] = total
    return fixup64(T, True), _dist(x), x


def entropy_table64(logits, total=65536):
    """logits (rows, w).  Returns (table int64 (rows, w + 1), margin (rows, w - 1) of the rounded counts a_0..a_{w-2},
    the unrounded counts + 0.5)."""
    x = np.asarray(logits, np.float32).astype(np.float64)
    t = np.exp(x - x.max(1, keepdims=True))
    S = np.cumsum(t, 1)
    p = t / S[:, -1:]
    val = total * p[:, :-1] + 0.5
    a = np.floor(val).astype(np.int64)
    gamma = _U * S[:, 1:].sum(1) / S[:, -1]                                # running-sum bound, relative
    margin = _dist(val) - total * p[:, :-1] * gamma[:, None]
    rows, nw = x.shape
    T = np.zeros((rows, nw + 1), np.int64)
    T[:, 1:nw] = np.minimum(np.cumsum(a, 1), total)
    T[:, nw] = total
    return fixup64(T, False), margin, val


def clear_rows(margin):
    """rows whose every bin is outside the margin"""
    return (margin >= MARGIN).all(1)


def compare(T_kernel, T64, margin, x, gmm):
    """Check a kernel's integer table against the float64 one.  Returns (ok, how) per row.
    how == 0: every bin is outside the margin, and the row must equal the float64 row exactly.
    how == 1: some bins are inside the margin, but the float64 row needs no fix-up and stays clear of it under any +-1
              at those bins (GMM: interior bins at least 3 apart; softmax: every count >= 3 and no clipping); then the
              rounded values themselves can be read off the kernel's row (the GMM bins / the softmax counts T[i+1] - T[i])
              and each must be the float64 integer outside the margin, and one of the two integers next to x inside it.
    how == 2: not compared (an ambiguous bin next to the fix-up or the clipping)."""
    Tk, T64 = np.asarray(T_kernel, np.int64), np.asarray(T64, np.int64)
    rows = Tk.shape[0]
    clear = clear_rows(margin)
    ok = np.ones(rows, bool)
    how = np.full(rows, 2, np.int8)
    ok[clear] = (Tk[clear] == T64[clear]).all(1)
    how[clear] = 0
    lo = np.floor(x).astype(np.int64)
    if gmm:
        got = Tk[:, 1:-1]
        inner = np.concatenate([np.zeros((rows, 1), np.int64), lo, T64[:, -1:]], 1)
        safe = (np.diff(inner, axis=1) >= 3).all(1)
    else:
        got = np.diff(Tk, axis=1)[:, :-1]
        safe = (lo >= 3).all(1) & (lo.sum(1) + lo.shape[1] + 3 <= T64[:, -1])
    alt = lo + np.where(x - lo > 0.5, 1, -1)
    amb = margin < MARGIN
    binok = np.where(amb, (got == lo) | (got == alt), got == lo).all(1) & (Tk[:, 0] == 0) & (Tk[:, -1] == T64[:, -1])
    sel = ~clear & safe
    ok[sel] = binok[sel]
    how[sel] = 1
    return ok, how


def check_table_properties(T, total=65536):
    """T[0] = 0, T[n] = total, strictly increasing (no empty symbol): the tables the fix-up guarantees.  Returns the
    indices of the rows that break a property."""
    T = np.asarray(T, np.int64)
    bad = (T[:, 0] != 0) | (T[:, -1] != total) | (np.diff(T, axis=1) <= 0).any(1)
    return np.nonzero(bad)[0]
