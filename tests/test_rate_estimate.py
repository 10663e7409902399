"""CPU: the reference of the codec's rate estimate (lic360_codec_estimate, FusedCodec.estimate) and the bound between a stream's
ideal code length and the bytes the host coder (csrc/coder.cpp) writes for it.  tests/test_gpu_rate_estimate.py checks the GPU
estimate against both.

The bound.  Every table has total 2^16.  The coder keeps low, high (32 bits) and R = high - low + 1; symbol i with bins
T[s] < T[s+1], p_i = (T[s+1] - T[s]) / 2^16, sets
    R' = floor(T[s+1] R / 2^16) - floor(T[s] R / 2^16),   so   R p_i - 1 < R' < R p_i + 1,
then renormalises: each shift -- a matching top bit that is written, or an underflow bit that is only counted as pending --
doubles R exactly, and afterwards R > 2^30 (low < 2^30 or high >= 3 * 2^30 once low < 2^31 <= high).  Hence R p_i > 2^14 and
    R' = R p_i 2^e_i   with   |e_i| < log2(1 + 2^-14) < 2^-13 bits.
Starting from R = 2^32 and taking log2 over the N coded symbols, the number of shifts is
    S = I + (log2 R_N - 32) - sum(e_i),   I = sum(-log2 p_i),   log2 R_N in (30, 32],
so I - 2 - N 2^-13 < S < I + N 2^-13.  The stream holds the S - u shifted-out bits, where u is the count of underflow bits still
pending at the end: the coder never writes them, because the terminator alone -- one `1` bit (lic360_coder_finish_mem) and zero
padding to a byte, the decoder reading zeros past the end -- already names a point inside the final interval.  So
    8 len in [S - u + 1, S - u + 8]   and   -(1 + u + N 2^-13) < 8 len - I <= 8 + N 2^-13
(equality only for N = 0: an empty stream is the terminator byte).
u is the one term the tables do not fix (a stream whose final interval straddles a dyadic point at k successive scales ends
with k pending bits); it is a few bits in practice and the tests allow PENDING_ALLOWANCE.  The floor divisions cost at most
2^-13 bits per symbol in either direction; the final range at most 2 bits; terminator and padding 1 to 8 bits.
"""
import math

import numpy as np
import pytest

import probe_nets as pn
from util import random_tables, rng, synthetic_latent

PENDING_ALLOWANCE = 16


def bits_from_tables(T, labels, mask=None):
    """Ideal code length 16 - log2(T[s+1] - T[s]) in float64 of every symbol, T (N, n+1) integer CDF rows of total 65536 in
    coding order, labels (N,); 0 where mask < 0.5 (the encoder skips those positions, as coder.cpp does)."""
    T = np.asarray(T, np.int64)
    lab = np.asarray(labels, np.int64)
    out = np.zeros(len(lab))
    keep = np.ones(len(lab), bool) if mask is None else ~(np.asarray(mask, np.float32) < 0.5)
    r = np.nonzero(keep)[0]
    width = T[r, lab[r] + 1] - T[r, lab[r]]
    assert (width > 0).all(), "a coded symbol has an empty bin"
    out[r] = 16.0 - np.log2(width.astype(np.float64))
    return out


def stream_bound(n_coded):
    """(lower, upper) of 8 * len(stream) - I for a stream of n_coded symbols (module docstring)"""
    return -(1 + PENDING_ALLOWANCE + n_coded * 2.0 ** -13), 8 + n_coded * 2.0 ** -13


def assert_within_bound(nbytes, ideal_bits, n_coded, what=""):
    lo, hi = stream_bound(n_coded)
    d = 8 * nbytes - ideal_bits
    assert lo <= d <= hi, "%s: 8 * %d bytes - %.3f ideal bits = %.3f, outside (%.3f, %.3f)" % (what, nbytes, ideal_bits, d, lo, hi)


def test_bits_from_tables_by_hand():
    T = np.array([[0, 8192, 16384, 32768, 65536], [0, 1, 2, 3, 65536], [0, 16384, 32768, 49152, 65536]])
    got = bits_from_tables(T, [3, 0, 2], [1.0, 0.5, 0.49])
    assert np.array_equal(got, [1.0, 16.0, 0.0])
    assert np.array_equal(bits_from_tables(T, [2, 3, 1]), [2.0, 16.0 - math.log2(65533), 2.0])
    # a NaN mask is coded, as by the coder (mask < 0.5 is false)
    assert bits_from_tables(T[:1], [0], [np.nan])[0] == 3.0


@pytest.mark.parametrize("H,W", [(2, 2), (8, 16), (6, 130)])
@pytest.mark.parametrize("name", pn.PROBES)
def test_probe_streams_within_bound(name, H, W):
    """the exact tables of every probe network: both streams the host coder writes are within the bound of their ideal length"""
    q, mask, lv = synthetic_latent(300 + H + W, H=H, W=W)
    Tc, lab_c, msk, Ti, lab_i = pn.expected_tables(pn.probe_params(name), q, mask, lv)
    bi, bc = pn.host_encode(Ti, lab_i, None), pn.host_encode(Tc, lab_c, msk)
    assert_within_bound(len(bi), math.fsum(bits_from_tables(Ti, lab_i)), len(lab_i), "importance stream")
    assert_within_bound(len(bc), math.fsum(bits_from_tables(Tc, lab_c, msk)), int((msk >= 0.5).sum()), "code stream")


def test_random_tables_within_bound():
    """long streams of skewed random tables: the bound holds with a few bits to spare on each side of a large I"""
    r = rng(7)
    for ncode, rows in ((8, 60000), (49, 20000)):
        T = random_tables(r, rows, ncode)
        lab = r.integers(0, ncode, rows)
        mask = (r.random(rows) < 0.7).astype(np.float32)
        ideal = math.fsum(bits_from_tables(T, lab, mask))
        assert ideal > 1e4
        assert_within_bound(len(pn.host_encode(T, lab, mask)), ideal, int(mask.sum()), "ncode %d" % ncode)


def test_all_masked_code_stream_is_one_byte():
    """nothing coded: I = 0 and the stream is the terminator byte alone (8 len - I = 8, the top of the bound)"""
    r = rng(8)
    T = random_tables(r, 500, 8)
    lab = r.integers(0, 8, 500)
    mask = np.zeros(500, np.float32)
    assert bits_from_tables(T, lab, mask).sum() == 0
    b = pn.host_encode(T, lab, mask)
    assert b == b"\x80"
    assert_within_bound(len(b), 0.0, 0)
