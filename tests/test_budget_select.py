"""CPU: the byte bound and the two-stage offset search of FusedCodec.encode_to_budget (lic360_pipeline.select_budget_offset), driven by
fake estimates whose bounds are set per offset."""
import pytest

import lic360_pipeline as pl


def _est(bound):
    """an estimate whose budget_bound is exactly `bound` bytes: the importance stream takes 1 byte, the code stream bound - 1"""
    return {"imp_bits": 0.0, "imp_symbols": 0, "code_bits": 8.0 * bound - 16.0, "code_symbols": 0}


def _fake(bounds_of):
    calls = []

    def estimate(offsets):
        calls.append(list(offsets))
        return [_est(bounds_of(k)) for k in offsets]

    return estimate, calls


STAGE1 = [0, 8, 16, 24, 32, 40, 48]


def test_stream_bytes_bound():
    assert pl.stream_bytes_bound(0.0, 0) == 1  # the terminator byte
    assert pl.stream_bytes_bound(8.0 * 100 - 8, 0) == 100
    assert pl.stream_bytes_bound(8.0 * 100 - 7, 0) == 100
    assert pl.stream_bytes_bound(8.0 * 100 - 9, 0) == 99
    # N/8192 bits of slack per stream
    assert pl.stream_bytes_bound(8.0 * 100 - 8 - 1.0, 8192) == 100
    assert pl.stream_bytes_bound(8.0 * 100 - 8 - 1.0, 8191) == 99
    # a double total a rounding below an integer boundary counts as on it
    assert pl.stream_bytes_bound(8.0 * 100 - 8 - 1e-9, 0) == 100
    assert pl.budget_bound({"imp_bits": 792.0, "imp_symbols": 0, "code_bits": 8.0 * 7 - 8, "code_symbols": 0}) == 107


def test_monotone_rate_and_a_tie_at_the_boundary():
    est, calls = _fake(lambda k: 1000 - 10 * k)
    k, bounds = pl.select_budget_offset(est, 700)
    assert calls == [STAGE1, [25, 26, 27, 28, 29, 30, 31]]
    assert k == 30 and bounds[30] == 700  # a bound equal to the budget fits
    assert sorted(bounds) == sorted(STAGE1 + calls[1])
    assert bounds == {o: 1000 - 10 * o for o in bounds}
    k, _ = pl.select_budget_offset(_fake(lambda k: 1000 - 10 * k)[0], 699)
    assert k == 31


def test_fit_at_offset_zero_stops_after_one_call():
    est, calls = _fake(lambda k: 500 - k)
    k, bounds = pl.select_budget_offset(est, 500)
    assert k == 0 and calls == [STAGE1] and sorted(bounds) == STAGE1


def test_non_monotone_rate():
    table = {0: 1000, 8: 900, 16: 800, 24: 2000, 32: 100, 40: 5000, 48: 50}
    table.update({o: 850 for o in range(9, 16)})
    table[9] = 790
    est, calls = _fake(lambda k: table.get(k, 10 ** 6))
    k, bounds = pl.select_budget_offset(est, 800)
    assert calls == [STAGE1, list(range(9, 16))]
    assert k == 9  # below k1 = 16, although 10..15 do not fit
    # stage 2 finds nothing: k1 itself
    table.update({o: 801 for o in range(9, 16)})
    k, _ = pl.select_budget_offset(_fake(lambda k: table.get(k, 10 ** 6))[0], 800)
    assert k == 16
    # a later stage-1 offset that fits does not replace the smallest one
    k, _ = pl.select_budget_offset(_fake(lambda k: table.get(k, 10 ** 6))[0], 100)
    assert k == 32


def test_no_offset_fits():
    est, calls = _fake(lambda k: 1000 - k)
    with pytest.raises(RuntimeError, match="no level offset"):
        pl.select_budget_offset(est, 951)
    assert calls == [STAGE1]
    k, _ = pl.select_budget_offset(_fake(lambda k: 1000 - k)[0], 952)
    assert k == 48
