"""CPU: the searches of FusedCodec.encode_batch_to_budget, per latent (select_budget_offsets) and with one shared offset
(select_shared_offset), driven by fake estimates of (latent, offset) pairs like those of test_budget_select.py."""
import pytest

import lic360_pipeline as pl
from test_budget_select import STAGE1, _est


def _fake_pairs(bounds_of):
    """estimate((latent, offset) pairs) whose budget_bound is bounds_of(latent, offset); records every call"""
    calls = []

    def estimate(pairs):
        calls.append(list(pairs))
        return [_est(bounds_of(k, t)) for k, t in pairs]

    return estimate, calls


def _split_est(imp_bytes, code_bytes):
    """an estimate whose importance stream is bounded by imp_bytes and its code stream by code_bytes, each 0.5 byte below the
    next integer: a bound of the summed bits would be one byte larger than the sum of the per-stream bounds"""
    return {"imp_bits": 8.0 * imp_bytes - 8 + 4, "imp_symbols": 0, "code_bits": 8.0 * code_bytes - 8 + 4, "code_symbols": 0}


def test_per_latent_search_is_the_single_search_of_each_latent():
    tables = [lambda t: 1000 - 10 * t, lambda t: 500 - t, lambda t: 2000 - 30 * t]
    budgets, tops = [700, 500, 1000], [48, 48, 56]
    est, calls = _fake_pairs(lambda k, t: tables[k](t))
    got = pl.select_budget_offsets(est, budgets, tops)
    for k in range(3):
        single, single_calls = _fake_pairs(lambda _, t, k=k: tables[k](t))
        want = pl.select_budget_offset(lambda offs: single([(0, t) for t in offs]), budgets[k], tops[k])
        assert got[k] == want, k
    assert [o for o, _ in got] == [30, 0, 34]
    # one call per stage: stage 1 of all three latents, then stage 2 of the two that need it
    assert calls[0] == [(0, t) for t in STAGE1] + [(1, t) for t in STAGE1] + [(2, t) for t in STAGE1 + [56]]
    assert calls[1] == [(0, t) for t in range(25, 32)] + [(2, t) for t in range(33, 40)]
    assert len(calls) == 2


def test_per_latent_search_with_different_max_offsets():
    est, calls = _fake_pairs(lambda k, t: 1000 - 10 * t)
    got = pl.select_budget_offsets(est, [1000 - 10 * 51, 1000 - 10 * 70 + 5], [53, 96])
    assert [o for o, _ in got] == [51, 70]
    assert max(got[0][1]) == 53 and max(got[1][1]) == 96
    assert calls[1] == [(0, t) for t in range(49, 53)] + [(1, t) for t in range(65, 72)]


def test_max_batch_chunking_leaves_the_evaluated_offsets_unchanged():
    tables = [lambda t: 1000 - 10 * t, lambda t: 800 - 5 * t, lambda t: 600 - t]
    budgets, tops = [650, 700, 590], [48, 60, 48]
    est, calls = _fake_pairs(lambda k, t: tables[k](t))
    want = pl.select_budget_offsets(est, budgets, tops)
    for max_batch in (1, 3, 7, 16, 1000):
        est_b, calls_b = _fake_pairs(lambda k, t: tables[k](t))
        assert pl.select_budget_offsets(est_b, budgets, tops, max_batch=max_batch) == want, max_batch
        assert all(len(c) <= max_batch for c in calls_b)
        assert sum(calls_b, []) == sum(calls, []), "the same pairs in the same order"
    for max_batch in (1, 5, 16):
        est_a, calls_a = _fake_pairs(lambda k, t: tables[k](t))
        est_b, calls_b = _fake_pairs(lambda k, t: tables[k](t))
        assert pl.select_shared_offset(est_a, 1500, 3, 60) == pl.select_shared_offset(est_b, 1500, 3, 60, max_batch=max_batch)
        assert sum(calls_a, []) == sum(calls_b, []) and all(len(c) <= max_batch for c in calls_b)


def test_per_latent_no_fit_names_the_lowest_latent():
    est, calls = _fake_pairs(lambda k, t: 1000 - t)
    with pytest.raises(RuntimeError, match=r"^encode_to_budget: no level offset up to 48 fits 900 bytes \(bound at offset 48: 952 "
                                           r"bytes\) \(latent 2\)$"):
        pl.select_budget_offsets(est, [10 ** 6, 952, 900, 800], [48] * 4)
    assert len(calls) == 1, "no stage 2 after a latent that fits nothing"


def test_shared_bound_sums_the_per_stream_floors():
    # each latent: importance stream bound 10 bytes, code stream bound 100 - t bytes, both with half a byte of slack
    calls = []

    def estimate(pairs):
        calls.append(list(pairs))
        return [_split_est(10, 100 - t + k) for k, t in pairs]

    per_latent = lambda k, t: 10 + 100 - t + k  # noqa: E731
    assert pl.budget_bound(_split_est(10, 100)) == 110
    e = _split_est(10, 100)
    assert pl.stream_bytes_bound(e["imp_bits"] + e["code_bits"] + 8, 0) == 111, "one bound of both streams' bits, terminators included"
    offset, bounds, per = pl.select_shared_offset(estimate, per_latent(0, 20) + per_latent(1, 20), 2, 48)
    assert offset == 20
    assert bounds == {t: per_latent(0, t) + per_latent(1, t) for t in bounds}
    assert per == {t: [per_latent(0, t), per_latent(1, t)] for t in bounds}
    assert calls[0] == [(k, t) for t in STAGE1 for k in range(2)]
    assert calls[1] == [(k, t) for t in range(17, 24) for k in range(2)]


def test_shared_tie_at_the_boundary_and_between_two_bounds():
    tables = [lambda t: 1000 - 10 * t, lambda t: 500 - 4 * t]
    est = lambda: _fake_pairs(lambda k, t: tables[k](t))  # noqa: E731
    total = lambda t: tables[0](t) + tables[1](t)  # noqa: E731
    offset, bounds, _ = pl.select_shared_offset(est()[0], total(30), 2, 48)
    assert offset == 30 and bounds[30] == total(30), "a summed bound equal to the budget fits"
    offset, _, _ = pl.select_shared_offset(est()[0], total(30) - 1, 2, 48)
    assert offset == 31, "a budget between two summed bounds takes the larger offset"


def test_shared_non_monotone_rate():
    table = {0: 1000, 8: 900, 16: 380, 24: 2000, 32: 100, 40: 5000, 48: 50}
    table.update({t: 425 for t in range(9, 16)})
    table[11] = 390
    est, calls = _fake_pairs(lambda k, t: table.get(t, 10 ** 6) // 2 + k)
    offset, bounds, _ = pl.select_shared_offset(est, 400, 2, 48)
    assert offset == 11 and bounds[11] == 195 + 196
    assert [t for _, t in calls[1]][::2] == list(range(9, 16))


def test_shared_max_offset_and_no_fit():
    est, calls = _fake_pairs(lambda k, t: 1000 - 10 * t)
    offset, bounds, _ = pl.select_shared_offset(est, 2 * (1000 - 10 * 51), 2, 53)
    assert offset == 51 and max(bounds) == 53
    est, calls = _fake_pairs(lambda k, t: 1000 - t)
    with pytest.raises(RuntimeError, match=r"no level offset up to 60 fits 1879 bytes \(bound at offset 60: 1880 bytes\)$"):
        pl.select_shared_offset(est, 1879, 2, 60)
    assert len(calls) == 1


def test_select_budget_offset_with_a_bound_callable():
    calls = []

    def estimate(offsets):
        calls.append(list(offsets))
        return [1000 - 10 * t for t in offsets]

    k, bounds = pl.select_budget_offset(estimate, 700, bound=lambda b: b)
    assert k == 30 and calls == [STAGE1, list(range(25, 32))] and bounds[30] == 700
