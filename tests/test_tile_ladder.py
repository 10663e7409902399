"""CPU: the ladder container (pack_ladder_streams / unpack_ladder_streams), its cuts (ladder_to_tiles) and the multi-budget search
(select_shared_offsets) that TileCodec.encode_ladder runs, driven by fake estimates of (latent, offset) pairs."""
import struct

import pytest

import lic360_pipeline as pl
import lic360_shard as sh
from test_budget_select import STAGE1, _est

ROWS, COLS, H, W = 2, 3, 8, 12
T = ROWS * COLS


def _streams(R, seed=0):
    """R rungs of T stream pairs of distinct lengths and contents (some empty)"""
    return [[(bytes([(seed + r * 7 + k) % 251]) * ((r + k) % 4), bytes([(seed + 3 * r + k) % 241]) * (r * 5 + k + 1))
             for k in range(T)] for r in range(R)]


# ---- container -----------------------------------------------------------------------------------------------------------------
def test_ladder_round_trip_and_layout():
    offsets, rungs = [0, 9, 48, 60], _streams(4)
    blob = sh.pack_ladder_streams(ROWS, COLS, H, W, offsets, rungs)
    assert blob[:4] == b"L3L1"
    assert struct.unpack_from("<IIIII", blob, 4) == (ROWS, COLS, H, W, 4)
    assert list(struct.unpack_from("<4I", blob, 24)) == offsets
    head = sh.ladder_header_bytes(4, T)
    assert head == 24 + 4 * 4 + 8 * 4 * T
    lens = struct.unpack_from("<%dI" % (8 * T), blob, 40)
    assert list(lens) == [n for r in rungs for a, b in r for n in (len(a), len(b))]  # rung-major
    assert blob[head:] == b"".join(a + b for r in rungs for a, b in r)
    assert sh.unpack_ladder_streams(blob) == (ROWS, COLS, H, W, offsets, rungs)
    one = sh.pack_ladder_streams(1, 1, 2, 2, [5], [[(b"", b"")]])
    assert sh.unpack_ladder_streams(one) == (1, 1, 2, 2, [5], [[(b"", b"")]])


def test_pack_ladder_streams_rejects_bad_input():
    rungs = _streams(2)
    with pytest.raises(ValueError):
        sh.pack_ladder_streams(3, COLS, H, W, [0, 1], rungs)  # the grid does not divide the latent
    with pytest.raises(ValueError):
        sh.pack_ladder_streams(ROWS, COLS, H, W, [0], rungs)  # offsets and rungs disagree
    with pytest.raises(ValueError):
        sh.pack_ladder_streams(ROWS, COLS, H, W, [], [])  # no rung
    with pytest.raises(ValueError):
        sh.pack_ladder_streams(ROWS, COLS, H, W, [0, -1], rungs)
    with pytest.raises(ValueError):
        sh.pack_ladder_streams(ROWS, COLS, H, W, [0, 1.0], rungs)
    with pytest.raises(ValueError):
        sh.pack_ladder_streams(ROWS, COLS, H, W, [0, 1], [rungs[0], rungs[1][:-1]])  # a rung short of a tile


def test_unpack_ladder_streams_rejects_malformed_containers():
    blob = sh.pack_ladder_streams(ROWS, COLS, H, W, [0, 8, 16], _streams(3))
    head = sh.ladder_header_bytes(3, T)

    def with_field(i, v):
        return blob[:4 + 4 * i] + struct.pack("<I", v) + blob[8 + 4 * i:]

    bad = [
        b"",
        blob[:23],                                 # shorter than the fixed header
        b"L3T1" + blob[4:],                        # another container's magic
        with_field(0, 3),                          # rows do not divide H
        with_field(1, 0),                          # no columns
        with_field(4, 0),                          # no rung
        with_field(4, 1000),                       # more rungs than the header holds
        blob[:head - 1],                           # truncated header
        blob[:-1],                                 # truncated payload
        blob + b"\0",                              # trailing bytes
        blob[:head - 4] + struct.pack("<I", struct.unpack_from("<I", blob, head - 4)[0] + 1) + blob[head:],  # lengths do not add up
    ]
    for i, b in enumerate(bad):
        with pytest.raises(ValueError):
            sh.unpack_ladder_streams(b)
        with pytest.raises(ValueError):
            sh.ladder_to_tiles(b, 0)


def test_ladder_to_tiles_is_pack_tile_streams_of_the_chosen_streams():
    offsets, rungs = [3, 17, 40], _streams(3, seed=5)
    blob = sh.pack_ladder_streams(ROWS, COLS, H, W, offsets, rungs)
    for r in range(3):
        cut = sh.ladder_to_tiles(blob, r)
        assert cut == sh.pack_tile_streams(ROWS, COLS, H, W, rungs[r])
        assert sh.unpack_tile_streams(cut) == (ROWS, COLS, H, W, rungs[r])
    pick = [2, 0, 1, 1, 0, 2]
    cut = sh.ladder_to_tiles(blob, pick)
    assert cut == sh.pack_tile_streams(ROWS, COLS, H, W, [rungs[r][k] for k, r in enumerate(pick)])
    assert sh.ladder_to_tiles(blob, tuple(pick)) == cut
    for bad in (3, -1, [0] * (T - 1), [0] * (T + 1), [0, 0, 0, 0, 0, 3], [0, 0, 0, 0, 0, -1], [0, 0, 0, 0, 0, 1.0], True):
        with pytest.raises(ValueError):
            sh.ladder_to_tiles(blob, bad)


# ---- the multi-budget search ---------------------------------------------------------------------------------------------------
def _fake_pairs(bounds_of):
    """estimate((latent, offset) pairs) whose budget_bound is bounds_of(latent, offset); records every call"""
    calls = []

    def estimate(pairs):
        calls.append(list(pairs))
        return [_est(bounds_of(k, t)) for k, t in pairs]

    return estimate, calls


def _alone(bounds_of, budget, K, top):
    est, _ = _fake_pairs(bounds_of)
    return pl.select_shared_offset(est, budget, K, top)


def _check_search(bounds_of, budgets, K, top, max_batch=None):
    est, calls = _fake_pairs(bounds_of)
    got = pl.select_shared_offsets(est, budgets, K, top, max_batch)
    assert len(got) == len(budgets)
    for r, b in enumerate(budgets):
        assert got[r] == _alone(bounds_of, b, K, top), r
    pairs = sum(calls, [])
    assert len(pairs) == len(set(pairs)), "a pair estimated twice"
    if max_batch is not None:
        assert all(len(c) <= max_batch for c in calls)
    want = set((k, t) for _, own, _ in got for t in own for k in range(K))
    assert set(pairs) == want, "only the offsets some budget evaluates"
    return got, calls


def test_each_budget_equals_the_single_search():
    tables = [lambda t: 1000 - 10 * t, lambda t: 500 - 3 * t, lambda t: 800 - 7 * t]

    def bounds_of(k, t):
        return tables[k](min(t, 48))

    total = [sum(tables[k](t) for k in range(3)) for t in range(49)]
    budgets = [total[0], total[3], total[17] + 1, total[31], total[48], total[8], total[25]]
    got, calls = _check_search(bounds_of, budgets, 3, 48)
    assert [o for o, _, _ in got] == [0, 3, 17, 31, 48, 8, 25]
    # stage 1 once for every budget, then one call with the union of the stage-2 offsets
    assert calls[0] == [(k, t) for t in STAGE1 for k in range(3)]
    assert calls[1] == [(k, t) for t in sorted(set(range(1, 8)) | set(range(17, 24)) | set(range(25, 32)) | set(range(41, 48)))
                        for k in range(3)]
    assert len(calls) == 2
    # two budgets that share a stage 2 share its estimates
    got, calls = _check_search(bounds_of, [total[3], total[5]], 3, 48)
    assert [o for o, _, _ in got] == [3, 5] and len(calls[1]) == 3 * 7


def test_non_monotone_rate_takes_each_budgets_own_offsets():
    """Budget A alone stops at 16 (stage 2: 9..15); budget B alone stops at 8 and evaluates 1..7, where offset 5 dips below A's
    budget.  The smallest fit over the union of evaluated offsets would give A offset 5; its own search gives 16."""
    def bound(t):
        if t == 5:
            return 250
        return {0: 1000, 8: 600}.get(t, 700 if t < 8 else 400 if t < 16 else 300)

    budget_a, budget_b = 350, 650
    got, _ = _check_search(lambda k, t: bound(t), [budget_a, budget_b], 1, 48)
    assert got[0][0] == 16 and got[1][0] == 5
    union = {t: b for _, own, _ in got for t, b in own.items()}
    assert min(t for t, b in union.items() if b <= budget_a) == 5 != got[0][0]
    assert 5 not in got[0][1]


@pytest.mark.parametrize("max_batch", [1, 4, 7, 16, 1000])
def test_passes_of_at_most_max_batch_pairs(max_batch):
    def bounds_of(k, t):
        return (900 - 11 * t + 13 * k) if t != 20 else 100  # a dip at 20

    budgets = [2600, 2000, 1500, 1000]
    got, calls = _check_search(bounds_of, budgets, 3, 56, max_batch)
    est, full = _fake_pairs(bounds_of)
    assert pl.select_shared_offsets(est, budgets, 3, 56) == got
    assert sum(calls, []) == sum(full, []), "the same pairs in the same order"


def test_max_offset_off_the_grid():
    got, calls = _check_search(lambda k, t: 2000 - 20 * t, [2000 - 20 * 50, 2000 - 20 * 52], 1, 53)
    assert [o for o, _, _ in got] == [50, 52]
    assert calls[0] == [(0, t) for t in STAGE1 + [53]]
    assert calls[1] == [(0, t) for t in range(49, 53)]


def test_the_lowest_budget_no_offset_fits_is_reported():
    est, calls = _fake_pairs(lambda k, t: 1000 - 10 * t)
    with pytest.raises(RuntimeError) as e:
        pl.select_shared_offsets(est, [900, 400, 600, 300], 1, 48)
    with pytest.raises(RuntimeError) as alone:
        pl.select_shared_offset(_fake_pairs(lambda k, t: 1000 - 10 * t)[0], 400, 1, 48)
    assert str(e.value) == str(alone.value) + " (rung 1)"
    assert len(calls) == 1, "no stage 2 once a budget fails"
