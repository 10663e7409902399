"""CPU: the float64 table reference (ref64.py) against the reference extension's recorded tables, and the adversarial
table inputs the GPU table tests use."""
import numpy as np
import pytest

import op_cases as oc
import ref64
from util import ops_golden, rng


def _comparable(T, mg, x, gmm):
    return ref64.compare(T, T, mg, x, gmm)[1] != 2


def adversarial_gmm():
    """(w, d, m) rows at the edges of the GMM table formula: negative deltas (clamped to 1e-6), delta 0 (-> exactly 1e-6)
    with means on a bin edge and half a bin away, means at +-40 (all mass in an end bin: interior bins of 65535/65536,
    the fix-up), mixture logits of +-80, tied maxima and all equal.  Only the combinations that ref64.compare() can
    check are kept (13 of 160 have an ambiguous bin next to the fix-up)."""
    rows = []
    for lg in ([0, 0, 0], [80, -80, -80], [-80, 80, 80], [3, 3, -2], [1.5, -0.5, 0.25]):
        for dl in ([-1, -0.5, -2], [0, 0, 0], [0.5, 1, 2], [-1, 0, 0.75]):
            for mn in ([0.5, 0.5, 0.5], [1, -2, 3], [-40, -40, -40], [40, 40, 40], [-40, 0.5, 40], [-3.5, 3.5, 0],
                       [2.5, -1.5, 0.5], [0, 0, 0]):
                rows.append((lg, dl, mn))
    a = np.array(rows, np.float32)
    a = a[_comparable(*ref64.gmm_table64(a[:, 0], a[:, 1], a[:, 2]), True)]
    return a[:, 0], a[:, 1], a[:, 2]


def adversarial_logits(w=49):
    """softmax rows at the edges: one-hot +60 with the rest at -60 (expf underflows: zero-width bins and the fix-up),
    two tied maxima, all equal, a one-hot at each end, and rows where the clipping at total acts."""
    out = []
    for k in (0, 1, w // 2, w - 2, w - 1):
        x = np.full(w, -60.0)
        x[k] = 60
        out.append(x)
    for k0, k1 in ((0, 1), (3, w - 1), (w - 2, w - 1)):
        x = np.full(w, -60.0)
        x[[k0, k1]] = 60
        out.append(x)
    out.append(np.zeros(w))
    out.append(np.full(w, 7.0))
    out.append(np.linspace(-20, 0, w))
    out.append(np.linspace(0, -20, w))
    x = np.zeros(w)
    x[: w // 2] = 12
    out.append(x)
    out = np.array(out, np.float32)
    return out[_comparable(*ref64.entropy_table64(out), False)]


def _gmm_golden_cases():
    out = []
    for name, seed, hw, rows in (("small", 301, (8, 16), 100), ("full", 302, (16, 32), 512), ("one", 303, (4, 4), 1)):
        w, d, m = oc._gmm_inputs(seed, hw[0] * hw[1])
        out.append(("gmm_table_" + name, w[:rows], d[:rows], m[:rows]))
    for name, seed, rows in (("b1", 311, 90), ("b2", 312, 128)):
        out.append(("gmm_table_batch_" + name,) + oc._gmm_inputs(seed, rows))
    return out


def _entropy_golden_cases():
    out = []
    for name, hw, rows, nstep, seed in (("imp49", (8, 16), 32, 49, 321), ("small5", (4, 8), 32, 5, 322), ("max64", (4, 4), 16, 64, 323)):
        x = (rng(seed).standard_normal((hw[0] * hw[1], nstep)) * 3).astype(np.float32)   # op_cases._mk_entropy_table
        x[::7] *= 6
        out.append(("entropy_table_" + name, x[:rows]))
    return out


def test_gmm_table64_equals_reference_tables():
    """On the reference's recorded GMM tables, the float64 table equals the reference's on every row outside the margin,
    and the rounded bins agree wherever compare() can read them off."""
    g = ops_golden()
    total = clear = 0
    for key, w, d, m in _gmm_golden_cases():
        gold = g[key + "/table"]
        T, mg, x = ref64.gmm_table64(w, d, m)
        ok, how = ref64.compare(gold, T, mg, x, True)
        assert ok.all(), (key, np.nonzero(~ok)[0][:5])
        assert len(ref64.check_table_properties(gold)) == 0, key
        total += len(gold)
        clear += (how == 0).sum()
        assert (how == 2).sum() <= 0.25 * len(gold), key
    # 7 bins, each inside the margin with probability 0.2 at random inputs: about a fifth of the 831 rows are clear
    assert total == 831 and clear >= 0.15 * total, (total, clear)


def test_entropy_table64_equals_reference_tables():
    g = ops_golden()
    clear = 0
    for key, x in _entropy_golden_cases():
        gold = g[key + "/table"]
        T, mg, val = ref64.entropy_table64(x)
        ok, how = ref64.compare(gold, T, mg, val, False)
        assert ok.all(), (key, np.nonzero(~ok)[0][:5])
        assert len(ref64.check_table_properties(gold)) == 0, key
        clear += (how == 0).sum()
    assert clear >= 15


def test_adversarial_rows_are_clear_and_valid():
    """the adversarial sets reach the table edges they are meant for, and their tables are valid"""
    w, d, m = adversarial_gmm()
    T, mg, _ = ref64.gmm_table64(w, d, m)
    assert len(w) == 147 and ref64.clear_rows(mg).sum() == 128
    assert len(ref64.check_table_properties(T)) == 0
    assert (T[:, 7] == 65535).sum() >= 20 and (T[:, 1] == 65529).sum() >= 10   # overflow-bit bins, all mass in bin 0
    assert (T[:, 1:8] == np.arange(1, 8)).all(1).sum() >= 10                  # all mass in bin 7
    lg = adversarial_logits()
    T, mg, _ = ref64.entropy_table64(lg)
    assert len(lg) == 11 and ref64.clear_rows(mg).sum() == 9
    assert len(ref64.check_table_properties(T)) == 0
    assert (T[:, 1:-1] >= 65535).any() and (T[:, 1:-1] == 32768).any()


@pytest.mark.parametrize("gmm", [True, False])
def test_fixup_matches_oracle_and_never_leaves_an_empty_bin(gmm):
    """fixup64 restates the oracle's fix-up (both rules) on arbitrary non-decreasing integer rows, including runs of equal
    bins at 0 and at total; the fixed rows are always strictly increasing."""
    from oracle import oracle as O
    r = rng(7 + gmm)
    n = 8 if gmm else 49
    raw = np.sort(r.choice([0, 1, 2, 65534, 65535, 65536, 30000, 30001], (4000, n - 1)), 1)
    raw = np.concatenate([np.zeros((4000, 1), np.int64), raw, np.full((4000, 1), 65536)], 1)
    mine = ref64.fixup64(raw.copy(), gmm)
    assert len(ref64.check_table_properties(mine)) == 0
    if gmm:
        # the oracle's gmm_table with delta -> 1e-6 and one component puts each bin at 0 or 65536 exactly: compare on those
        m = np.where(r.random((500, 1)) < 0.5, -40, 40).astype(np.float32) * np.ones((1, 3), np.float32)
        tab = O.gmm_table(np.zeros((500, 3), np.float32), np.full((500, 3), -1, np.float32), m)[0]
        T, _, _ = ref64.gmm_table64(np.zeros((500, 3)), np.full((500, 3), -1), m)
        assert np.array_equal(tab.astype(np.int64), T)
    else:
        lg = adversarial_logits()
        assert np.array_equal(O.entropy_table(lg).astype(np.int64), ref64.entropy_table64(lg)[0])
