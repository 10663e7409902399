"""CPU: the offset search of FusedCodec.encode_to_budget with a protection map (select_budget_offset with max_offset = 48 + max P),
driven by the fake estimates of test_budget_select.py, and the latitude preset (lic360_pipeline.latitude_protection)."""
import math

import numpy as np
import pytest
import torch

import lic360_pipeline as pl
from test_budget_select import STAGE1, _fake


def _linear(k):
    return 1000 - 10 * k


def test_max_offset_off_the_grid_evaluates_it_and_a_short_stage_two():
    est, calls = _fake(_linear)
    k, bounds = pl.select_budget_offset(est, _linear(51), max_offset=53)
    assert calls == [STAGE1 + [53], [49, 50, 51, 52]]
    assert k == 51 and sorted(bounds) == sorted(STAGE1 + [53, 49, 50, 51, 52])
    # the fit at max_offset itself: stage 2 between 48 and 53 finds nothing
    est, calls = _fake(_linear)
    k, _ = pl.select_budget_offset(est, _linear(53), max_offset=53)
    assert k == 53 and calls == [STAGE1 + [53], [49, 50, 51, 52]]
    # a stage-1 point one above the previous one leaves no offset for stage 2
    est, calls = _fake(_linear)
    k, _ = pl.select_budget_offset(est, _linear(49), max_offset=49)
    assert k == 49 and calls == [STAGE1 + [49]]


def test_max_offset_on_the_grid():
    est, calls = _fake(_linear)
    k, _ = pl.select_budget_offset(est, _linear(56), max_offset=56)
    assert k == 56 and calls == [STAGE1 + [56], list(range(49, 56))]
    est, calls = _fake(_linear)
    k, _ = pl.select_budget_offset(est, _linear(70) + 5, max_offset=96)
    assert calls == [list(range(0, 97, 8)), list(range(65, 72))]
    assert k == 70
    est, calls = _fake(_linear)
    k, _ = pl.select_budget_offset(est, _linear(96), max_offset=96)
    assert k == 96 and calls == [list(range(0, 97, 8)), list(range(89, 96))]


def test_default_max_offset_is_the_uniform_search():
    for budget in (1000, 700, 699, 521, 520):
        a, calls_a = _fake(_linear)
        b, calls_b = _fake(_linear)
        assert pl.select_budget_offset(a, budget) == pl.select_budget_offset(b, budget, max_offset=48)
        assert calls_a == calls_b


@pytest.mark.parametrize("max_offset", [53, 56, 96])
def test_no_offset_fits_names_max_offset(max_offset):
    est, calls = _fake(_linear)
    with pytest.raises(RuntimeError, match=r"no level offset up to %d fits %d bytes \(bound at offset %d: %d bytes\)"
                       % (max_offset, _linear(max_offset) - 1, max_offset, _linear(max_offset))):
        pl.select_budget_offset(est, _linear(max_offset) - 1, max_offset=max_offset)
    assert len(calls) == 1 and calls[0][-1] == max_offset


@pytest.mark.parametrize("h,w,levels", [(32, 64, 16), (7, 10, 48), (64, 128, 5), (1, 3, 48)])
def test_latitude_protection_is_the_formula(h, w, levels):
    p = pl.latitude_protection(h, w, levels)
    assert p.shape == (1, 1, h, w) and p.dtype == torch.int32 and p.device == torch.device("cpu")
    phi = math.pi / 2 - math.pi * (np.arange(h) + 0.5) / h
    want = np.round(levels * np.cos(phi)).astype(np.int32)
    got = p.numpy()[0, 0]
    assert np.array_equal(got, np.repeat(want[:, None], w, axis=1))
    assert np.array_equal(got, got[::-1]), "north / south symmetry"
    eq = [h // 2] if h % 2 else [h // 2 - 1, h // 2]
    assert all(got[i, 0] == got.max() for i in eq), "the maximum is on the equator rows"
    assert got.min() >= 0 and got.max() <= levels


def test_latitude_protection_rows_and_errors():
    p = pl.latitude_protection(16, 32, 48)[0, 0]
    assert p[0, 0] < p[4, 0] < p[7, 0] and p[7, 0] == 48 and p[0, 0] == round(48 * math.cos(math.pi / 2 - math.pi / 32))
    for bad in (49, -1, 2.5):
        with pytest.raises(RuntimeError, match="integer in"):
            pl.latitude_protection(16, 32, bad)
    assert torch.equal(pl.latitude_protection(8, 8, 0), torch.zeros((1, 1, 8, 8), dtype=torch.int32))
