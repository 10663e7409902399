"""GPU parity tests: every op of the hot path, through the C-ABI (via the `lic360` mirror), against
 (1) the CPU oracle, (2) golden outputs of the reference CUDA extension recorded on a B200 (tests/golden/),
 (3) the live reference extension when oracle/_ref/lic360_ref*.so is present."""
import hashlib

import numpy as np
import pytest

from op_cases import CASES
from util import ops_golden, rel_err

pytestmark = pytest.mark.gpu


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _mine(case):
    import lic360
    before = lic360.launch_count()
    out = case.run(lic360, "cuda:0")
    assert lic360.launch_count() > before or case.name.startswith("code_contex"), "no native kernel was launched"
    return out


def _compare(case, got, exp, against_cuda_reference, skip=()):
    keys = [k for k in exp if k in got and k not in skip]
    assert keys, "nothing to compare"
    for k in keys:
        a, b = got[k], exp[k]
        assert a.shape == b.shape, (case.name, k, a.shape, b.shape)
        if k in case.exact or (k in case.libm and against_cuda_reference):
            assert np.array_equal(a, b), "%s/%s: %d of %d entries differ" % (case.name, k, int((a != b).sum()), a.size)
        elif k in case.libm:
            # integers derived through expf/erff: glibc (oracle) vs libdevice (device) may differ by one count
            d = np.abs(a.astype(np.int64) - b.astype(np.int64))
            assert d.max() <= 1 and (d > 0).mean() <= 5e-3, "%s/%s: max diff %d, frac %.4f" % (case.name, k, d.max(), (d > 0).mean())
        else:
            tol = case.close[k] if against_cuda_reference else case.oracle_close.get(k, case.close[k])
            assert rel_err(a, b) <= tol, "%s/%s: rel err %.3g > %.1g" % (case.name, k, rel_err(a, b), tol)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_vs_oracle(case):
    got = _mine(case)
    exp = case.oracle(levels=got[case.levels_from_device]) if case.levels_from_device else case.oracle()
    _compare(case, got, exp, against_cuda_reference=False)
    if case.levels_from_device:  # and the device's exp() levels themselves against libm, float tier
        key = case.levels_from_device
        assert rel_err(got[key], case.oracle()[key]) <= case.close[key]


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_vs_reference_extension(case, ref_ext):
    """Live against the reference extension when it is built.  Without it, this is the same check as test_vs_golden: the
    reference's outputs for the same seeded inputs, recorded on a B200 (tests/golden/ops_golden_*.npz)."""
    if ref_ext is None:
        _compare_with_golden(case)
        return
    got = _mine(case)
    ref = case.run(ref_ext, "cuda:0")
    _compare(case, got, ref, against_cuda_reference=True, skip=case.skip_ref)


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_vs_golden(case):
    _compare_with_golden(case)


def _compare_with_golden(case):
    gold = ops_golden()
    keys = [k[len(case.name) + 1:] for k in gold if k.startswith(case.name + "/")]
    if not keys:
        pytest.skip("no golden entry for this case")
    got = _mine(case)
    exp = {}
    for k in keys:
        if k.endswith("#sha256"):
            base = k[:-7]
            assert _sha(got[base]) == str(gold[case.name + "/" + k]), "%s/%s: sha256 differs from the reference" % (case.name, base)
        elif k.endswith("#sub"):  # strided subsample of a large float-tier array (make_golden.py)
            base, ref = k[:-4], gold[case.name + "/" + k]
            sub = np.ascontiguousarray(got[base]).reshape(-1)[::got[base].size // 8192][:8192]
            assert rel_err(sub, ref) <= case.close[base], "%s/%s: rel err %.3g vs the reference subsample" % (case.name, base, rel_err(sub, ref))
        else:
            exp[k] = gold[case.name + "/" + k]
    if exp:
        _compare(case, got, exp, against_cuda_reference=True, skip=case.skip_ref)
