"""CPU: the probe networks' closed form (probe_nets.py) against the oracle's context conv, and the expected streams
against the oracle's whole CPU codec."""
import numpy as np
import pytest

import probe_nets as pn
from oracle.cpu_codec import CpuCodec
from util import synthetic_latent


@pytest.mark.parametrize("name", pn.PROBES)
@pytest.mark.parametrize("H,W", [(2, 2), (8, 16), (10, 14)])
def test_closed_form_equals_oracle_conv(name, H, W):
    """closed form (mask rule stated in numpy, forbidden taps skipped) == oracle.cconv_ec through CpuCodec._net_ec
    (lic360_oracle.c:70), bit for bit, for both networks; and the probe really carries signal to the tables"""
    params = pn.probe_params(name)
    q, mask, lv = synthetic_latent(11, H=H, W=W)
    y_code, y_imp = pn.closed_form(params, q, mask, lv)
    cpu = CpuCodec(params)
    x = pn.code_input(q, mask)
    assert np.array_equal(cpu._net_ec(params['code'], x, 48, 3), y_code)
    from oracle import oracle as O
    ref_imp = cpu._net_ec(params['imp'], O.scale(lv, -1.0, 2.0 / 47), 1, 1)[0]
    assert np.array_equal(ref_imp, y_imp)
    assert np.array_equal(pn.imp_input(lv), O.scale(lv, -1.0, 2.0 / 47)[0])   # (1, H/2, W/2)
    if H * W > 4:   # the weight logits and the means depend on the decoded neighbours
        assert len(np.unique(y_code[2])) > 4 and len(np.unique(y_imp[10 if name != "E" else 24])) > 1


def test_forbidden_taps_would_change_the_output():
    """the forbidden taps sit where the input is nonzero: the same weight on an allowed tap changes the network output, so
    a packer that keeps a forbidden tap writes different bytes"""
    params = pn.probe_params("R")
    q, mask, lv = synthetic_latent(12, H=8, W=16)
    want = pn.closed_form(params, q, mask, lv)[0]
    loose = dict(params['code'])
    # move the forbidden weights onto allowed taps of the same layer: the first layer's own-group centre -> left tap
    loose['net.0.weight'] = loose['net.0.weight'].copy()
    loose['net.0.weight'][:, 0::4, :, 2, 1] += loose['net.0.weight'][:, 0::4, :, 2, 2]
    got = pn.net_forward(loose, pn.code_input(q, mask), 48, 3)
    assert not np.array_equal(got, want)


@pytest.mark.parametrize("name", pn.PROBES)
def test_expected_streams_equal_cpu_codec(name):
    """the expected streams (closed form -> float64 tables -> coding order -> product host coder) equal what the oracle's
    CPU codec writes (oracle conv, glibc tables, oracle coder), and the CPU codec decodes them"""
    params = pn.probe_params(name)
    H, W = 8, 16
    q, mask, lv = synthetic_latent(13, H=H, W=W)
    bi, bc = pn.expected_streams(params, q, mask, lv)
    cpu = CpuCodec(params)
    assert cpu.encode_imp(lv) == bi
    assert cpu.encode_code(q, mask) == bc
    assert np.array_equal(cpu.decode_imp(bi, H // 2, W // 2), lv)
    code, m = cpu.decode(bi, bc, H // 2, W // 2)
    assert np.array_equal(m, mask) and np.array_equal(code, q * mask)


def test_probe_tables_reach_the_edges():
    """the extreme-table probe codes symbols through the fix-up, the overflow bins and one-hot / tied softmax rows"""
    q, mask, lv = synthetic_latent(14, H=24, W=72)
    Tc, lab, msk, Ti, li = pn.expected_tables(pn.probe_params("E"), q, mask, lv)
    cod = msk > 0.5
    assert (Tc[cod, 7] == 65535).sum() > 1000            # overflow bit of the top interior bin
    assert (Tc[cod, 1] >= 65529).sum() > 1000            # all mass in bin 0 (means at -40)
    assert (Tc[cod, 1:8] == np.arange(1, 8)).all(1).sum() > 1000   # all mass in bin 7 (means at +40)
    assert (Tc[cod, 4] == 32768).sum() > 100             # a mean on a bin edge, delta 1e-6
    steps = np.diff(Ti.astype(np.int64), axis=1)
    assert (steps.max(1) == 32768).sum() > 10 and (steps.max(1) > 65000).sum() > 10
    # every coded symbol has a non-empty bin
    assert (Tc[np.arange(len(lab)), lab + 1] > Tc[np.arange(len(lab)), lab])[cod].all()
