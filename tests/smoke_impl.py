"""__graft_entry__.smoke(): one small invocation of the hot path on cuda:0, checked against the oracle."""
import os
import tempfile

import numpy as np
import torch


def run_smoke():
    import lic360
    import lic360_codec_ops as ops
    from oracle import oracle as O
    from op_cases import BY_NAME
    from util import rel_err, synthetic_latent, t, n

    dev = "cuda:0"
    l0 = lic360.launch_count()
    # 1. FIRST (so that the wavefront-engine kernels -- wf_old4_kernel, wf_chain4_kernel, wf_chain1_kernel -- are inside the
    # driver's launch window): the product path, the fused native codec, both streams, encode -> bitstreams -> decode == input
    import lic360_pipeline as pl
    q2, mask2, lv2 = synthetic_latent(8, H=16, W=32)
    cp = pl.make_codec_params(dev, seed=5)
    fused = pl.FusedCodec(cp, H=16, W=32)
    bi, bc = fused.encode(t(q2, dev), t(mask2, dev), t(lv2, dev))
    code, mup = fused.decode(bi, bc)
    assert np.array_equal(n(code), q2 * mask2) and np.array_equal(n(mup), mask2), "fused codec round trip failed"
    # ... checked against the oracle: the CPU rendition of the same codec (oracle/cpu_codec.py) emits streams of the same size
    # (the conv is float-tier, so single bins may differ by one count; the op-level checks below are the exact ones)
    from oracle import cpu_codec
    cpu = cpu_codec.CpuCodec(cpu_codec.params_to_numpy({k: {kk: vv.cpu() for kk, vv in v.items()} for k, v in cp.items()}))
    ci, cc = cpu.encode(q2, mask2, lv2)
    assert abs(len(ci) - len(bi)) <= 2 and abs(len(cc) - len(bc)) <= max(2, 0.002 * len(cc)), (len(ci), len(bi), len(cc), len(bc))
    fused_launches = lic360.launch_count() - l0
    # 2. one masked context-conv layer: whole-frame (EC) and wavefront (DC) forms against the oracle, EC == DC bitwise
    ec = BY_NAME["cconv_ec_batch_hidden_g12"].run(lic360, dev)["out"]
    dc = BY_NAME["cconv_dc_batch_hidden_g12"].run(lic360, dev)["out"]
    ref = BY_NAME["cconv_ec_batch_hidden_g12"].oracle()["out"]
    assert rel_err(ec, ref) <= 1e-5, rel_err(ec, ref)
    assert np.array_equal(ec.view(np.int32), dc.view(np.int32)), "EC != DC"
    # 3. GMM -> CDF tables
    c = BY_NAME["gmm_table_full"]
    got, exp = c.run(lic360, dev)["table"], c.oracle()["table"]
    assert np.abs(got.astype(np.int64) - exp).max() <= 1 and (np.diff(got, axis=1) > 0).all()
    # 4. tiny end-to-end code stream (per-op loops): encode -> bitstream -> decode == input
    q, mask, _ = synthetic_latent(7, H=8, W=16)
    params = ops.make_entropy_params(48, 4, 3, 3, seed=3, device=dev)
    with tempfile.TemporaryDirectory() as d:
        fn = os.path.join(d, "code")
        ops.EntEncoder(lic360, params).encode(t(q, dev), t(mask, dev), fn)
        rec = n(ops.EntDecoder(lic360, params).decode(t(mask, dev), fn))
        nbytes = os.path.getsize(fn)
    assert np.array_equal(rec, q * mask), "round trip failed"
    torch.cuda.synchronize()
    print("smoke OK: conv rel err %.2e, EC==DC bitwise, tables within 1 count of the oracle, round trip of %d symbols in %d bytes, "
          "fused codec round trip in %d+%d bytes (CPU oracle codec: %d+%d), %d native launches (%d by the fused codec)"
          % (rel_err(ec, ref), int(mask.sum()), nbytes, len(bi), len(bc), len(ci), len(cc), lic360.launch_count() - l0, fused_launches))
