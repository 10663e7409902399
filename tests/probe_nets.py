"""Probe networks for the entropy codec: parameters whose fp32 arithmetic is exact, so the network outputs, the CDF tables
and the two bitstreams are known at every position without running any kernel.

The code-stream network reads (q - 3.5) * mask, a multiple of 0.5 in [-3.5, 3.5].  The probes put weights that are powers
of two on a few taps, with dyadic biases and the default PReLU slope 0.25: every partial sum is a short dyadic number,
exactly representable in fp32, so any summation order gives the same bits (this repo's, the reference's lane tree, the
oracle's double accumulation, the closed form below).  The importance network reads levels * 2/47 - 1, which is not
dyadic: there every output has at most two nonzero addends (a power-of-two product and the bias), and the sum of two
floats is rounded once in any order.  closed_form() checks both properties layer by layer.

Tables are steered into the regions ref64 can state exactly: deltas of 1e-6 or 2^-12 * value (every bin edge but an
exact hit saturates the normal CDF), mixture logits scaled by 256 or 512 (two components either tie or differ by 32 or
more), softmax logits of 0, +-60 or 4096 * value (one-hot, two or three tied maxima).  The extreme-table probe takes the
adversarial GMM rows of test_ref64 as per-group biases.

Every probe also puts nonzero weights on taps the context mask forbids (future positions, the own-group centre of the
first layer, groups above the output's); the closed form skips them, so a mask rule off by one in any packer changes
the bytes.
"""
import numpy as np

from oracle import oracle as O

G, CPG, NLAST = 48, 4, 3
LAYER_KEYS = ['net.0'] + ['net.%d.conv%d' % (b, c) for b in range(1, 6) for c in (1, 2)] + ['net.6']
FORBIDDEN = 2.0
PROBES = ("R", "P", "E")


def _empty(ngroup, cpg, nlast, nsets):
    p = {}
    lead = (nsets,) if nsets else ()
    for li, k in enumerate(LAYER_KEYS):
        cin = ngroup * (1 if li == 0 else cpg)
        cout = ngroup * (nlast if li == 11 else cpg)
        p[k + '.weight'] = np.zeros(lead + (cout, cin, 5, 5), np.float32)
        p[k + '.bias'] = np.zeros(lead + (cout,), np.float32)
        if li < 11:
            p[k + '.relu'] = np.full(lead + (cout,), 0.25, np.float32)
    return p


def _code_R(p):
    """R terms: layer 0 reads the same group's left neighbour (wavefront p-1); the last layer reads the centre tap of the
    same group (a Q term).  Weight logits [256 y, 0, 0], delta 2^-12 y, means y, y + 1/2 (a bin edge), 1 - y."""
    W0, W6, b6 = p['net.0.weight'], p['net.6.weight'], p['net.6.bias']
    for g in range(G):
        W0[:, 4 * g, g, 2, 1] = 1
        W6[0, 3 * g, 4 * g, 2, 2] = 256
        W6[1, 3 * g, 4 * g, 2, 2] = 2.0 ** -12
        W6[2, 3 * g, 4 * g, 2, 2] = 1
        W6[2, 3 * g + 1, 4 * g, 2, 2] = 1
        b6[2, 3 * g + 1] = 0.5
        W6[2, 3 * g + 2, 4 * g, 2, 2] = -1
        b6[2, 3 * g + 2] = 1


def _code_P(p):
    """P terms (wavefront <= p-2: group g-2 at the centre, the up-left neighbour) into hidden channel 1; a hidden path
    through blocks 2 and 4 (PReLU of negative values, a Q term and R terms: group g-1 at the centre, the left neighbour of
    a hidden channel) into channel 3; residual adds carry both.  The last layer mixes channels 1 (centre and the up
    neighbour) and 3."""
    W0, b0 = p['net.0.weight'], p['net.0.bias']
    c21, b21, c22 = p['net.2.conv1.weight'], p['net.2.conv1.bias'], p['net.2.conv2.weight']
    c41, c42, b42 = p['net.4.conv1.weight'], p['net.4.conv2.weight'], p['net.4.conv2.bias']
    W6, b6 = p['net.6.weight'], p['net.6.bias']
    for g in range(G):
        if g >= 2:
            W0[:, 4 * g + 1, g - 2, 2, 2] = 1
        W0[:, 4 * g + 1, g, 1, 1] = 0.5
        b0[:, 4 * g + 1] = 0.25
        c21[:, 4 * g + 2, 4 * g + 1, 2, 2] = 1
        if g >= 1:
            c21[:, 4 * g + 2, 4 * (g - 1) + 1, 2, 2] = -0.5
        b21[:, 4 * g + 2] = -0.5
        c22[:, 4 * g + 2, 4 * g + 2, 2, 2] = 2
        c41[:, 4 * g + 3, 4 * g + 2, 2, 2] = -1
        c41[:, 4 * g + 3, 4 * g + 1, 2, 1] = 1
        c42[:, 4 * g + 3, 4 * g + 3, 2, 2] = 1
        b42[:, 4 * g + 3] = 0.125
        W6[0, 3 * g, 4 * g + 1, 2, 2] = 512
        W6[0, 3 * g + 1, 4 * g + 1, 1, 2] = -512
        W6[1, 3 * g, 4 * g + 3, 2, 2] = 2.0 ** -20
        W6[2, 3 * g, 4 * g + 3, 2, 2] = 1
        W6[2, 3 * g + 1, 4 * g + 1, 2, 2] = 1
        b6[2, 3 * g + 1] = -1
        W6[2, 3 * g + 2, 4 * g + 2, 2, 2] = 0.5


def _code_E(p):
    """Extreme tables: even groups are bias-only with the adversarial GMM rows of test_ref64 (negative and zero deltas,
    means on bin edges and at +-40, logits of +-80, tied and equal logits; the rows clear of the rounding margin); odd
    groups are the R probe."""
    import ref64
    from test_ref64 import adversarial_gmm
    _code_R(p)
    w, d, m = adversarial_gmm()
    clear = ref64.clear_rows(ref64.gmm_table64(w, d, m)[1])
    w, d, m = w[clear], d[clear], m[clear]
    W6, b6 = p['net.6.weight'], p['net.6.bias']
    for g in range(0, G, 2):
        r = (g // 2) * (len(w) // 24)
        W6[:, 3 * g:3 * g + 3] = 0
        b6[0, 3 * g:3 * g + 3], b6[1, 3 * g:3 * g + 3], b6[2, 3 * g:3 * g + 3] = w[r], d[r], m[r]


def _code_forbidden(p):
    """nonzero weights on taps the mask removes (constraint 5: kh + kw + g_in < g_out + 4; 6: <=)"""
    W0 = p['net.0.weight']
    c11, c42, W6 = p['net.1.conv1.weight'], p['net.4.conv2.weight'], p['net.6.weight']
    for g in range(G):
        W0[:, 4 * g, g, 2, 2] = FORBIDDEN             # own group, own position: not yet decoded
        W0[:, 4 * g + 1, g, 2, 3] = FORBIDDEN         # right neighbour
        W0[:, 4 * g + 2, g, 3, 1] = FORBIDDEN         # down-left: wavefront p
        if g + 1 < G:
            W0[:, 4 * g, g + 1, 2, 1] = FORBIDDEN     # group g+1, left: wavefront p
            c11[:, 4 * g, 4 * (g + 1), 2, 2] = FORBIDDEN
            W6[:, 3 * g, 4 * (g + 1) + 1, 2, 2] = FORBIDDEN
        c11[:, 4 * g + 1, 4 * g, 3, 2] = FORBIDDEN    # below
        c42[:, 4 * g + 3, 4 * g + 3, 3, 3] = FORBIDDEN
        W6[:, 3 * g + 2, 4 * g + 1, 2, 3] = FORBIDDEN


def _imp(p, extreme):
    """Importance net: hidden channel 4 = PReLU(level of the upper neighbour, scaled), the one tap in the stack.
    Logits: index 10 = 4096 * h (one-hot when the upper level is above 23.5), 20 and 30 = 0 (two tied maxima below it,
    three at the top row); the extreme variant instead ties 0 and 48 at +60 and one-hots index 24 above 23.5.
    All others -60 (expf underflows: zero-width bins and the fix-up)."""
    W0, W6, b6 = p['net.0.weight'], p['net.6.weight'], p['net.6.bias']
    W0[4, 0, 1, 2] = 1
    W0[4, 0, 2, 2] = FORBIDDEN
    W0[4, 0, 2, 3] = FORBIDDEN
    p['net.1.conv1.weight'][4, 4, 3, 2] = FORBIDDEN
    b6[:] = -60
    if extreme:
        b6[0] = b6[48] = 60
        W6[24, 4, 2, 2] = 4096
    else:
        W6[10, 4, 2, 2] = 4096
        b6[10] = 0
        b6[20] = b6[30] = 0
    W6[10, 4, 3, 2] = FORBIDDEN


def probe_params(name):
    """numpy parameters in codec form ({'code': ..., 'imp': ...}, lic360_codec_ops.make_entropy_params layout)"""
    code, imp = _empty(G, CPG, NLAST, 3), _empty(1, 144, 49, None)
    {"R": _code_R, "P": _code_P, "E": _code_E}[name](code)
    _code_forbidden(code)
    _imp(imp, name == "E")
    return {'code': code, 'imp': imp}


def to_torch(params, device):
    import torch
    return {k: {kk: torch.from_numpy(vv).to(device).contiguous() for kk, vv in v.items()} for k, v in params.items()}


# ---- closed form ----------------------------------------------------------------------------------------------------
def _layer(x, Wt, b, slope, ngroup, constrain, resid=None):
    """x (Cin, H, W) float64 -> (Cout, H, W): the masked conv over the nonzero taps the mask keeps, + bias, PReLU, + resid.
    Also checks that fp32 gives the same bits in any order: forward and reverse fp32 accumulation of the addends agree,
    and every output of more than two nonzero addends is their exact sum."""
    Cout, Cin = Wt.shape[:2]
    cin_g, cout_g = Cin // ngroup, Cout // ngroup
    H, W = x.shape[1:]
    xp = np.pad(x, ((0, 0), (2, 2), (2, 2)))
    o, i, kh, kw = np.nonzero(Wt)
    lim = o // cout_g + 4 - (1 if constrain == 5 else 0)
    keep = kh + kw + i // cin_g <= lim
    out = np.zeros((Cout, H, W))
    addends = [[] for _ in range(Cout)]
    for oo, ii, hh, ww in zip(o[keep], i[keep], kh[keep], kw[keep]):
        addends[oo].append(float(Wt[oo, ii, hh, ww]) * xp[ii, hh:hh + H, ww:ww + W])
    for oo in range(Cout):
        terms = addends[oo] + [np.full((H, W), float(b[oo]))]
        tot = np.sum(terms, 0)
        f32 = np.zeros((H, W), np.float32)
        r32 = np.zeros((H, W), np.float32)
        for a in terms:
            f32 = (f32 + a.astype(np.float32)).astype(np.float32)
        for a in terms[::-1]:
            r32 = (r32 + a.astype(np.float32)).astype(np.float32)
        nnz = sum((a != 0).astype(np.int64) for a in terms)
        assert all(np.array_equal(a, a.astype(np.float32)) for a in terms), "a product is not an fp32 value"
        assert np.array_equal(f32, r32), "layer output %d depends on the summation order" % oo
        assert np.array_equal(np.where(nnz > 2, tot, f32), f32), \
            "layer output %d has more than two addends and is not exact" % oo
        out[oo] = f32
    if slope is not None:
        out = np.where(out > 0, out, out * slope[:, None, None].astype(np.float64))
    if resid is not None:
        s = out + resid
        assert np.array_equal(s, s.astype(np.float32))
        out = s
    return out


def net_forward(p, x, ngroup, nsets):
    """x (nsets, Cin, H, W) -> (nsets, Cout, H, W) float32: 12 masked convs, PReLU, 5 residual adds"""
    outs = []
    for s in range(nsets):
        def L(k, v, act=True, resid=None):
            w = p[k + '.weight'][s] if nsets > 1 else p[k + '.weight']
            b = p[k + '.bias'][s] if nsets > 1 else p[k + '.bias']
            a = None
            if act:
                a = p[k + '.relu'][s] if nsets > 1 else p[k + '.relu']
            return _layer(v, w, b, a, ngroup, 5 if k == 'net.0' else 6, resid)
        y = L('net.0', x[s].astype(np.float64))
        for blk in range(1, 6):
            y = L('net.%d.conv2' % blk, L('net.%d.conv1' % blk, y), resid=y)
        outs.append(L('net.6', y, act=False))
    return np.stack(outs).astype(np.float32)


def code_input(q, mask):
    return ((q[0] - 3.5) * mask[0]).astype(np.float32)[None].repeat(3, 0)   # (3, 48, H, W)


def imp_input(lv):
    # ScaleOp / TileInput: fmaf(level, 2/47, -1); the product of a small integer and a float is exact in float64
    return (lv[0].astype(np.float64) * np.float64(np.float32(2.0 / 47)) - 1.0).astype(np.float32)   # (1, H/2, W/2)


def closed_form(params, q, mask, lv):
    """network outputs of both streams: code (3, 144, H, W) = [weight, delta, mean] nets, imp (49, H/2, W/2)"""
    y_code = net_forward(params['code'], code_input(q, mask), G, 3)
    y_imp = net_forward(params["imp"], imp_input(lv)[None], 1, 1)[0]
    return y_code, y_imp


# ---- coding order and expected streams ------------------------------------------------------------------------------
def coding_order(H, W, ngroup):
    """(group, row, col) of every coded symbol in stream order: wavefront steps psum = 0..H+W+G-3, within a step the
    diagonals of its slab (oracle.slab) in index order, rows ascending within a diagonal (oracle.code_contex)."""
    idx, plan = O.code_contex(H, W)
    out = []
    for psum in range(H + W + ngroup - 2):
        st, ln = O.slab(plan, H, W, ngroup, psum)
        th, tw = idx[st:st + ln], idx[H * W + st:H * W + st + ln]
        out.append(np.stack([psum - th - tw, th, tw], 1))
    return np.concatenate(out).astype(np.int64)


def expected_tables(params, q, mask, lv):
    """ref64 tables in coding order: (code tables, code labels, code mask, imp tables, imp labels), with the rows the
    coder reads checked to be clear of the rounding margin"""
    import ref64
    y_code, y_imp = closed_form(params, q, mask, lv)
    H, W = q.shape[2:]
    c, h, w = coding_order(H, W, G).T
    gw = y_code[0].reshape(G, 3, H, W)[c, :, h, w]
    gd = y_code[1].reshape(G, 3, H, W)[c, :, h, w]
    gm = y_code[2].reshape(G, 3, H, W)[c, :, h, w]
    Tc, mc, _ = ref64.gmm_table64(gw, gd, gm)
    lab_c = q[0, c, h, w].astype(np.int32)
    msk = mask[0, c, h, w].astype(np.float32)
    coded = msk > 0.5
    assert ref64.clear_rows(mc[coded]).all(), "a coded code-stream row is inside the rounding margin"
    _, hi, wi = coding_order(H // 2, W // 2, 1).T
    Ti, mi, _ = ref64.entropy_table64(y_imp[:, hi, wi].T)
    assert ref64.clear_rows(mi).all(), "an importance row is inside the rounding margin"
    return Tc.astype(np.int32), lab_c, msk, Ti.astype(np.int32), lv[0, 0, hi, wi].astype(np.int32)


def host_encode(tab, lab, mask):
    """the product's host coder (lic360_coder_encodes, pinned against the reference's coder classes by test_oracle_coder)"""
    import ctypes
    from lic360 import _lib
    L = _lib.LIB
    h = ctypes.c_void_p(L.lic360_coder_create(b"unused", 3.5))
    try:
        assert L.lic360_coder_start_encoder_mem(h) == 0
        if tab.shape[0]:
            tab, lab = np.ascontiguousarray(tab, np.int32), np.ascontiguousarray(lab, np.int32)
            mask = None if mask is None else np.ascontiguousarray(mask, np.float32)
            rc = L.lic360_coder_encodes(h, tab.ctypes.data, tab.shape[1] - 1, lab.ctypes.data,
                                        None if mask is None else mask.ctypes.data, tab.shape[0])
            if rc:
                raise RuntimeError(L.lic360_last_error().decode())
        n = L.lic360_coder_finish_mem(h)
        buf = np.zeros(max(n, 1), np.uint8)
        L.lic360_coder_get_bytes(h, buf.ctypes.data, n)
        return buf[:n].tobytes()
    finally:
        L.lic360_coder_destroy(h)


def expected_streams(params, q, mask, lv):
    """(importance stream, code stream) the codec must write for this latent"""
    Tc, lab_c, msk, Ti, lab_i = expected_tables(params, q, mask, lv)
    return host_encode(Ti, lab_i, None), host_encode(Tc, lab_c, msk)
