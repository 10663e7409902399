"""numpy front-end of canon_conv.c: the canonical fp32 order of the masked context conv (header of csrc/conv.cu),
bit for bit, on the CPU.  layer() is one CconvEc / CconvDc layer, net() the 12-layer entropy network of the codec
(lic360_codec_ops._Net wiring: layer 0, five residual blocks, the last layer without PReLU)."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "canon_conv.c")
_FLAGS = ["-O3", "-mavx2", "-mfma", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC"]
CANONICAL, FLAT_CHAIN, PQR = 0, 1, 2  # variants: the canonical order and two orders it must tell apart from


def _load():
    so = os.path.join(_HERE, "libcanon_conv.so")
    if not os.access(_HERE, os.W_OK):  # a read-only checkout: build into the temporary directory
        so = os.path.join(tempfile.gettempdir(), "lic360_canon_conv_%d.so" % os.getuid())
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(_SRC):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call(["gcc"] + _FLAGS + ["-o", tmp, _SRC, "-lm"])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    lib.canon_cconv.argtypes = [ctypes.c_void_p] * 6 + [ctypes.c_int] * 9
    lib.canon_cconv.restype = None
    return lib


_L = _load()


def _f(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float32)


def layer(x, w, b, slope, G, constrain, nsets=1, resid=None, variant=CANONICAL):
    """x (N, Cin, H, W), w ((nsets,) Cout, Cin, 5, 5), b / slope ((nsets,) Cout), slope None = no PReLU,
    resid (N, Cout, H, W) or None -> (N, Cout, H, W) float32; images n use parameter set n // (N / nsets)."""
    x, w, b, slope, resid = _f(x), _f(w), _f(b), _f(slope), _f(resid)
    N, Cin, H, W = x.shape
    Cout = w.shape[-4]
    assert w.shape[-4:] == (Cout, Cin, 5, 5) and w.size == nsets * Cout * Cin * 25 and b.size == nsets * Cout
    assert Cin % G == 0 and Cout % G == 0 and N % nsets == 0 and constrain in (5, 6)
    assert resid is None or resid.shape == (N, Cout, H, W)
    out = np.empty((N, Cout, H, W), np.float32)
    p = lambda a: None if a is None else a.ctypes.data
    _L.canon_cconv(p(x), p(w), p(b), p(slope), p(resid), p(out), N, Cin, Cout, G, H, W, constrain, nsets, variant)
    return out


def allowed(Cout, Cin, G, constrain):
    """(Cout, Cin, 5, 5) bool: the taps the context mask keeps (g_in <= glim - 1, or <= glim for constrain 6)"""
    g_out = (np.arange(Cout) // (Cout // G))[:, None, None, None]
    g_in = (np.arange(Cin) // (Cin // G))[None, :, None, None]
    k = np.arange(5)
    glim = g_out + 4 - k[:, None] - k[None, :]
    return g_in <= glim - (1 if constrain == 5 else 0)


def dynamic_input(r, shape):
    """x ~ N(0, 1) * 2^U(-6, 6), 10% exact +0 and 10% -0 (the code stream feeds (q - 3.5) * 0 = -0)"""
    x = r.standard_normal(shape) * 2.0 ** r.uniform(-6, 6, shape)
    z = r.random(shape)
    x[z < 0.1] = 0.0
    x[(z >= 0.1) & (z < 0.2)] = -0.0
    return x.astype(np.float32)


def layer_params(r, nsets, G, Cin, Cout, constrain):
    """He-normal weights with NaN on every tap the mask forbids, random bias and PReLU slope ((nsets,) leading dim)"""
    lead = (nsets,) if nsets else ()
    w = (r.standard_normal(lead + (Cout, Cin, 5, 5)) * (2.0 / (Cin * 25)) ** 0.5).astype(np.float32)
    w[..., ~allowed(Cout, Cin, G, constrain)] = np.nan
    b = (r.standard_normal(lead + (Cout,)) * 0.1).astype(np.float32)
    a = (0.25 + 0.1 * r.standard_normal(lead + (Cout,))).astype(np.float32)
    return w, b, a


def exact64(x, w, b, G, constrain, nsets=1):
    """float64 reference of the conv before PReLU / residual: (S, A, n) with S (N, Cout, H, W) the sum of the kept
    products and the bias (products of floats are exact in float64; the float64 sum is off by ~n * 2^-53 * A),
    A the sum of their magnitudes, n (Cout,) the number of fp32 roundings on the path of any term of one output in the
    canonical order (one per kept tap, one per block fold, three for P + R + Q + bias)"""
    x = np.asarray(x, np.float64)
    N, Cin, H, W = x.shape
    w = np.asarray(w, np.float32).reshape(nsets, -1, Cin, 5, 5)
    b = np.asarray(b, np.float32).reshape(nsets, -1).astype(np.float64)
    Cout = w.shape[1]
    keep = allowed(Cout, Cin, G, constrain)
    wm = np.where(keep, w, 0).astype(np.float64)
    xp = np.pad(x, ((0, 0), (0, 0), (2, 2), (2, 2)))
    per = N // nsets
    S = np.zeros((N, Cout, H, W))
    A = np.zeros((N, Cout, H, W))
    for n in range(N):
        s = n // per
        for kh in range(5):
            for kw in range(5):
                xs = xp[n, :, kh:kh + H, kw:kw + W].reshape(Cin, H * W)
                S[n] += (wm[s, :, :, kh, kw] @ xs).reshape(Cout, H, W)
                A[n] += (np.abs(wm[s, :, :, kh, kw]) @ np.abs(xs)).reshape(Cout, H, W)
        S[n] += b[s][:, None, None]
        A[n] += np.abs(b[s])[:, None, None]
    cin_g = Cin // G
    nops = keep.reshape(Cout, -1).sum(1) + (Cin + 15) // 16 + 2 * ((cin_g + 15) // 16) + 3
    return S, A, nops


def gamma(n, unit=2.0 ** -24):
    n = np.asarray(n, np.float64)
    return n * unit / (1 - n * unit)


def error_bound(S, A, nops, slope, resid, nsets=1, conv_gamma=None):
    """(reference, bound): an fp32 evaluation of the layer in any summation order with at most nops roundings on the
    path of each term is within bound of reference.  The conv: gamma_n * A, plus the float64 sum's own error.  PReLU:
    the computed and the exact sum can only have different signs when both are within the conv bound, so the error
    grows to max(1, |slope|) times it, plus the rounding of v * slope.  Residual: plus the rounding of the final add.
    conv_gamma replaces gamma_n for a kernel with a different error model (the tensor-core pass)."""
    u = 2.0 ** -24
    N, Cout = S.shape[:2]
    cg = gamma(nops) if conv_gamma is None else np.asarray(conv_gamma, np.float64)
    E = cg[None, :, None, None] * A + gamma(nops.max(), 2.0 ** -53) * A
    ref = S
    if slope is not None:
        sl = np.asarray(slope, np.float32).reshape(nsets, Cout).astype(np.float64).repeat(N // nsets, 0)[:, :, None, None]
        ref = np.where(S > 0, S, S * sl)
        E = np.maximum(1, np.abs(sl)) * E + u * np.abs(sl) * (np.abs(S) + E)
    if resid is not None:
        ref = ref + np.asarray(resid, np.float64)
        E = E + u * (np.abs(ref) + E)
    return ref, E


def net(params, x, ngroup, nsets):
    """params: codec-form dict of numpy arrays (lic360_codec_ops.make_entropy_params keys, leading dim nsets when
    nsets > 1); x (nsets, Cin, H, W) -> (nsets, Cout, H, W) float32, image s through parameter set s"""
    p = {k: np.asarray(v, np.float32) for k, v in params.items()}

    def L(k, v, act=True, resid=None):
        return layer(v, p[k + '.weight'], p[k + '.bias'], p[k + '.relu'] if act else None, ngroup,
                     5 if k == 'net.0' else 6, nsets, resid)
    y = L('net.0', x)
    for blk in range(1, 6):
        y = L('net.%d.conv2' % blk, L('net.%d.conv1' % blk, y), resid=y)
    return L('net.6', y, act=False)
