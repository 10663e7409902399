"""Entropy codec of one ERP image latent: importance stream + code stream, encode and decode.

This is the call a user of the reference makes through test/lic360_demo.py (`encoding` :339-368: ImpEntEncoderFast
then EntEncoderFast on the outputs of CMP_Encoder; `decoding` :376-404: ImpEntDecoder -> Imp2mask -> Dtow ->
EntDecoder), packaged as one object so that bench.py and the tests drive exactly the path the metric is quoted on.

`PerOpCodec` drives the per-op loops (lic360_codec_ops.py) on any backend exposing the `lic360` op surface -- this
repo's mirror or the reference extension.
"""
import ctypes
import os
import tempfile

import torch

import lic360_codec_ops as ops
from lic360._lib import LIB, check

LAYER_KEYS = ['net.0'] + ['net.%d.conv%d' % (b, c) for b in range(1, 6) for c in (1, 2)] + ['net.6']


def make_codec_params(device, seed=2024):
    """Seeded random-init parameters of both entropy networks in the model-idx-3 shape (the architecture is fixed:
    channels=192, code_channels=192, quant_levels=8, test/model_zoo.py:337; the index only selects a weight file)."""
    return {
        'code': ops.make_entropy_params(48, 4, 3, 3, seed, device),
        'imp': ops.make_entropy_params(1, 144, 49, None, seed + 1, device),
    }


class PerOpCodec(object):
    def __init__(self, backend, params, gid=0, workdir=None):
        self.backend, self.gid = backend, gid
        self.dev = 'cuda:%d' % gid
        self.imp_enc = ops.ImpEntEncoder(backend, params['imp'], 48, gid)
        self.code_enc = ops.EntEncoder(backend, params['code'], 48, 8, gid)
        self.imp_dec = ops.ImpEntDecoder(backend, params['imp'], 48, gid)
        self.code_dec = ops.EntDecoder(backend, params['code'], 48, 8, gid)
        self.i2m = backend.Imp2maskOp(48, 192, gid, False)
        self.d2w = backend.DtowOp(2, True, gid, False)
        self._tmp = tempfile.mkdtemp(prefix='lic360_', dir=workdir or ('/dev/shm' if os.path.isdir('/dev/shm') else None))

    def encode(self, code, mask, imap_quant, name='img'):
        """code, mask: (1,48,H/8,W/8) device tensors (qy_up, mask_up); imap_quant: (1,1,H/16,W/16) importance levels.
        Returns (bytes of <name>_imp, bytes of <name>), lic360_demo.py:361-365."""
        fo = os.path.join(self._tmp, name)
        self.imp_enc.encode(imap_quant, fo + '_imp')
        self.code_enc.encode(code, mask, fo)
        with open(fo + '_imp', 'rb') as f1, open(fo, 'rb') as f2:
            return f1.read(), f2.read()

    def decode(self, imp_bytes, code_bytes, h, w, name='img'):
        """h, w: importance-map size (H/16, W/16). Returns (code, mask_up) like lic360_demo.py:395-398."""
        fo = os.path.join(self._tmp, name)
        with open(fo + '_imp', 'wb') as f1, open(fo, 'wb') as f2:
            f1.write(imp_bytes)
            f2.write(code_bytes)
        levels = self.imp_dec.decode(fo + '_imp', h, w, self.dev)
        mask_up = self.d2w.forward(self.i2m.forward(levels)[0])[0]
        code = self.code_dec.decode(mask_up, fo)
        return code, mask_up


class FusedCodec(object):
    """The product path: one image per codec on its own CUDA stream, the whole encode / decode loop in native code
    (csrc/codec.cu): one graph replay + one host coder call per wavefront step, no Python in the loop."""

    def __init__(self, params, H=64, W=128, gid=0, mode=None):
        """mode: None / 0 = graph replay per wavefront step (several images in flight per GPU), 2 = low latency (one persistent
        chain kernel per decode; one image at a time), 1 = serialized per-kernel timing (profiling)."""
        self.H, self.W, self.gid = H, W, gid
        self.dev = torch.device('cuda', gid)
        h = LIB.lic360_codec_create(gid, H, W)
        if not h:
            check(1)
        self._h = ctypes.c_void_p(h)
        # the codec packs the weights on its OWN stream: whatever produced them on torch's stream must have finished
        torch.cuda.current_stream(self.dev).synchronize()
        for sid, key, G, cpg, nlast, nsets in ((0, 'code', 48, 4, 3, 3), (1, 'imp', 1, 144, 49, None)):
            p = params[key]
            for layer, lk in enumerate(LAYER_KEYS):
                cin = G * (1 if layer == 0 else cpg)
                cout = G * (nlast if layer == 11 else cpg)
                lead = () if nsets is None else (nsets,)
                w = self._param(p[lk + '.weight'], lead + (cout, cin, 5, 5), lk + '.weight')
                b = self._param(p[lk + '.bias'], lead + (cout,), lk + '.bias')
                slope = p.get(lk + '.relu')
                if slope is not None:
                    slope = self._param(slope, lead + (cout,), lk + '.relu')
                elif layer != 11:
                    raise RuntimeError("FusedCodec: %s.%s.relu is missing" % (key, lk))
                check(LIB.lic360_codec_set_layer(self._h, sid, layer, w.data_ptr(), b.data_ptr(),
                                                 None if slope is None else slope.data_ptr()))

        if mode:
            self.set_mode(mode)

    def _param(self, t, shape, name):
        """float32, contiguous, on the codec's device, of the reference's shape -- anything else would be read as garbage
        (or fault) by the native packer."""
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.device != self.dev:
            raise RuntimeError("FusedCodec: parameter %s must live on %s" % (name, self.dev))
        if t.dtype != torch.float32:
            raise RuntimeError("FusedCodec: parameter %s must be float32 (got %s)" % (name, t.dtype))
        if tuple(t.shape) != tuple(shape):
            raise RuntimeError("FusedCodec: parameter %s has shape %s, expected %s" % (name, tuple(t.shape), tuple(shape)))
        t = t.detach()
        if not t.is_contiguous():
            t = t.contiguous()
            torch.cuda.current_stream(self.dev).synchronize()  # the copy ran on torch's stream, the packer reads on the codec's
        return t

    def __del__(self):
        h = getattr(self, '_h', None)
        if h and LIB is not None:
            LIB.lic360_codec_destroy(h)
            self._h = None

    def _f32(self, t, shape):
        if not (t.is_cuda and t.dtype == torch.float32 and t.device == self.dev):
            raise RuntimeError("FusedCodec: expected a float32 tensor on %s" % self.dev)
        if tuple(t.shape) != shape:
            raise RuntimeError("FusedCodec: expected shape %s, got %s" % (shape, tuple(t.shape)))
        return t.contiguous()

    def _stream_bytes(self, sid):
        n = LIB.lic360_codec_stream_size(self._h, sid)
        buf = (ctypes.c_uint8 * max(n, 1))()
        LIB.lic360_codec_stream_copy(self._h, sid, buf, n)
        return bytes(buf[:n])

    def encode(self, code, mask, imap_quant, name=None):
        code = self._f32(code, (1, 48, self.H, self.W))
        mask = self._f32(mask, (1, 48, self.H, self.W))
        imp = self._f32(imap_quant, (1, 1, self.H // 2, self.W // 2))
        torch.cuda.current_stream(self.dev).synchronize()  # inputs were produced on torch's stream
        check(LIB.lic360_codec_encode(self._h, code.data_ptr(), mask.data_ptr(), imp.data_ptr()))
        return self._stream_bytes(1), self._stream_bytes(0)

    def estimate(self, code, mask, imap_quant):
        """The rate of the latent `encode` would code, without the arithmetic coder: the same networks and integer CDF rows, and for
        every coded symbol its ideal code length 16 - log2(T[s+1] - T[s]) bits (include/lic360_b200.h, lic360_codec_estimate).

        Returns {'code_bits': float, 'imp_bits': float, 'code_map': (1,48,H,W), 'imp_map': (1,1,H/2,W/2)}: the totals of the code and
        importance streams and the bits of every symbol as float32 tensors on the codec's device (0 where mask < 0.5).  The image
        is 8H x 8W pixels, so its rate is (code_bits + imp_bits) / (64 H W) bits per pixel.  For each stream, with N coded symbols
        and I its total, the bytes `encode` writes satisfy -(1 + u + N/8192) <= 8 * len(stream) - I <= 8 + N/8192, where u is the
        number of pending underflow bits the coder drops at the end (a few at most in practice; derivation in
        tests/test_rate_estimate.py).  Raises RuntimeError on the inputs `encode` refuses, with the same message."""
        code = self._f32(code, (1, 48, self.H, self.W))
        mask = self._f32(mask, (1, 48, self.H, self.W))
        imp = self._f32(imap_quant, (1, 1, self.H // 2, self.W // 2))
        code_map = torch.empty((1, 48, self.H, self.W), dtype=torch.float32, device=self.dev)
        imp_map = torch.empty((1, 1, self.H // 2, self.W // 2), dtype=torch.float32, device=self.dev)
        totals = (ctypes.c_double * 2)()
        torch.cuda.current_stream(self.dev).synchronize()  # inputs were produced on torch's stream
        check(LIB.lic360_codec_estimate(self._h, code.data_ptr(), mask.data_ptr(), imp.data_ptr(), code_map.data_ptr(),
                                        imp_map.data_ptr(), totals))
        return {'code_bits': totals[0], 'imp_bits': totals[1], 'code_map': code_map, 'imp_map': imp_map}

    def decode(self, imp_bytes, code_bytes, h=None, w=None, name=None):
        code = torch.empty((1, 48, self.H, self.W), dtype=torch.float32, device=self.dev)
        mask = torch.empty((1, 48, self.H, self.W), dtype=torch.float32, device=self.dev)
        torch.cuda.current_stream(self.dev).synchronize()
        check(LIB.lic360_codec_decode(self._h, imp_bytes, len(imp_bytes), code_bytes, len(code_bytes), code.data_ptr(),
                                      mask.data_ptr()))
        return code, mask

    def set_mode(self, mode):
        """0: pipelined graph replay per step (default); 1: serialized launches with per-kernel CUDA-event timing; 2: low latency
        (one persistent code-stream chain kernel per decode, include/lic360_b200.h)."""
        check(LIB.lic360_codec_set_mode(self._h, int(mode)))

    def kernel_times(self, stream_id=0):
        """After a mode-1 decode: ms spent per kernel class of one stream (0 = code, 1 = importance)."""
        out = (ctypes.c_double * 5)()
        check(LIB.lic360_codec_kernel_times(self._h, stream_id, out, 5))
        return {'old_ms': out[0], 'prev_ms': out[1], 'chain_ms': out[2], 'scatter_rows_ms': out[3], 'steps': int(out[4])}

    def last_timing(self):
        out = (ctypes.c_double * 6)()
        LIB.lic360_codec_last_timing(self._h, out, 6)
        return {'total_ms': out[0], 'host_coder_ms': out[1], 'gpu_wait_ms': out[2], 'imp_stream_ms': out[3],
                'gpu_steps_ms': out[4], 'imp_gpu_steps_ms': out[5]}
