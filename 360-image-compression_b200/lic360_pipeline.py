"""Entropy codec of one ERP image latent: importance stream + code stream, encode and decode.

This is the call a user of the reference makes through test/lic360_demo.py (`encoding` :339-368: ImpEntEncoderFast
then EntEncoderFast on the outputs of CMP_Encoder; `decoding` :376-404: ImpEntDecoder -> Imp2mask -> Dtow ->
EntDecoder), packaged as one object so that bench.py and the tests drive exactly the path the metric is quoted on.

`PerOpCodec` drives the per-op loops (lic360_codec_ops.py) on any backend exposing the `lic360` op surface -- this
repo's mirror or the reference extension.
"""
import ctypes
import math
import os
import tempfile

import torch

import lic360_codec_ops as ops
from lic360._lib import LIB, check, cstream

LAYER_KEYS = ['net.0'] + ['net.%d.conv%d' % (b, c) for b in range(1, 6) for c in (1, 2)] + ['net.6']


def make_codec_params(device, seed=2024):
    """Seeded random-init parameters of both entropy networks in the model-idx-3 shape (the architecture is fixed:
    channels=192, code_channels=192, quant_levels=8, test/model_zoo.py:337; the index only selects a weight file)."""
    return {
        'code': ops.make_entropy_params(48, 4, 3, 3, seed, device),
        'imp': ops.make_entropy_params(1, 144, 49, None, seed + 1, device),
    }


def _protect_map(protect, imap_quant):
    """protect as lic360_imp_levels_to_mask_protected reads it: a (K,1,h,w) integer tensor on imap_quant's device with values in
    [0, 48], converted to contiguous int32 (K = 1 for one latent)"""
    if not (isinstance(protect, torch.Tensor) and protect.device == imap_quant.device and not protect.dtype.is_floating_point
            and not protect.dtype.is_complex and protect.dtype != torch.bool and tuple(protect.shape) == tuple(imap_quant.shape)):
        raise RuntimeError("levels_to_mask: protect must be a (%d,1,h,w) integer tensor on %s, like the importance map"
                           % (imap_quant.shape[0], imap_quant.device))
    p = protect.to(torch.int32).contiguous()
    lo, hi = int(p.min()), int(p.max())
    if lo < 0 or hi > 48:
        raise RuntimeError("levels_to_mask: protect values must lie in [0, 48] (got %d .. %d)" % (lo, hi))
    return p


def levels_to_mask(imap_quant, offsets, protect=None):
    """Candidate importance maps for rate control and the code masks the decoder derives from them (lic360_imp_levels_to_mask,
    lic360_imp_levels_to_mask_protected).

    imap_quant: (1,1,h,w) float32 CUDA tensor of importance levels as `encode` reads them (s = int(level), the symbol it codes);
    offsets: K integers t >= 0; protect: None, or a (1,1,h,w) integer tensor on the same device with values P in [0, 48].
    Returns (levels, masks) on the input's device: levels (K,1,h,w) = max(s - max(t - P, 0), 0) for t = offsets[j] (P = 0 without
    a map: max(s - t, 0)) and masks (K,48,2h,2w), channel c at (y, x) = 1 iff 4c + 2 (y % 2) + x % 2 < 4 * level(y/2, x/2).
    A cell keeps its level until t > P.  `encode(code, masks[j:j+1], levels[j:j+1])` gives streams that decode to exactly masks[j]."""
    if not (isinstance(imap_quant, torch.Tensor) and imap_quant.is_cuda and imap_quant.dtype == torch.float32
            and imap_quant.dim() == 4 and tuple(imap_quant.shape[:2]) == (1, 1)):
        raise RuntimeError("levels_to_mask: expected a (1,1,h,w) float32 CUDA tensor")
    offs = [int(k) for k in offsets]
    K, (h, w) = len(offs), imap_quant.shape[2:]
    dev = imap_quant.device
    levels = torch.empty((K, 1, h, w), dtype=torch.float32, device=dev)
    masks = torch.empty((K, 48, 2 * h, 2 * w), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        lv = imap_quant.contiguous()
        offs_c = (ctypes.c_int * max(K, 1))(*offs)
        if protect is None:
            check(LIB.lic360_imp_levels_to_mask(lv.data_ptr(), h, w, offs_c, K, levels.data_ptr(), masks.data_ptr(), cstream(lv)))
        else:
            p = _protect_map(protect, imap_quant)
            check(LIB.lic360_imp_levels_to_mask_protected(lv.data_ptr(), h, w, offs_c, K, p.data_ptr(), levels.data_ptr(),
                                                          masks.data_ptr(), cstream(lv)))
    return levels, masks


def levels_to_mask_batch(imap_quant, cand_latent, cand_offset, protect=None):
    """levels_to_mask of J candidates of K importance maps (lic360_imp_levels_to_mask_batch): imap_quant (K,1,h,w) float32 CUDA;
    candidate j is map cand_latent[j] in [0, K) at offset cand_offset[j] >= 0; protect: None or a (K,1,h,w) integer map per latent,
    checked as levels_to_mask checks it.  Returns (levels (J,1,h,w), masks (J,48,2h,2w)); entry j is bit-identical to
    levels_to_mask(imap_quant[k:k+1], [t], protect[k:k+1]) of its latent k and offset t."""
    if not (isinstance(imap_quant, torch.Tensor) and imap_quant.is_cuda and imap_quant.dtype == torch.float32
            and imap_quant.dim() == 4 and imap_quant.shape[1] == 1):
        raise RuntimeError("levels_to_mask_batch: expected a (K,1,h,w) float32 CUDA tensor")
    lat, offs = [int(k) for k in cand_latent], [int(t) for t in cand_offset]
    if len(lat) != len(offs):
        raise RuntimeError("levels_to_mask_batch: %d latents for %d offsets" % (len(lat), len(offs)))
    (K, _, h, w), J = imap_quant.shape, len(lat)
    dev = imap_quant.device
    levels = torch.empty((J, 1, h, w), dtype=torch.float32, device=dev)
    masks = torch.empty((J, 48, 2 * h, 2 * w), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        lv = imap_quant.contiguous()
        p = None if protect is None else _protect_map(protect, imap_quant)
        check(LIB.lic360_imp_levels_to_mask_batch(lv.data_ptr(), K, h, w, None if p is None else p.data_ptr(), J,
                                                  (ctypes.c_int * max(J, 1))(*lat), (ctypes.c_int * max(J, 1))(*offs),
                                                  levels.data_ptr(), masks.data_ptr(), cstream(lv)))
    return levels, masks


def latitude_protection(h, w, levels, device=None):
    """Protection map (1,1,h,w) int32 for encode_to_budget / levels_to_mask that follows ERP's cos-latitude area weight: row i gets
    round(levels * cos(phi_i)), phi_i = pi/2 - pi (i + 0.5) / h its centre latitude.  The equator rows keep their levels longest,
    the polar rows, which ERP oversamples by 1 / cos(phi), are lowered first.  levels: integer in [0, 48]; device: any torch
    device (CPU included).  Combine maps with torch.maximum."""
    levels = _preset_levels(levels)
    phi = math.pi / 2 - math.pi * (torch.arange(h, dtype=torch.float64) + 0.5) / h
    rows = torch.round(levels * torch.cos(phi)).to(torch.int32)
    return rows.view(1, 1, h, 1).expand(1, 1, h, w).contiguous().to(device)


def viewport_protection(h, w, views, levels, fov=0.6, device=None):
    """Protection map (1,1,h,w) int32 for encode_to_budget / levels_to_mask: `levels` on the cells the chosen viewports see, 0
    elsewhere.  views: indices into MultiProject's 14 viewports (lic360_operator._modules.VIEWPORT_THETAS / VIEWPORT_PHIS; 1 is the
    front view, 12 and 13 the poles); fov: the viewports' field of view in units of pi (MultiProject's default); device: a CUDA
    device (default: the current one).  Combine maps with torch.maximum, e.g. with latitude_protection.

    A cell is in the footprint iff it carries a non-zero bilinear weight for at least one pixel of a chosen viewport, rendered by
    lic360.ProjectsOp (the projection MultiProject's viewport metrics use) from the h x w grid at n x n pixels: one forward, then
    one backward whose gradient is 1 on the chosen viewports and 0 elsewhere; the footprint is where the scattered weight is > 0.

    Why n leaves no holes: neighbouring viewport pixels are at most p = 2 tan(a) / (n - 1) apart on the sphere, a = fov * pi / 2
    (at the viewport's centre; rectilinear pixels get denser towards its edges), and a pixel's bilinear taps cover the two cells
    on either side of it along each axis.  So every cell inside the viewport is hit where p is below two cells, 2 pi / h along a
    column and 4 pi cos(phi) / w along a row at latitude phi.  n = 2w meets this away from the poles (for the default fov up to
    |phi| of 83 degrees); where a chosen viewport comes closer to a pole, the cells of the rows there narrow with cos(phi), and
    the first row, 2 pi sin(pi / h) / w wide, is the narrowest: n is raised to meet the bound at the highest latitude the viewport
    reaches, capped at that row, with a factor 1.25 for the uneven directions of the pixel grid around the pole.  That costs
    O(h w) pixels per side for the polar and the +-0.25 viewports (about 720 at h, w = 64, 128), and 2w for the equator ones."""
    from lic360 import ProjectsOp
    from lic360_operator._modules import VIEWPORT_PHIS, VIEWPORT_THETAS
    levels = _preset_levels(levels)
    views = [int(v) for v in views]
    if not views or not all(0 <= v < len(VIEWPORT_THETAS) for v in views):
        raise RuntimeError("viewport_protection: views must be a non-empty list of indices in [0, %d)" % len(VIEWPORT_THETAS))
    if not 0 < fov < 1:
        raise RuntimeError("viewport_protection: fov must lie in (0, 1) (units of pi)")
    device = torch.device('cuda') if device is None else torch.device(device)
    if device.type != 'cuda':
        raise RuntimeError("viewport_protection: the footprint is computed on a CUDA device (got %s)" % device)
    if device.index is None:
        device = torch.device('cuda', torch.cuda.current_device())
    a = fov * math.pi / 2
    reach = max(abs(VIEWPORT_PHIS[v]) for v in views) * math.pi + math.atan(math.sqrt(2) * math.tan(a))  # the corners' latitude
    lat = min(reach, math.pi / 2 - math.pi / h)
    n = max(2 * w, math.ceil(1.25 * math.tan(a) * max(w / (2 * math.pi * math.cos(lat)), h / math.pi)) + 1)
    op = ProjectsOp(n, n, VIEWPORT_THETAS, VIEWPORT_PHIS, fov, False, device.index)
    op.forward(torch.zeros((1, 1, h, w), dtype=torch.float32, device=device))
    top = torch.zeros((len(VIEWPORT_THETAS), 1, n, n), dtype=torch.float32, device=device)
    top[views] = 1
    weight = op.backward(top)[0]
    return (weight > 0).to(torch.int32) * levels


def view_footprint(h, w, thetas, phis, fov, device=None):
    """Exact footprints of V rectilinear views on an h x w ERP grid (lic360_view_footprint): a (V,1,h,w) int32 tensor on `device` (a
    CUDA device, default the current one), 1 where the cell intersects the view's field, 0 elsewhere.  thetas, phis: V view
    directions in units of pi, as MultiProject's (view (0, 0) is its front view 1); fov: one field of view in units of pi for all
    views, or V of them, each in (0, 1).  Cells follow ProjectsOp's grid convention (include/lic360_b200.h); h and w even."""
    th = [float(x) for x in thetas]
    ph = [float(x) for x in phis]
    fovs = [float(x) for x in fov] if isinstance(fov, (list, tuple)) else [float(fov)] * len(th)
    if not th or len(ph) != len(th) or len(fovs) != len(th):
        raise RuntimeError("view_footprint: need V >= 1 thetas, V phis and one or V fovs (got %d, %d, %d)" % (len(th), len(ph), len(fovs)))
    device = torch.device('cuda') if device is None else torch.device(device)
    if device.type != 'cuda':
        raise RuntimeError("view_footprint: the footprint is computed on a CUDA device (got %s)" % device)
    V = len(th)
    out = torch.empty((V, 1, int(h), int(w)), dtype=torch.int32, device=device)
    arr = ctypes.c_float * V
    with torch.cuda.device(out.device):
        check(LIB.lic360_view_footprint(int(h), int(w), V, arr(*th), arr(*ph), arr(*fovs), out.data_ptr(), cstream(out)))
    return out


def view_protection(h, w, thetas, phis, fov, levels, margin=0, device=None):
    """Protection map (1,1,h,w) int32 for encode_to_budget / encode_batch_to_budget at any head orientation: `levels` on the union of
    the views' footprints (view_footprint), dilated by `margin` cells (longitude wraps round the seam, latitude stops at the poles),
    0 elsewhere.  Combine maps with torch.maximum, as viewport_protection's."""
    levels = _preset_levels(levels)
    if isinstance(margin, bool) or not isinstance(margin, int) or margin < 0:
        raise RuntimeError("view_protection: margin must be an int >= 0 (got %r)" % (margin,))
    fp = view_footprint(h, w, thetas, phis, fov, device).amax(dim=0, keepdim=True)
    if margin:
        mw = min(margin, int(w))  # a wider margin wraps onto columns already covered
        wide = torch.nn.functional.pad(fp.float(), (mw, mw, 0, 0), mode='circular')
        fp = torch.nn.functional.max_pool2d(wide, (2 * margin + 1, 2 * mw + 1), stride=1, padding=(margin, 0)).to(torch.int32)
    return fp * levels


def _preset_levels(levels):
    if int(levels) != levels or not 0 <= levels <= 48:
        raise RuntimeError("protection levels must be an integer in [0, 48] (got %r)" % (levels,))
    return int(levels)


def stream_bytes_bound(bits, symbols):
    """Most bytes a stream of `symbols` coded symbols with exact-table total `bits` can take: 8 len <= I + 8 + N/8192 (derived in
    tests/test_rate_estimate.py); the 1e-6 absorbs the rounding of the double total."""
    return int(math.floor((bits + 8 + symbols / 8192.0) / 8 + 1e-6))


def budget_bound(est):
    """bytes both streams of an estimate (a dict of FusedCodec.estimate_batch) can take at most"""
    return stream_bytes_bound(est['imp_bits'], est['imp_symbols']) + stream_bytes_bound(est['code_bits'], est['code_symbols'])


def _stage1_offsets(max_offset):
    """stage 1 of select_budget_offset: 0, 8, 16, ... up to max_offset, and max_offset itself when it is not on that grid"""
    return list(range(0, max_offset + 1, 8)) + ([max_offset] if max_offset % 8 else [])


def _stage2_offsets(stage1, bounds, max_bytes, max_offset):
    """stage 2 of select_budget_offset from the stage-1 bounds: the offsets strictly between the stage-1 offset before the first
    that fits, k1, and k1 (none when k1 is 0); RuntimeError if no stage-1 offset fits"""
    fit = [j for j, k in enumerate(stage1) if bounds[k] <= max_bytes]
    if not fit:
        raise RuntimeError("encode_to_budget: no level offset up to %d fits %d bytes (bound at offset %d: %d bytes)"
                           % (max_offset, max_bytes, max_offset, bounds[max_offset]))
    j = fit[0]
    return list(range(stage1[j - 1] + 1, stage1[j])) if j > 0 and stage1[j] - stage1[j - 1] > 1 else []


def _smallest_fit(bounds, max_bytes):
    return min(k for k, b in bounds.items() if b <= max_bytes)


def select_budget_offset(estimate, max_bytes, max_offset=48, bound=budget_bound):
    """The level offset encode_to_budget codes: `estimate(offsets)` returns one estimate per offset; an offset fits when its bound
    (`bound(estimate)`, budget_bound by default) is at most max_bytes.  Stage 1 evaluates offsets 0, 8, 16, ... up to max_offset, and
    max_offset itself when it is not on that grid; if the smallest that fits, k1, is not 0, stage 2 evaluates the offsets strictly
    between the stage-1 offset before k1 and k1 (the seven offsets k1 - 7 .. k1 - 1 on the grid).  The answer is the smallest
    evaluated offset that fits; the rate is not assumed to fall monotonically with the offset.  Returns (offset, {offset: bound in
    bytes} of every offset evaluated); RuntimeError if no offset of stage 1 fits."""
    bounds = {}

    def run(offsets):
        for k, est in zip(offsets, estimate(offsets)):
            bounds[k] = bound(est)

    stage1 = _stage1_offsets(max_offset)
    run(stage1)
    stage2 = _stage2_offsets(stage1, bounds, max_bytes, max_offset)
    if stage2:
        run(stage2)
    return _smallest_fit(bounds, max_bytes), bounds


def _chunked(estimate, items, max_batch):
    """estimate(items) in calls of at most max_batch items (None: one call), concatenated"""
    step = len(items) if max_batch is None else int(max_batch)
    out = []
    for i in range(0, len(items), max(step, 1)):
        out += estimate(items[i:i + step])
    return out


def select_budget_offsets(estimate, max_bytes, max_offsets, max_batch=None):
    """select_budget_offset of K latents side by side, each with its own budget max_bytes[k] and max_offset max_offsets[k]:
    `estimate(pairs)` returns one estimate per (latent, offset) pair and is called with at most max_batch pairs.  Stage 1 of every
    latent runs first, then stage 2 of every latent that needs one; latent k evaluates exactly the offsets select_budget_offset
    evaluates for it alone, so its result is the same.  Returns [(offset, bounds)] per latent; RuntimeError with
    select_budget_offset's message followed by ' (latent k)' for the lowest latent where no stage-1 offset fits."""
    K = len(max_offsets)
    bounds = [{} for _ in range(K)]

    def run(pairs):
        for (k, t), est in zip(pairs, _chunked(estimate, pairs, max_batch)):
            bounds[k][t] = budget_bound(est)

    stage1 = [_stage1_offsets(m) for m in max_offsets]
    run([(k, t) for k in range(K) for t in stage1[k]])
    stage2 = []
    for k in range(K):
        try:
            stage2 += [(k, t) for t in _stage2_offsets(stage1[k], bounds[k], max_bytes[k], max_offsets[k])]
        except RuntimeError as e:
            raise RuntimeError("%s (latent %d)" % (e, k)) from None
    if stage2:
        run(stage2)
    return [(_smallest_fit(b, m), b) for b, m in zip(bounds, max_bytes)]


def select_shared_offset(estimate, max_bytes, K, max_offset, max_batch=None):
    """One offset for K latents together in max_bytes bytes: select_budget_offset whose bound of an offset t is the sum over the
    latents of budget_bound(estimate of (k, t)), each stream's bound floored on its own.  `estimate(pairs)` as in
    select_budget_offsets, at most max_batch pairs per call.  Returns (offset, {t: summed bound}, {t: [bound of latent k]});
    RuntimeError (select_budget_offset's message) when no offset fits."""
    per = {}

    def estimate_offsets(offsets):
        ests = _chunked(estimate, [(k, t) for t in offsets for k in range(K)], max_batch)
        out = [ests[i * K:(i + 1) * K] for i in range(len(offsets))]
        for t, e in zip(offsets, out):
            per[t] = [budget_bound(x) for x in e]
        return out

    offset, bounds = select_budget_offset(estimate_offsets, max_bytes, max_offset, bound=lambda ests: sum(map(budget_bound, ests)))
    return offset, bounds, per


def select_shared_offsets(estimate, budgets, K, max_offset, max_batch=None):
    """select_shared_offset for R budgets at once, e.g. the rungs of a quality ladder: stage 1 runs once for all budgets, then the
    stage 2 of every budget, with each (latent, offset) pair estimated once in calls of at most max_batch pairs.  Budget r evaluates
    exactly the offsets select_shared_offset evaluates for it alone, and its fit is the smallest over those offsets only (the rate is
    not assumed to fall monotonically with the offset, so an offset another budget evaluated could change the answer).  Returns
    [(offset, {t: summed bound}, {t: [bound of latent k]})] per budget, each equal to select_shared_offset(estimate, budgets[r], K,
    max_offset); RuntimeError with select_budget_offset's message followed by ' (rung r)' for the lowest budget no offset fits."""
    per, summed = {}, {}

    def run(offsets):
        ests = _chunked(estimate, [(k, t) for t in offsets for k in range(K)], max_batch)
        for i, t in enumerate(offsets):
            per[t] = [budget_bound(x) for x in ests[i * K:(i + 1) * K]]
            summed[t] = sum(per[t])

    stage1 = _stage1_offsets(max_offset)
    run(stage1)
    stage2 = []
    for r, b in enumerate(budgets):
        try:
            stage2.append(_stage2_offsets(stage1, summed, b, max_offset))
        except RuntimeError as e:
            raise RuntimeError("%s (rung %d)" % (e, r)) from None
    run(sorted(set(t for s in stage2 for t in s)))
    out = []
    for b, s in zip(budgets, stage2):
        own = {t: summed[t] for t in stage1 + s}
        out.append((_smallest_fit(own, b), own, {t: per[t] for t in own}))
    return out


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

    def _latents(self, K, code, mask, imap_quant):
        """K latents as the native calls read them: code, mask (K,48,H,W) and imap_quant (K,1,H/2,W/2), float32 and contiguous on the
        codec's device (mask None: not checked, returned as None), once torch's stream has produced them."""
        code = self._f32(code, (K, 48, self.H, self.W))
        mask = None if mask is None else self._f32(mask, (K, 48, self.H, self.W))
        imp = self._f32(imap_quant, (K, 1, self.H // 2, self.W // 2))
        torch.cuda.current_stream(self.dev).synchronize()
        return code, mask, imp

    def _stream_bytes(self, sid):
        n = LIB.lic360_codec_stream_size(self._h, sid)
        buf = (ctypes.c_uint8 * max(n, 1))()
        LIB.lic360_codec_stream_copy(self._h, sid, buf, n)
        return bytes(buf[:n])

    def encode(self, code, mask, imap_quant, name=None):
        code, mask, imp = self._latents(1, code, mask, imap_quant)
        check(LIB.lic360_codec_encode(self._h, code.data_ptr(), mask.data_ptr(), imp.data_ptr()))
        return self._stream_bytes(1), self._stream_bytes(0)

    def _batch_stream_bytes(self, k, sid):
        n = LIB.lic360_codec_batch_stream_size(self._h, k, sid)
        if n < 0:
            check(1)
        buf = (ctypes.c_uint8 * max(n, 1))()
        LIB.lic360_codec_batch_stream_copy(self._h, k, sid, buf, n)
        return bytes(buf[:n])

    def encode_batch(self, code, mask, imap_quant):
        """`encode` of K latents in one pass (lic360_codec_encode_batch): code, mask (K,48,H,W), imap_quant (K,1,H/2,W/2).

        Both networks run once at batch K; the host codes the 2K streams on the codec's worker threads, the importance streams while
        the code network still runs.  Returns K pairs (imp_bytes, code_bytes), in the order `encode` returns them; pair k is
        byte-identical to encode() of latent k alone.  A latent encode would refuse raises encode's message followed by
        ' (latent k)', for the first such k."""
        K = int(code.shape[0]) if code.dim() == 4 else -1
        code, mask, imp = self._latents(K, code, mask, imap_quant)
        check(LIB.lic360_codec_encode_batch(self._h, K, code.data_ptr(), mask.data_ptr(), imp.data_ptr()))
        return [(self._batch_stream_bytes(k, 1), self._batch_stream_bytes(k, 0)) for k in range(K)]

    def estimate(self, code, mask, imap_quant):
        """The rate of the latent `encode` would code, without the arithmetic coder: the same networks and integer CDF rows, and for
        every coded symbol its ideal code length 16 - log2(T[s+1] - T[s]) bits (include/lic360_b200.h, lic360_codec_estimate).

        Returns {'code_bits': float, 'imp_bits': float, 'code_map': (1,48,H,W), 'imp_map': (1,1,H/2,W/2)}: the totals of the code and
        importance streams and the bits of every symbol as float32 tensors on the codec's device (0 where mask < 0.5).  The image
        is 8H x 8W pixels, so its rate is (code_bits + imp_bits) / (64 H W) bits per pixel.  For each stream, with N coded symbols
        and I its total, the bytes `encode` writes satisfy -(1 + u + N/8192) <= 8 * len(stream) - I <= 8 + N/8192, where u is the
        number of pending underflow bits the coder drops at the end (a few at most in practice; derivation in
        tests/test_rate_estimate.py).  Raises RuntimeError on the inputs `encode` refuses, with the same message."""
        code, mask, imp = self._latents(1, code, mask, imap_quant)
        code_map = torch.empty((1, 48, self.H, self.W), dtype=torch.float32, device=self.dev)
        imp_map = torch.empty((1, 1, self.H // 2, self.W // 2), dtype=torch.float32, device=self.dev)
        totals = (ctypes.c_double * 2)()
        check(LIB.lic360_codec_estimate(self._h, code.data_ptr(), mask.data_ptr(), imp.data_ptr(), code_map.data_ptr(),
                                        imp_map.data_ptr(), totals))
        return {'code_bits': totals[0], 'imp_bits': totals[1], 'code_map': code_map, 'imp_map': imp_map}

    def estimate_batch(self, code, mask, imap_quant, maps=True):
        """`estimate` of K latents in one pass (lic360_codec_estimate_batch): code, mask (K,48,H,W), imap_quant (K,1,H/2,W/2).

        Returns one dict per latent with estimate()'s keys plus 'code_symbols' and 'imp_symbols', the numbers of coded symbols
        (mask >= 0.5, and every importance position).  Latent k's totals and maps are bit-identical to estimate() of that latent
        alone.  The maps are views into (K,...) tensors, or None with maps=False.  A latent encode would refuse raises encode's
        message followed by ' (latent k)', for the first such k."""
        K = int(code.shape[0]) if code.dim() == 4 else -1
        code, mask, imp = self._latents(K, code, mask, imap_quant)
        code_map = imp_map = None
        if maps:
            code_map = torch.empty((K, 48, self.H, self.W), dtype=torch.float32, device=self.dev)
            imp_map = torch.empty((K, 1, self.H // 2, self.W // 2), dtype=torch.float32, device=self.dev)
        totals = (ctypes.c_double * max(2 * K, 1))()
        counts = (ctypes.c_longlong * max(2 * K, 1))()
        check(LIB.lic360_codec_estimate_batch(self._h, K, code.data_ptr(), mask.data_ptr(), imp.data_ptr(),
                                              None if code_map is None else code_map.data_ptr(),
                                              None if imp_map is None else imp_map.data_ptr(), totals, counts))
        return [{'code_bits': totals[2 * k], 'imp_bits': totals[2 * k + 1], 'code_symbols': counts[2 * k],
                 'imp_symbols': counts[2 * k + 1], 'code_map': None if code_map is None else code_map[k:k + 1],
                 'imp_map': None if imp_map is None else imp_map[k:k + 1]} for k in range(K)]

    def encode_to_budget(self, code, imap_quant, max_bytes, protect=None):
        """Encode the latent in at most max_bytes bytes (both streams) by lowering its importance levels: candidate k codes the
        levels max(s - k, 0) with the mask the decoder derives from them (levels_to_mask), so the result always decodes.  The
        offset comes from select_budget_offset on batched exact-table estimates (two estimate_batch calls, 7 latents each at
        most without protect), where a candidate fits when the proven upper bound of its stream lengths (stream_bytes_bound) is
        at most max_bytes; then one encode of the chosen candidate.

        protect: None, or a (1,1,H/2,W/2) integer map P in [0, 48] on the codec's device (latitude_protection,
        viewport_protection, or their torch.maximum): candidate k then lowers each cell by max(k - P, 0), so a region keeps its
        levels while the others are lowered, and the offsets run up to 48 + max P, where every level is 0.  The streams are
        ordinary streams; decode needs no map.

        Returns {'imp_bytes', 'code_bytes', 'offset', 'levels' (1,1,H/2,W/2), 'mask' (1,48,H,W), 'bound': bytes bound of the
        chosen offset, 'bounds': {offset: bound} of every offset evaluated}.  RuntimeError when no offset fits, and when the
        encoded streams exceed max_bytes (the bound would be broken: never returned silently)."""
        code, _, imp = self._latents(1, code, None, imap_quant)
        max_bytes = int(max_bytes)
        if protect is not None:
            protect = _protect_map(protect, imp)
        max_offset = 48 if protect is None else 48 + int(protect.max())
        cands = {}

        def estimate(offsets):
            levels, masks = levels_to_mask(imp, offsets, protect)
            for j, k in enumerate(offsets):
                cands[k] = (levels[j:j + 1], masks[j:j + 1])
            return self.estimate_batch(code.expand(len(offsets), -1, -1, -1), masks, levels, maps=False)

        offset, bounds = select_budget_offset(estimate, max_bytes, max_offset)
        levels, mask = cands[offset]
        imp_bytes, code_bytes = self.encode(code, mask, levels)
        if len(imp_bytes) + len(code_bytes) > max_bytes:
            raise RuntimeError("encode_to_budget: offset %d encoded to %d bytes, above its bound of %d and the budget of %d bytes"
                               % (offset, len(imp_bytes) + len(code_bytes), bounds[offset], max_bytes))
        return {'imp_bytes': imp_bytes, 'code_bytes': code_bytes, 'offset': offset, 'levels': levels, 'mask': mask,
                'bound': bounds[offset], 'bounds': bounds}

    def _candidates(self, code, imp, protect, pairs):
        """lic360_codec_estimate_candidates on checked inputs: one estimate dict (estimate_batch's keys, no maps) per (latent, offset)"""
        J = len(pairs)
        lat = (ctypes.c_int * max(J, 1))(*[int(k) for k, _ in pairs])
        off = (ctypes.c_int * max(J, 1))(*[int(t) for _, t in pairs])
        totals = (ctypes.c_double * max(2 * J, 1))()
        counts = (ctypes.c_longlong * max(2 * J, 1))()
        check(LIB.lic360_codec_estimate_candidates(self._h, int(code.shape[0]), code.data_ptr(), imp.data_ptr(),
                                                   None if protect is None else protect.data_ptr(), J, lat, off, totals, counts))
        return [{'code_bits': totals[2 * j], 'imp_bits': totals[2 * j + 1], 'code_symbols': counts[2 * j],
                 'imp_symbols': counts[2 * j + 1], 'code_map': None, 'imp_map': None} for j in range(J)]

    def _budget_inputs(self, code, imap_quant, protect):
        K = int(code.shape[0]) if code.dim() == 4 else -1
        code, _, imp = self._latents(K, code, None, imap_quant)
        if protect is not None:
            protect = _protect_map(protect, imp)
        return K, code, imp, protect

    def estimate_candidates(self, code, imap_quant, cand_latent, cand_offset, protect=None):
        """estimate_batch(maps=False) of J rate-control candidates given as (latent, offset) pairs, without materialising them
        (lic360_codec_estimate_candidates): code (K,48,H,W), imap_quant (K,1,H/2,W/2) and protect None or (K,1,H/2,W/2) as in
        levels_to_mask_batch.  Candidate j is latent cand_latent[j] lowered by cand_offset[j]; its dict is bit-identical to
        estimate_batch of the candidate's levels and mask (levels_to_mask) with its latent's code.  A candidate encode would refuse
        raises encode's message followed by ' (candidate j)', for the first such j."""
        K, code, imp, protect = self._budget_inputs(code, imap_quant, protect)
        lat, offs = list(cand_latent), list(cand_offset)
        if len(lat) != len(offs):
            raise RuntimeError("estimate_candidates: %d latents for %d offsets" % (len(lat), len(offs)))
        return self._candidates(code, imp, protect, list(zip(lat, offs)))

    def encode_candidates(self, code, imap_quant, cand_latent, cand_offset, protect=None):
        """encode_batch of J rate-control candidates given as (latent, offset) pairs, without materialising them
        (lic360_codec_encode_candidates): the inputs as in estimate_candidates.  Returns J pairs (imp_bytes, code_bytes); pair j is
        byte-identical to encode_batch of the candidate's levels and mask (levels_to_mask_batch) with its latent's code.  A candidate
        encode would refuse raises encode's message followed by ' (candidate j)', for the first such j."""
        K, code, imp, protect = self._budget_inputs(code, imap_quant, protect)
        lat, offs = [int(k) for k in cand_latent], [int(t) for t in cand_offset]
        if len(lat) != len(offs):
            raise RuntimeError("encode_candidates: %d latents for %d offsets" % (len(lat), len(offs)))
        J = len(lat)
        check(LIB.lic360_codec_encode_candidates(self._h, K, code.data_ptr(), imp.data_ptr(), None if protect is None else protect.data_ptr(),
                                                 J, (ctypes.c_int * max(J, 1))(*lat), (ctypes.c_int * max(J, 1))(*offs)))
        return [(self._batch_stream_bytes(j, 1), self._batch_stream_bytes(j, 0)) for j in range(J)]

    def encode_batch_to_budget(self, code, imap_quant, max_bytes, protect=None, shared=False, max_batch=16):
        """encode_to_budget of K latents, with batched estimates and one encode_batch: code (K,48,H,W), imap_quant (K,1,H/2,W/2),
        protect None or an integer (K,1,H/2,W/2) map per latent (as encode_to_budget's).  Candidates are estimated as (latent,
        offset) pairs (estimate_candidates), at most max_batch per pass: max_batch bounds the encoder buffers, which grow with the
        batch, and does not change the result.

        shared=False: max_bytes is one int for every latent or a list of K.  Stage 1 of every latent runs in as few passes as
        max_batch allows, then stage 2 of every latent that needs one, then one encode_batch of the K chosen candidates
        (select_budget_offsets).  Returns K dicts; dict k equals encode_to_budget(code[k:k+1], imap_quant[k:k+1], max_bytes[k],
        protect[k:k+1]) exactly, streams included.

        shared=True: max_bytes is one int for all 2K streams, and one offset t is applied to every latent, so all are lowered alike.
        t fits when the sum over the latents of budget_bound(estimate of latent k at t) is at most max_bytes (select_shared_offset,
        offsets up to the largest 48 + max P_k).  Returns {'results': K dicts with encode_to_budget's keys, 'bound' and 'bounds'
        being the latent's own, 'offset': t, 'bound': the summed bound at t, 'bounds': {t: summed bound} of every offset
        evaluated}.  K = 1 gives encode_to_budget's offset, bounds and streams.

        RuntimeError, with nothing returned, when no offset fits or the written bytes exceed their budget: encode_to_budget's
        message, followed by ' (latent k)' for the lowest such latent in the per-latent mode."""
        K, code, imp, protect = self._budget_inputs(code, imap_quant, protect)
        if isinstance(max_batch, bool) or not isinstance(max_batch, int) or max_batch < 1:
            raise RuntimeError("encode_batch_to_budget: max_batch must be a positive int (got %r)" % (max_batch,))
        tops = [48] * K if protect is None else [48 + int(m) for m in protect.amax(dim=(1, 2, 3)).tolist()]

        def estimate(pairs):
            return self._candidates(code, imp, protect, pairs)

        if shared:
            if isinstance(max_bytes, (list, tuple)):
                raise RuntimeError("encode_batch_to_budget: shared=True takes one budget for all latents")
            budget = int(max_bytes)
            offset, bounds, per = select_shared_offset(estimate, budget, K, max(tops), max_batch)
            offsets, budgets = [offset] * K, None
        else:
            budgets = [int(b) for b in max_bytes] if isinstance(max_bytes, (list, tuple)) else [int(max_bytes)] * K
            if len(budgets) != K:
                raise RuntimeError("encode_batch_to_budget: %d budgets for %d latents" % (len(budgets), K))
            picks = select_budget_offsets(estimate, budgets, tops, max_batch)
            offsets = [o for o, _ in picks]
        levels, masks = levels_to_mask_batch(imp, range(K), offsets, protect)
        streams = self.encode_batch(code, masks, levels)
        results = []
        for k, (imp_bytes, code_bytes) in enumerate(streams):
            own = {t: per[t][k] for t in bounds} if shared else picks[k][1]
            results.append({'imp_bytes': imp_bytes, 'code_bytes': code_bytes, 'offset': offsets[k], 'levels': levels[k:k + 1],
                            'mask': masks[k:k + 1], 'bound': own[offsets[k]], 'bounds': own})
        if not shared:
            for k, r in enumerate(results):
                size = len(r['imp_bytes']) + len(r['code_bytes'])
                if size > budgets[k]:
                    raise RuntimeError("encode_to_budget: offset %d encoded to %d bytes, above its bound of %d and the budget of %d "
                                       "bytes (latent %d)" % (r['offset'], size, r['bound'], budgets[k], k))
            return results
        size = sum(len(r['imp_bytes']) + len(r['code_bytes']) for r in results)
        if size > budget:
            raise RuntimeError("encode_to_budget: offset %d encoded to %d bytes, above its bound of %d and the budget of %d bytes"
                               % (offset, size, bounds[offset], budget))
        return {'results': results, 'offset': offset, 'bound': bounds[offset], 'bounds': bounds}

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

    def engine_info(self, stream_id=0):
        """The decoder's kernel choices for one stream (0 = code, 1 = importance), fixed at creation (lic360_codec_engine_info)."""
        out = (ctypes.c_int * 13)()
        check(LIB.lic360_codec_engine_info(self._h, stream_id, out, 13))
        return {'chain': ('generic', 'chain4', 'chain1')[out[0]], 'dsm': bool(out[1]), 'cluster': out[2], 'chain_threads': out[3],
                'chain_smem': out[4], 'max_len': out[5], 'c1_lenp': out[6], 'c1_kpc': out[7], 'chain_tasks': out[8],
                'old_positions_per_lane': out[9], 'parts4': out[10], 'parts': out[11], 'tail_rounds': out[12]}

    def last_timing(self):
        out = (ctypes.c_double * 6)()
        LIB.lic360_codec_last_timing(self._h, out, 6)
        return {'total_ms': out[0], 'host_coder_ms': out[1], 'gpu_wait_ms': out[2], 'imp_stream_ms': out[3],
                'gpu_steps_ms': out[4], 'imp_gpu_steps_ms': out[5]}
