"""Operator modules of the context-model entropy path -- constructor/forward signatures, parameter names and shapes
are those of the reference package `lic360_operator` (file:line cited per class), so state dicts
(lic360_demo.py:296-322,348-355) and call sites load unchanged."""
import math

import numpy as np
import torch
from torch import nn

import lic360
from .BaseOpModule import BaseOpModule
from . import _functions as F_


def _ops(ctor, device_list, *args):
    return {gid: ctor(*args, gid) for gid in device_list}


class _PlanModule(BaseOpModule):
    """set_param / restart of the stateful wavefront modules (CconvDc.py:72-78, TileExtract.py:27-33, ...)."""

    def set_param(self, p1, p2):
        for gid in self.op.keys():
            self.op[gid].set_param(p1.to('cuda:{}'.format(gid)), p2)

    def restart(self):
        for gid in self.op.keys():
            self.op[gid].restart()


# ------------------------------------------------------------------------------------------- context convolution
def _conv_params(mod, shape_w, shape_b, act, init):
    mod.weight = nn.Parameter(init(shape_w))
    mod.bias = nn.Parameter(torch.zeros(shape_b) if init is torch.empty else init(shape_b))
    mod.act = act
    mod.relu = nn.Parameter(torch.zeros(shape_b) if init is torch.empty else init(shape_b)) if act else None


class _CconvModule(object):
    _batch = False

    def _setup(self, opcls, ngroup, c_in, c_out, kernel_size, batch, hidden, act, device, time_it):
        constrain = 6 if hidden else 5
        channel, nout = ngroup * c_in, ngroup * c_out
        self.op = {gid: opcls(channel, ngroup, nout, kernel_size, constrain, gid, time_it) for gid in self.device_list}
        if batch is None:  # CconvEc.py:67-70: uninitialised weight, zero bias / slope
            _conv_params(self, (nout, channel, kernel_size, kernel_size), (nout,), act, torch.empty)
        else:              # CconvEc.py:87-90: U[0,1) everything
            _conv_params(self, (batch, nout, channel, kernel_size, kernel_size), (batch, nout), act, torch.rand)

    def forward(self, x):
        sfx = '_batch' if self._batch else ''
        if self.act:
            return F_.ForwardOnly.apply(self.op, 'forward_act' + sfx, 1, x, self.weight, self.bias, self.relu)
        return F_.ForwardOnly.apply(self.op, 'forward' + sfx, 1, x, self.weight, self.bias)


class CconvEc(_CconvModule, BaseOpModule):
    """CconvEc.py:60-76."""

    def __init__(self, ngroup, c_in, c_out, kernel_size, hidden=False, act=True, device=0, time_it=False):
        BaseOpModule.__init__(self, device)
        self._setup(lic360.CconvEcOp, ngroup, c_in, c_out, kernel_size, None, hidden, act, device, time_it)


class CconvEcBatch(_CconvModule, BaseOpModule):
    """CconvEc.py:79-95."""
    _batch = True

    def __init__(self, ngroup, c_in, c_out, kernel_size, batch=3, hidden=False, act=True, device=0, time_it=False):
        BaseOpModule.__init__(self, device)
        self._setup(lic360.CconvEcOp, ngroup, c_in, c_out, kernel_size, batch, hidden, act, device, time_it)


class CconvDc(_CconvModule, _PlanModule):
    """CconvDc.py:58-82."""

    def __init__(self, ngroup, c_in, c_out, kernel_size, hidden=False, act=True, device=0, time_it=False):
        BaseOpModule.__init__(self, device)
        self._setup(lic360.CconvDcOp, ngroup, c_in, c_out, kernel_size, None, hidden, act, device, time_it)


class CconvDcBatch(_CconvModule, _PlanModule):
    """CconvDc.py:85-108."""
    _batch = True

    def __init__(self, ngroup, c_in, c_out, kernel_size, batch=3, hidden=False, act=True, device=0, time_it=False):
        BaseOpModule.__init__(self, device)
        self._setup(lic360.CconvDcOp, ngroup, c_in, c_out, kernel_size, batch, hidden, act, device, time_it)


class MaskConv2(BaseOpModule):
    """MaskConstrain.py:24-38: training form -- mask the weights in place, then a dense cuDNN conv2d."""

    def __init__(self, ngroup, c_in, c_out, kernel_size, hidden=False, device=0, time_it=False):
        super(MaskConv2, self).__init__(device)
        constrain = 6 if hidden else 5
        self.op = {gid: lic360.MaskConstrainOp(constrain, ngroup, gid, time_it) for gid in self.device_list}
        self.weight = nn.Parameter(torch.empty((c_out * ngroup, c_in * ngroup, kernel_size, kernel_size), dtype=torch.float32))
        torch.nn.init.kaiming_normal_(self.weight)
        self.bias = nn.Parameter(torch.zeros(c_out * ngroup, dtype=torch.float32))
        self.pad = kernel_size // 2

    def forward(self, x):
        self.weight.data = F_.MaskConstrainFn.apply(self.weight.data, self.op)
        return nn.functional.conv2d(x, self.weight, self.bias, padding=self.pad)


# ------------------------------------------------------------------------------------------- wavefront plumbing
class CodeContex(BaseOpModule):
    """CodeContex.py:21-29: returns (idx_mat on the GPU, plane_idx on the CPU)."""

    def __init__(self, device=0, time_it=False):
        super(CodeContex, self).__init__(device)
        self.op = {gid: lic360.CodeContexOp(gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.ForwardOnly.apply(self.op, 'forward', 2, x)


class TileExtract(_PlanModule):
    """TileExtract.py:20-37: returns (packed rows, count)."""
    _method = 'forward'

    def __init__(self, ngroup, label, device=0, time_it=False):
        super(TileExtract, self).__init__(device)
        self.op = {gid: lic360.TileExtractOp(ngroup, label, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.ForwardOnly.apply(self.op, self._method, 2, x if x.is_contiguous() else x.contiguous())


class TileExtractBatch(TileExtract):
    """TileExtract.py:52-67."""
    _method = 'forward_batch'


class TileInput(_PlanModule):
    """TileInput.py:21-37."""

    def __init__(self, ngroup, bias=0., scale=1., replicate=1, device=0, time_it=False):
        super(TileInput, self).__init__(device)
        self.op = {gid: lic360.TileInputOp(ngroup, bias, scale, replicate, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.ForwardOnly.apply(self.op, 'forward', 1, x if x.is_contiguous() else x.contiguous())


class TileAdd(_PlanModule):
    """TileAdd.py:19-34: in-place residual add on the slab."""

    def __init__(self, ngroup, device=0, time_it=False):
        super(TileAdd, self).__init__(device)
        self.op = {gid: lic360.TileAddOp(ngroup, gid, time_it) for gid in self.device_list}

    def forward(self, x, y):
        return F_.TileAddFn.apply(x, y, self.op)


# ------------------------------------------------------------------------------------------- CDF tables / entropy loss
class EntropyGmmTable(BaseOpModule):
    """EntropyGmmTable.py:23-32."""

    def __init__(self, nstep, bias, num_gaussian, total_region=65536, beta=1e-6, device=0, time_it=False):
        super(EntropyGmmTable, self).__init__(device)
        self.op = {gid: lic360.EntropyGmmTableOp(nstep, bias, num_gaussian, total_region, beta, gid, time_it)
                   for gid in self.device_list}

    def forward(self, weight, delta, mean, ntop):
        c = lambda t: t if t.is_contiguous() else t.contiguous()
        return F_.ForwardOnly.apply(self.op, 'forward', 1, c(weight), c(delta), c(mean), ntop)


class EntropyBatchGmmTable(EntropyGmmTable):
    """EntropyGmmTable.py:49-57."""

    def forward(self, x, ntop):
        return F_.ForwardOnly.apply(self.op, 'forward_batch', 1, x if x.is_contiguous() else x.contiguous(), ntop)


class EntropyTable(BaseOpModule):
    """EntropyTable.py:20-29."""

    def __init__(self, nstep, totoal_region=65536, device=0, time_it=False):
        super(EntropyTable, self).__init__(device)
        self.op = {gid: lic360.EntropyTableOp(nstep, totoal_region, gid, time_it) for gid in self.device_list}

    def forward(self, x, count):
        return F_.ForwardOnly.apply(self.op, 'forward', 1, x, count)


class EntropyGmm(BaseOpModule):
    """EntropyGmm.py:22-31."""

    def __init__(self, num_gaussian=3, ignore_label=0, device=0, time_it=False):
        super(EntropyGmm, self).__init__(device)
        self.op = {gid: lic360.EntropyGmmOp(num_gaussian, ignore_label, gid, time_it) for gid in self.device_list}

    def forward(self, weight, delta, mean, label):
        return F_.EntropyGmmFn.apply(weight, delta, mean, label, self.op)


class ContextReshape(BaseOpModule):
    """ContextReshape.py:22-29."""

    def __init__(self, ngroup, device=0, time_it=False):
        super(ContextReshape, self).__init__(device)
        self.op = {gid: lic360.ContextReshapeOp(ngroup, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, False, x)


class ContextShift(BaseOpModule):
    """ContextShift.py:22-30."""

    def __init__(self, inv, cpn=1, device=0, time_it=False):
        super(ContextShift, self).__init__(device)
        self.op = {gid: lic360.ContexShiftOp(inv, cpn, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, False, x)


# ------------------------------------------------------------------------------------------- quantisation / importance
class QUANT(BaseOpModule):
    """QUANT.py:31-44."""

    def __init__(self, channel, bin_num, check_iters=100, weight_decay=0.9, ntop=1, top_alpha=0.1, device_id=0,
                 time_flag=False):
        super(QUANT, self).__init__(device_id)
        ta = 1. / (bin_num + 1)
        dev = 'cuda:%d' % self.device_list[0]
        w = torch.full((channel, bin_num), math.log(ta), dtype=torch.float32)
        w[:, 0] = ta
        self.weight = nn.Parameter(w.to(dev))
        self.count = nn.Parameter(torch.zeros((channel, bin_num), dtype=torch.float32).to(dev))
        self.op = {gid: lic360.QuantOp(channel, bin_num, weight_decay, check_iters, ntop, top_alpha, gid, time_flag)
                   for gid in self.device_list}

    def forward(self, x):
        return F_.QuantFn.apply(x, self.weight, self.count, self.op, self.training)


class Dquant(BaseOpModule):
    """Dquant.py:21-31."""

    def __init__(self, channel, bin_num, device=0, time_it=False):
        super(Dquant, self).__init__(device)
        self.weight = nn.Parameter(torch.zeros((channel, bin_num), dtype=torch.float32).to('cuda:%d' % self.device_list[0]))
        self.op = {gid: lic360.DquantOp(channel, bin_num, gid, time_it) for gid in self.device_list}

    def forward(self, x, mask):
        return F_.ForwardOnly.apply(self.op, 'forward', 1, x if x.is_contiguous() else x.contiguous(), mask, self.weight)


class ImpMap(BaseOpModule):
    """ImpMap.py:59-72."""

    def __init__(self, rt, alpha, gamma, levels, scale_constrain=1., scale_weight=1., imp_kernel=0, device=0, ntop=1,
                 time_it=False):
        super(ImpMap, self).__init__(device)
        self.op = {gid: lic360.ImpMapOp(levels, alpha, gamma, rt, scale_constrain, scale_weight, imp_kernel, ntop, gid, time_it)
                   for gid in self.device_list}
        self.level = levels
        self.ntop = ntop

    def forward(self, x, imp):
        return F_.ImpMapFn.apply(x, imp, self.level, self.op, self.ntop)


class Imp2mask(BaseOpModule):
    """Imp2mask.py:19-28."""

    def __init__(self, levels, channels, device=0, time_it=False):
        super(Imp2mask, self).__init__(device)
        self.op = {gid: lic360.Imp2maskOp(levels, channels, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.ForwardOnly.apply(self.op, 'forward', 1, x)


class Scale(BaseOpModule):
    """Scale.py:22-31."""

    def __init__(self, bias, scale, device=0, time_it=False):
        super(Scale, self).__init__(device)
        self.op = {gid: lic360.ScaleOp(bias, scale, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, False, x)


# ------------------------------------------------------------------------------------------- sphere geometry
class SpherePad(BaseOpModule):
    """SpherePad.py:24-33."""

    def __init__(self, pad, device=0, inplace=False, time_it=False):
        super(SpherePad, self).__init__(device)
        self.inplace = bool(inplace)
        self.op = {gid: lic360.SpherePadOp(pad, inplace, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, self.inplace, x)


class SphereTrim(BaseOpModule):
    """SphereTrim.py:24-31: zero the border in place."""

    def __init__(self, pad, device=0, time_it=False):
        super(SphereTrim, self).__init__(device)
        self.op = {gid: lic360.SphereTrimOp(pad, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, True, x)


class SphereCutEdge(BaseOpModule):
    """SphereCutEdge.py:24-33."""

    def __init__(self, pad, device=0, time_it=False):
        super(SphereCutEdge, self).__init__(device)
        self.op = {gid: lic360.SphereCutEdgeOp(pad, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, False, x)


class _ScaleResidualBlock(nn.Module):
    """SphereLatScaleNet.py:25-37."""

    def __init__(self, channels):
        super(_ScaleResidualBlock, self).__init__()
        self.net = nn.Sequential(nn.Conv1d(channels, channels, 3, 1, 1), nn.PReLU(channels),
                                 nn.Conv1d(channels, channels, 3, 1, 1), nn.PReLU(channels))

    def forward(self, x):
        return self.net(x) + x


class SphereLatScaleNet(BaseOpModule):
    """SphereLatScaleNet.py:39-63: per-latitude-band scale predicted by a tiny Conv1d net (which stays in torch)."""

    def __init__(self, npart, device=0, time_it=False):
        super(SphereLatScaleNet, self).__init__(device)
        self.op = {gid: lic360.SphereLatScaleOp(npart, gid, time_it) for gid in self.device_list}
        self.net = nn.Sequential(nn.Conv1d(1, 16, 3, 1, 1), nn.PReLU(16), _ScaleResidualBlock(16),
                                 _ScaleResidualBlock(16), nn.Conv1d(16, 1, 1, 1), nn.Sigmoid())
        self.net._modules['4'].bias.data.fill_(3)
        dev = 'cuda:%d' % self.device_list[0]
        self.net = self.net.to(dev)
        ct = np.fabs(np.cos((0.5 - (np.arange(npart) + 0.5) / npart) * np.pi))
        ct = ct / np.max(ct)
        self.data = nn.Parameter(torch.from_numpy(ct).type(torch.float32).to(dev).view(1, 1, npart), requires_grad=False)

    def forward(self, x):
        weight = self.net(self.data.data)
        return F_.SphereLatScaleFn.apply(x, weight, self.op)


class Dtow(BaseOpModule):
    """Dtow.py:22-32 (SURVEY s8f-1)."""

    def __init__(self, stride=2, d2w=False, device=0, time_it=False):
        super(Dtow, self).__init__(device)
        self.op = {gid: lic360.DtowOp(stride, d2w, gid, time_it) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, False, x)


# the 14 viewport directions of MultiProject (MultiProject.py:24-34), longitude theta and latitude phi in units of pi
VIEWPORT_THETAS = (-0.5, 0, 0.5, 1, -0.5, 0, 0.5, 1, -0.5, 0, 0.5, 1, 0, 0)
VIEWPORT_PHIS = (0, 0, 0, 0, 0.25, 0.25, 0.25, 0.25, -0.25, -0.25, -0.25, -0.25, 0.5, -0.5)


class MultiProject(BaseOpModule):
    """MultiProject.py:24-34 (SURVEY s8f-2): the 14 viewports (theta, phi in units of pi) of an ERP batch, (N,C,H,W) ->
    (14*N, C, h, w) viewport-major; backward scatters the viewport gradients back with the bilinear weights."""

    def __init__(self, h, w, fov=0.6, near=False, device_id=0, time_flag=False):
        super(MultiProject, self).__init__(device_id)
        self.thetas = list(VIEWPORT_THETAS)
        self.phis = list(VIEWPORT_PHIS)
        self.op = {gid: lic360.ProjectsOp(int(h), int(w), self.thetas, self.phis, fov, near, gid, time_flag) for gid in self.device_list}

    def forward(self, x):
        return F_.FwdBwd.apply(self.op, False, x)
