"""Drop-in for the reference's BiFPN (src/YetAnotherEfficientDet.py:154-442) on hand-written sm_100a kernels.

`BiFPN`, `SeparableConvBlock` keep the reference constructor / forward signatures and the exact `state_dict`
names and shapes (SURVEY.md A.4), so reference checkpoints load with strict `load_state_dict`.  `BiFPNStack` is an
`nn.Sequential` of cells (what `YetAnotherEfficientDet.__init__` builds at :639-644) whose forward runs ALL cells
as one op list through `mmd_bifpn_run`: intermediate tensors stay pre-BatchNorm in HBM and are normalised,
resampled, fused and swish-ed while the consuming kernel loads them.

CUDA only; parameters stay fp32 (master copies owned by PyTorch), activations are float32 or bfloat16 NHWC
(`channels_last`).  There is no CPU fallback and no PyTorch-op fallback.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib

_EPOCH_ATTR = "_mmd_stats_epoch"   # per-module count of train-mode forwards (they update running statistics through raw
                                   # pointers, behind PyTorch's version counters); eval plans of the same modules re-fold
                                   # their BatchNorms after one.  A plain attribute: id(module) can be reused after GC.
BN_MOMENTUM = 0.01   # src/YetAnotherEfficientDet.py:176
BN_EPS = 1e-3
_ALIGN = 256
KERNEL_CHANNELS = 112  # EfficientDet-D2 (the kernels' compile-time channel count)


# ------------------------------------------------------------------------------------------------------------
# parameter containers with the reference's module tree (names matter: they are the state_dict contract)
# ------------------------------------------------------------------------------------------------------------
class _ParamOnly(nn.Module):
    def forward(self, *a, **k):
        raise NotImplementedError(
            "%s only holds parameters for the fused sm_100a kernels; call the enclosing BiFPN / SeparableConvBlock"
            % type(self).__name__)


class Conv2dStaticSamePadding(_ParamOnly):
    """Parameter holder mirroring src/YetAnotherEfficientNet.py:27-65 (`.conv` is a plain nn.Conv2d, same init)."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, bias=True, groups=1, dilation=1, **kwargs):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size, stride=stride, bias=bias, groups=groups)


class MaxPool2dStaticSamePadding(_ParamOnly):
    """Stateless placeholder for src/YetAnotherEfficientNet.py:68-104 (the pooling is fused into the node kernels)."""

    def __init__(self, *args, **kwargs):
        super().__init__()


class _Stateless(_ParamOnly):
    pass


class SeparableConvBlock(nn.Module):
    """depthwise 3x3 (no bias) -> pointwise 1x1 (+bias) [-> BatchNorm(momentum .01, eps 1e-3)] [-> swish].
    Signature and state_dict of src/YetAnotherEfficientDet.py:154-192.  Called on its own, the block runs the
    configuration BiFPN uses (out_channels == in_channels, norm=True, activation=False); the other configurations
    (norm=False towers and headers of the detection heads) are parameter holders driven by Regressor / Classifier
    (mm_distillnet_b200/heads.py), as in the reference, where nothing else instantiates them."""

    def __init__(self, in_channels, out_channels=None, norm=True, activation=False, onnx_export=False):
        super(SeparableConvBlock, self).__init__()
        if out_channels is None:
            out_channels = in_channels
        self.depthwise_conv = Conv2dStaticSamePadding(in_channels, in_channels, kernel_size=3, stride=1,
                                                      groups=in_channels, bias=False)
        self.pointwise_conv = Conv2dStaticSamePadding(in_channels, out_channels, kernel_size=1, stride=1)
        self.norm = norm
        if self.norm:
            self.bn = nn.BatchNorm2d(num_features=out_channels, momentum=BN_MOMENTUM, eps=BN_EPS)
        self.activation = activation
        if self.activation:
            self.swish = _Stateless()
        self._runner = _Runner()

    def forward(self, x):
        if not self.norm or self.activation or self.pointwise_conv.conv.out_channels != self.pointwise_conv.conv.in_channels:
            raise NotImplementedError("mm_distillnet_b200.SeparableConvBlock runs on its own in the BiFPN configuration only "
                                      "(out_channels == in_channels, norm=True, activation=False); the norm=False blocks "
                                      "of the detection heads are driven by mm_distillnet_b200.Regressor / Classifier")
        return self._runner.run([self], (x,), self.training, kind="sep")[0]


class BiFPN(nn.Module):
    """One BiFPN cell; signature, attribute names and semantics of src/YetAnotherEfficientDet.py:195-442."""

    def __init__(self, num_channels, conv_channels, first_time=False, epsilon=1e-4, onnx_export=False, attention=True):
        super(BiFPN, self).__init__()
        if num_channels != KERNEL_CHANNELS:   # D0/D1/D3.. (src/YetAnotherEfficientDet.py:611-629): fail at construction
            raise NotImplementedError("mm_distillnet_b200.BiFPN: the sm_100a kernels are built for num_channels=%d "
                                      "(EfficientDet-D2, compound_coef=2), got %d" % (KERNEL_CHANNELS, num_channels))
        self.epsilon = epsilon
        self.num_channels = num_channels
        self.conv_channels = list(conv_channels) if conv_channels is not None else None
        # construction order mirrors the reference so the same torch seed gives the same initial weights
        self.conv6_up = SeparableConvBlock(num_channels, onnx_export=onnx_export)
        self.conv5_up = SeparableConvBlock(num_channels, onnx_export=onnx_export)
        self.conv4_up = SeparableConvBlock(num_channels, onnx_export=onnx_export)
        self.conv3_up = SeparableConvBlock(num_channels, onnx_export=onnx_export)
        self.conv4_down = SeparableConvBlock(num_channels, onnx_export=onnx_export)
        self.conv5_down = SeparableConvBlock(num_channels, onnx_export=onnx_export)
        self.conv6_down = SeparableConvBlock(num_channels, onnx_export=onnx_export)
        self.conv7_down = SeparableConvBlock(num_channels, onnx_export=onnx_export)

        for lvl in (6, 5, 4, 3):
            setattr(self, "p%d_upsample" % lvl, _Stateless())
        for lvl in (4, 5, 6, 7):
            setattr(self, "p%d_downsample" % lvl, MaxPool2dStaticSamePadding(3, 2))
        self.swish = _Stateless()

        self.first_time = first_time
        if self.first_time:
            def proj(cin):
                return nn.Sequential(Conv2dStaticSamePadding(cin, num_channels, 1),
                                     nn.BatchNorm2d(num_channels, momentum=BN_MOMENTUM, eps=BN_EPS))
            self.p5_down_channel = proj(conv_channels[2])
            self.p4_down_channel = proj(conv_channels[1])
            self.p3_down_channel = proj(conv_channels[0])
            self.p5_to_p6 = nn.Sequential(Conv2dStaticSamePadding(conv_channels[2], num_channels, 1),
                                          nn.BatchNorm2d(num_channels, momentum=BN_MOMENTUM, eps=BN_EPS),
                                          MaxPool2dStaticSamePadding(3, 2))
            self.p6_to_p7 = nn.Sequential(MaxPool2dStaticSamePadding(3, 2))
            self.p4_down_channel_2 = proj(conv_channels[1])
            self.p5_down_channel_2 = proj(conv_channels[2])

        for name, n in (("p6_w1", 2), ("p5_w1", 2), ("p4_w1", 2), ("p3_w1", 2),
                        ("p4_w2", 3), ("p5_w2", 3), ("p6_w2", 3), ("p7_w2", 2)):
            setattr(self, name, nn.Parameter(torch.ones(n, dtype=torch.float32), requires_grad=True))
            setattr(self, name + "_relu", _Stateless())
        self.attention = attention
        self._runner = _Runner()

    def forward(self, inputs):
        """(p3, p4, p5) for a first cell, (p3..p7) otherwise -> (p3_out, ..., p7_out), as :289-318."""
        return self._runner.run([self], tuple(inputs), self.training, kind="cells")


class BiFPNStack(nn.Sequential):
    """nn.Sequential(*[BiFPN(...)]) (src/YetAnotherEfficientDet.py:639-644) executed as ONE fused op list."""

    def __init__(self, *cells):
        super().__init__(*cells)
        self._runner = _Runner()

    def fusable(self):
        cells = list(self)
        return len(cells) > 0 and all(isinstance(c, BiFPN) for c in cells) and len({c.training for c in cells}) == 1 and \
            all(not c.first_time for c in cells[1:])

    def forward(self, inputs):
        cells = list(self)
        if not self.fusable():
            for c in cells:
                inputs = c(inputs)
            return inputs
        return self._runner.run(cells, tuple(inputs), cells[0].training, kind="cells")


# ------------------------------------------------------------------------------------------------------------
# graph -> op list
# ------------------------------------------------------------------------------------------------------------
class _Holder:
    def __init__(self, **kw):
        self.__dict__.update(kw)


class _SepView:
    """(separable conv, BatchNorm) pair seen as one SeparableConvBlock: the heads share one conv across the pyramid levels
    and keep one BatchNorm per level (src/YetAnotherEfficientDet.py:455-459); `conv` overrides the pointwise parameters
    (zero-padded header halves)."""

    def __init__(self, sep, bn, conv=None):
        self.depthwise_conv = sep.depthwise_conv
        self.pointwise_conv = sep.pointwise_conv if conv is None else _Holder(conv=conv)
        self.bn = bn


class _IdentityBN:
    """gamma 1, beta 0, running mean 0, running var 1, eps 0: what a header without BatchNorm hands the kernels."""

    def __init__(self, const, Cc):
        self.weight, self.bias = const[0:Cc], const[Cc:2 * Cc]
        self.running_mean, self.running_var = const[Cc:2 * Cc], const[3 * Cc:4 * Cc]
        self.num_batches_tracked = None
        self.eps, self.momentum = 0.0, 0.0


class _Arena:
    def __init__(self):
        self.size = 0

    def alloc(self, nbytes):
        off = self.size
        self.size = (off + nbytes + _ALIGN - 1) // _ALIGN * _ALIGN
        return off


class _Tn:
    """A tensor of the plan.  `bn` is the (base, off) of its deferred-BatchNorm vector or None when final."""
    __slots__ = ("H", "W", "C", "base", "off", "bn", "consumers", "producer", "bn_mod")

    def __init__(self, H, W, Cc, base, off, bn=None, producer=None, bn_mod=None):
        self.H, self.W, self.C, self.base, self.off, self.bn = H, W, Cc, base, off, bn
        self.consumers = []
        self.producer = producer
        self.bn_mod = bn_mod      # nn.BatchNorm2d whose affine applies to this deferred tensor


class _OpN:
    __slots__ = ("kind", "ins", "modes", "conv", "bn", "dw", "fw", "fw_eps", "swish", "out", "save_d", "pidx",
                 "stats", "counter", "du", "slots", "glike", "bwd_counter", "cin", "gref", "packed", "aux", "praw", "tag",
                 "train", "gover", "head", "copy", "gpad", "dxref", "frozen")

    def __init__(self, kind):
        self.kind = kind
        self.ins, self.modes = [], []
        self.conv = self.bn = self.dw = self.fw = None
        self.fw_eps = 0.0
        self.swish = 0
        self.out = None
        self.save_d = None
        self.pidx = [None, None, None]
        self.stats = self.counter = self.du = self.bwd_counter = None
        self.slots = [None, None, None]
        self.glike = None      # BNAPPLY: (base, off) of the gradient of its output
        self.cin = 0
        self.gref = {}
        self.packed = None     # (base, off) of the packed parameter block (bf16 plans)
        self.aux = None        # bf16 plans, nodes with a pooled input: (base, off) of the POOLFUSE pre-pass output
        self.praw = None       # ... and of the raw value at each pooling arg-max (kept for the backward)
        self.tag = None        # (cell index, name) of the 3x3-s2 max-pool this op performs (debug_pool_argmax)
        self.train = None      # per-op override of the plan's mode (head headers: always 0, there is no BatchNorm)
        self.gover = None      # header halves: {"pw": ref, "pb": ref} rows of the zero-padded parameter gradients
        self.head = None       # HEAD_GATHER: (K, tot, off, act)
        self.copy = None       # COPY: (source tensor, destination pointer, floats)
        self.gpad = []         # HEAD_GATHER: (base, off) of the padded gradient of each input
        self.dxref = None      # ACT_FWD: (base, off) of the gradient its backward writes
        self.frozen = False    # NODE / PROJ of a training plan whose BatchNorm is in eval(): running statistics, no update


# fixed base indices
B_FWD, B_PERSIST, B_BWD, B_ZERO, B_EXT = 0, 1, 2, 3, 4


def _null_refs(obj):
    """A zero-initialised ctypes struct has MmdRef.base == 0 (a VALID base); make every reference NULL (base -1)."""
    for name, typ in obj._fields_:
        v = getattr(obj, name)
        if isinstance(v, _lib.Ref):
            v.base = -1
        elif isinstance(v, C.Structure):
            _null_refs(v)
        elif isinstance(v, C.Array) and len(v) and isinstance(v[0], C.Structure):
            for e in v:
                if isinstance(e, _lib.Ref):
                    e.base = -1
                else:
                    _null_refs(e)
    return obj


def _new_op():
    return _null_refs(_lib.Op())


def _new_cons():
    return _null_refs(_lib.Cons())


def _ref(pair):
    if pair is None:
        return _lib.Ref(-1, 0, 0)
    return _lib.Ref(int(pair[0]), 0, int(pair[1]))


def _tensor(t, with_bn=True):
    return _lib.Tensor(_ref((t.base, t.off)), _ref(t.bn if with_bn else None), t.H, t.W, t.C, 0)


def _ptr(t):
    return None if t is None else t.data_ptr()


class _Plan:
    """Op lists + arena layout for one (cells, shapes, dtype, mode) combination.  `frozen`: ids of the nn.BatchNorm2d
    modules that a training plan normalises with their running statistics (layers in eval() inside a train() module)."""

    def __init__(self, mods, kind, in_shapes, dtype, train, need_grad, in_need_grad, frozen=()):
        self.train, self.need_grad = train, need_grad and train
        self.frozen = frozenset(frozen) if train else frozenset()
        self.dtype = dtype
        self.esize = 4 if dtype == torch.float32 else 2
        self.B = in_shapes[0][0]
        self.n_in = len(in_shapes)
        self.in_need_grad = list(in_need_grad)
        self.fwd_arena, self.persist, self.bwd_arena, self.zero_arena = _Arena(), _Arena(), _Arena(), _Arena()
        self.pool_fwd, self.pool_bwd = [], []
        self.ops = []
        self.Cc = None
        self.params = self._collect_params(mods)
        self.mods = list(mods)
        self.state_tensors = [t for m in mods for t in list(m.parameters()) + list(m.buffers())]
        self.grad_off = {}
        self.copies = []     # head plans: zero-padded staging copies of the header parameters (COPY ops)
        grad_pad = {}
        if kind == "head":   # the header's 1x1 conv runs on C-row operands: its gradients are written C rows at a time
            hc = mods[0].header.pointwise_conv.conv
            rows = (hc.out_channels + hc.in_channels - 1) // hc.in_channels * hc.in_channels
            grad_pad = {id(hc.weight): rows * hc.in_channels, id(hc.bias): rows}
        if self.need_grad:   # parameter gradients: ONE flat fp32 buffer in parameter order at the head of the zero arena
            off = 0
            for p in self.params:   # every gradient starts 16-byte aligned (the kernels use 16-byte vector reductions)
                off = (off + 15) // 16 * 16
                self.grad_off[id(p)] = (off, p.numel(), tuple(p.shape))
                off += max(p.numel(), grad_pad.get(id(p), 0)) * 4
            self.grad_floats = off // 4
            self.zero_arena.alloc(off)
        ext = [_Tn(s[2], s[3], s[1], B_EXT + i, 0) for i, s in enumerate(in_shapes)]
        self.ext = ext
        self.n_out = {"cells": 5, "sep": 1, "head": 2}[kind]
        self.B_OUT = B_EXT + self.n_in
        self.B_GOUT = self.B_OUT + self.n_out
        self.B_GIN = self.B_GOUT + self.n_out
        self.B_CONST = self.B_GIN + self.n_in     # head plans: identity-BatchNorm constants
        self.n_bases = self.B_CONST + 1
        self.const = None
        if kind == "head":
            self._head(mods[0], ext)
        else:
            if kind == "sep":
                self.Cc = in_shapes[0][1]
                outs = [self._node(mods[0], [(ext[0], _lib.IN_SAME)], None, 0.0, swish=0)]
            else:
                outs = self._cells(mods, ext)
            self.out_shapes = [(self.B, self.Cc, t.H, t.W) for t in outs]
            self._finish_outputs(outs)
        self.fwd_ops = self._emit_fwd()
        self.bwd_ops = self._emit_bwd() if self.need_grad else None

    # ---- graph construction --------------------------------------------------------------------------------
    def _new_raw(self, H, W, bn_mod, train=None):
        n = self.B * H * W * self.Cc * self.esize
        t = _Tn(H, W, self.Cc, B_FWD, self.fwd_arena.alloc(n), producer=None, bn_mod=bn_mod)
        if self.train if train is None else train:
            t.bn = (B_FWD, self.fwd_arena.alloc(4 * self.Cc * 4))
        return t

    def _packed_storage(self, op):
        """bf16 plans: room for the op's packed parameter block (written by mmd_bifpn_prep)."""
        if self.dtype == torch.bfloat16:
            n = _lib.lib().mmd_packed_bytes(op.kind, op.cin if op.kind == _lib.OP_PROJ_FWD else self.Cc, self.Cc)
            op.packed = (B_PERSIST, self.persist.alloc(n))

    def _train_storage(self, op):
        self._packed_storage(op)
        if self.train if op.train is None else op.train:
            op.stats = (B_PERSIST, self.persist.alloc(_lib.STATS_REPLICAS * 2 * self.Cc * 8))
            op.counter = (B_PERSIST, self.persist.alloc(4))
            op.bwd_counter = (B_PERSIST, self.persist.alloc(4))
        else:
            if self.dtype == torch.bfloat16:
                # eval plans too: the persistent small-level chain keeps its grid-barrier words in the first node's counter
                op.counter = (B_PERSIST, self.persist.alloc(4))
            if self.need_grad:   # a header (no BatchNorm) inside a training plan
                op.bwd_counter = (B_PERSIST, self.persist.alloc(4))

    def _node(self, sep, ins, fw, fw_eps, swish=1, tag=None, train=None):
        op = _OpN(_lib.OP_NODE_FWD)
        op.tag = tag
        op.train = train
        op.ins = [t for t, _ in ins]
        op.modes = [m for _, m in ins]
        op.conv, op.bn, op.dw = sep.pointwise_conv.conv, sep.bn, sep.depthwise_conv.conv
        op.frozen = train is not False and id(sep.bn) in self.frozen
        op.fw, op.fw_eps, op.swish = fw, fw_eps, swish
        H = ins[0][0].H if ins[0][1] == _lib.IN_SAME else None
        W = ins[0][0].W if ins[0][1] == _lib.IN_SAME else None
        if H is None:   # first input is always SAME in BiFPN; keep the general rule explicit
            raise ValueError("the first input of a fusion node must be at the node's resolution")
        for t, m in ins:
            if m == _lib.IN_UP2 and (2 * t.H != H or 2 * t.W != W):
                raise ValueError("BiFPN: upsampled input %dx%d does not match level %dx%d (sizes must halve exactly)"
                                 % (t.H, t.W, H, W))
            if m == _lib.IN_POOL and ((t.H + 1) // 2 != H or (t.W + 1) // 2 != W):
                raise ValueError("BiFPN: pooled input %dx%d does not match level %dx%d" % (t.H, t.W, H, W))
            if m == _lib.IN_SAME and (t.H != H or t.W != W):
                raise ValueError("BiFPN: input %dx%d does not match level %dx%d" % (t.H, t.W, H, W))
        op.out = self._new_raw(H, W, sep.bn, train)
        op.out.producer = op
        self._train_storage(op)
        if self.dtype == torch.bfloat16 and _lib.IN_POOL in op.modes:
            n = self.B * H * W * self.Cc
            op.aux = (B_FWD, self.fwd_arena.alloc(n * self.esize))
            if self.need_grad:
                op.praw = (B_FWD, self.fwd_arena.alloc(n * self.esize))
        if self.need_grad:
            n = self.B * H * W * self.Cc
            op.save_d = (B_FWD, self.fwd_arena.alloc(n * self.esize))
            op.du = _Tn(H, W, self.Cc, B_BWD, self.bwd_arena.alloc(n * self.esize))
            for i, m in enumerate(op.modes):
                if m == _lib.IN_POOL:
                    op.pidx[i] = (B_FWD, self.fwd_arena.alloc(n))
                op.slots[i] = (B_ZERO, self.zero_arena.alloc(2 * self.Cc * 8))
        for i, t in enumerate(op.ins):
            t.consumers.append((op, i))
        self.ops.append(op)
        return op.out

    def _proj(self, seq, x):
        op = _OpN(_lib.OP_PROJ_FWD)
        op.ins, op.modes = [x], [_lib.IN_SAME]
        op.conv, op.bn = seq[0].conv, seq[1]
        op.frozen = id(seq[1]) in self.frozen
        op.cin = x.C
        op.out = self._new_raw(x.H, x.W, seq[1])
        op.out.producer = op
        self._train_storage(op)
        x.consumers.append((op, 0))
        self.ops.append(op)
        return op.out

    def _bnapply(self, src, mode, dst=None, tag=None):
        """dst = [pool](bn(src)); `dst` None allocates an arena tensor (P6/P7 synthesis)."""
        op = _OpN(_lib.OP_BNAPPLY)
        op.tag = tag
        op.ins, op.modes = [src], [mode]
        H, W = (src.H, src.W) if mode == _lib.IN_SAME else ((src.H + 1) // 2, (src.W + 1) // 2)
        n = self.B * H * W * self.Cc
        if dst is None:
            dst = _Tn(H, W, self.Cc, B_FWD, self.fwd_arena.alloc(n * self.esize))
        op.out = dst
        dst.producer = op
        if self.need_grad:
            if mode == _lib.IN_POOL:
                op.pidx[0] = (B_FWD, self.fwd_arena.alloc(n))
            if src.bn is not None:
                op.slots[0] = (B_ZERO, self.zero_arena.alloc(2 * self.Cc * 8))
        src.consumers.append((op, 0))
        self.ops.append(op)
        return dst

    def _cells(self, cells, ext):
        first = cells[0]
        self.Cc = first.num_channels
        S, U, P = _lib.IN_SAME, _lib.IN_UP2, _lib.IN_POOL
        if first.first_time:
            if len(ext) != 3:
                raise ValueError("a first_time BiFPN cell takes (p3, p4, p5), got %d inputs" % len(ext))
            c3, c4, c5 = ext
            for t, cin in zip(ext, first.conv_channels):
                if t.C != cin:
                    raise ValueError("BiFPN first cell: input has %d channels, expected %d" % (t.C, cin))
            p6_in = self._bnapply(self._proj(first.p5_to_p6, c5), P, tag=(0, "p6_in"))   # :324
            p7_in = self._bnapply(p6_in, P, tag=(0, "p7_in"))                            # :325
            p3_in = self._proj(first.p3_down_channel, c3)                     # :327-329
            p4_in = self._proj(first.p4_down_channel, c4)
            p5_in = self._proj(first.p5_down_channel, c5)
            p4_in2 = self._proj(first.p4_down_channel_2, c4)                  # :361-363
            p5_in2 = self._proj(first.p5_down_channel_2, c5)
        else:
            if len(ext) != 5:
                raise ValueError("a BiFPN cell takes (p3, p4, p5, p6, p7), got %d inputs" % len(ext))
            for t in ext:
                if t.C != self.Cc:
                    raise ValueError("BiFPN: input has %d channels, expected %d" % (t.C, self.Cc))
            p3_in, p4_in, p5_in, p6_in, p7_in = ext
            p4_in2, p5_in2 = p4_in, p5_in
        for ci, cell in enumerate(cells):
            if cell.num_channels != self.Cc:
                raise ValueError("all cells of a stack must share num_channels")
            e = cell.epsilon
            fw = (lambda name: getattr(cell, name)) if cell.attention else (lambda name: None)
            p6_up = self._node(cell.conv6_up, [(p6_in, S), (p7_in, U)], fw("p6_w1"), e)            # :338-341
            p5_up = self._node(cell.conv5_up, [(p5_in, S), (p6_up, U)], fw("p5_w1"), e)            # :344-347
            p4_up = self._node(cell.conv4_up, [(p4_in, S), (p5_up, U)], fw("p4_w1"), e)            # :350-353
            p3_out = self._node(cell.conv3_up, [(p3_in, S), (p4_up, U)], fw("p3_w1"), e)           # :356-359
            p4_out = self._node(cell.conv4_down, [(p4_in2, S), (p4_up, S), (p3_out, P)], fw("p4_w2"), e,
                                tag=(ci, "p3_out"))                                                        # :366-370
            p5_out = self._node(cell.conv5_down, [(p5_in2, S), (p5_up, S), (p4_out, P)], fw("p5_w2"), e,
                                tag=(ci, "p4_out"))                                                        # :373-377
            p6_out = self._node(cell.conv6_down, [(p6_in, S), (p6_up, S), (p5_out, P)], fw("p6_w2"), e,
                                tag=(ci, "p5_out"))                                                        # :380-384
            p7_out = self._node(cell.conv7_down, [(p7_in, S), (p6_out, P)], fw("p7_w2"), e,
                                tag=(ci, "p6_out"))                                                        # :387-390
            p3_in, p4_in, p5_in, p6_in, p7_in = p3_out, p4_out, p5_out, p6_out, p7_out
            p4_in2, p5_in2 = p4_in, p5_in
        return [p3_in, p4_in, p5_in, p6_in, p7_in]

    def _head(self, mod, ext):
        """Regressor / Classifier (src/YetAnotherEfficientDet.py:463-487, :508-533).  Per level: num_layers tower layers
        (shared separable conv, per-level BatchNorm, swish) as one-input nodes whose BatchNorm + swish is applied by the
        NEXT op on load; the header (no BatchNorm) as train=0 node ops on the header weights zero-padded to a multiple of
        C output rows (identity BatchNorm constants, so the eval-mode fold is a no-op); HEAD_GATHER places the valid
        channels into the concatenated [B, sum HW * anchors, k] result (sigmoid for the classifier); the `alignment`
        output is swish(bn(last tower layer)) of the LAST level."""
        Cc = self.Cc = mod.in_channels
        S = _lib.IN_SAME
        dev = self.params[0].device
        for t in ext:
            if t.C != Cc:
                raise ValueError("%s: input has %d channels, expected %d" % (type(mod).__name__, t.C, Cc))
        if len(ext) != len(mod.bn_list):
            raise ValueError("%s takes %d pyramid levels, got %d" % (type(mod).__name__, len(mod.bn_list), len(ext)))
        hc = mod.header.pointwise_conv.conv
        K = hc.out_channels
        n_half = (K + Cc - 1) // Cc
        rows = n_half * Cc
        one, zero = torch.ones(Cc, device=dev), torch.zeros(Cc, device=dev)
        self.const = torch.cat([one, zero, zero, one]).contiguous()     # scale | shift | mean | invstd of "no BatchNorm"
        ident = _IdentityBN(self.const, Cc)
        self.padw = torch.zeros(rows * Cc + rows, dtype=torch.float32, device=dev)
        for src, off, n in ((hc.weight, 0, K * Cc), (hc.bias, rows * Cc, K)):
            cp = _OpN(_lib.OP_COPY)
            cp.copy = (src, self.padw.data_ptr() + 4 * off, n)
            self.ops.append(cp)
            self.copies.append(cp)
        tot = sum(t.H * t.W for t in ext)
        res = _Tn(1, tot, K, self.B_OUT, 0)
        pos = 0
        for lvl, x in enumerate(ext):
            t = x
            for i in range(mod.num_layers):                                            # :467-470 / :511-514
                t = self._node(_SepView(mod.conv_list[i], mod.bn_list[lvl][i]), [(t, S)], None, 0.0, swish=0 if i == 0 else 1)
            ga = _OpN(_lib.OP_HEAD_GATHER)
            for j in range(n_half):                                                    # :473 / :517
                conv = _Holder(weight=self.padw[j * Cc * Cc:(j + 1) * Cc * Cc], bias=self.padw[rows * Cc + j * Cc: rows * Cc + (j + 1) * Cc])
                h = self._node(_SepView(mod.header, ident, conv), [(t, S)], None, 0.0, swish=1 if mod.num_layers > 0 else 0, train=False)
                hop = self.ops[-1]
                if self.need_grad:
                    goff = self.grad_off[id(hc.weight)][0], self.grad_off[id(hc.bias)][0]
                    hop.gover = {"pw": (B_ZERO, goff[0] + 4 * j * Cc * Cc), "pb": (B_ZERO, goff[1] + 4 * j * Cc)}
                    ga.gpad.append((B_BWD, self.bwd_arena.alloc(self.B * x.H * x.W * Cc * self.esize)))
                    ga.slots[j] = (B_ZERO, self.zero_arena.alloc(2 * Cc * 8))        # stays zero: no statistics flow back
                ga.ins.append(h)
                ga.modes.append(S)
                h.consumers.append((ga, j))
            ga.head = (K, tot, pos, 1 if mod.sigmoid_output else 0)
            ga.out = res
            self.ops.append(ga)
            pos += x.H * x.W
        # alignment[-1] (:472/:487, :515/:533): the activated last tower layer of the last level
        if mod.num_layers == 0:
            raise NotImplementedError("detection heads with num_layers == 0")
        v = self._bnapply(t, S) if self.train else t
        if self.train and self.need_grad:
            self.ops[-1].glike = (B_BWD, self.bwd_arena.alloc(self.B * t.H * t.W * Cc * self.esize))
        act = _OpN(_lib.OP_ACT_FWD)
        act.ins, act.modes = [v], [S]
        act.out = _Tn(t.H, t.W, Cc, self.B_OUT + 1, 0)
        if self.train and self.need_grad:
            act.dxref = self.ops[-1].glike
        self.ops.append(act)
        A = mod.num_anchors
        self.out_shapes = [(self.B, tot * A, K // A), (self.B, Cc, t.H, t.W)]
        self.out_ops = []

    def _finish_outputs(self, outs):
        """Train: the raw outputs are normalised into the user-visible tensors.  Eval: the producing kernels write
        the user-visible tensors directly (BatchNorm is folded into the 1x1 conv)."""
        self.out_ops = []
        for k, t in enumerate(outs):
            dst_base = self.B_OUT + k
            if self.train:
                dst = _Tn(t.H, t.W, self.Cc, dst_base, 0)
                self._bnapply(t, _lib.IN_SAME, dst)
                op = self.ops[-1]
                op.glike = (self.B_GOUT + k, 0)
                self.out_ops.append(op)
            else:
                t.base, t.off = dst_base, 0

    def _collect_params(self, mods):
        ps = []
        for m in mods:
            ps.extend(p for p in m.parameters())
        return ps

    # ---- emission ------------------------------------------------------------------------------------------
    def _fill_common(self, o, op):
        o.n_in = len(op.ins)
        for i, t in enumerate(op.ins):
            o.inp[i] = _tensor(t)
            o.mode[i] = op.modes[i]
            if t.bn is not None and t.bn_mod is not None:
                o.in_bn_w[i] = _ptr(t.bn_mod.weight)
                o.in_bn_b[i] = _ptr(t.bn_mod.bias)
        o.swish = op.swish
        o.fw = _ptr(op.fw)
        o.fw_eps = op.fw_eps
        if op.conv is not None:
            o.pw_w, o.pw_b = _ptr(op.conv.weight), _ptr(op.conv.bias)
            o.bn_w, o.bn_b = _ptr(op.bn.weight), _ptr(op.bn.bias)
            o.bn_rm, o.bn_rv = _ptr(op.bn.running_mean), _ptr(op.bn.running_var)
            o.bn_nbt = _ptr(op.bn.num_batches_tracked)
            o.bn_eps, o.bn_momentum = op.bn.eps, (op.bn.momentum if op.bn.momentum is not None else 0.1)
        if op.dw is not None:
            o.dw_w = _ptr(op.dw.weight)
        o.Cin = op.cin
        o.out = _tensor(op.out)
        o.save_d = _ref(op.save_d)
        o.packed = _ref(op.packed)
        o.frozen_bn = 1 if op.frozen else 0
        for i in range(3):
            o.pidx[i] = _ref(op.pidx[i])
            o.in_slot[i] = _ref(op.slots[i])

    def _emit_fwd(self):
        out = []
        for op in self.ops:
            o = _new_op()
            o.kind = op.kind
            if op.kind == _lib.OP_COPY:
                o.copy_src, o.copy_dst, o.copy_n = op.copy[0].data_ptr(), op.copy[1], op.copy[2]
                out.append(o)
                continue
            o.train = 1 if (self.train if op.train is None else op.train) else 0
            self._fill_common(o, op)
            if op.head is not None:
                o.head_K, o.head_tot, o.head_off, o.head_act = op.head
            o.stats, o.counter = _ref(op.stats), _ref(op.counter)
            if op.aux is not None:
                out.append(self._split_pooled(o, op))
            out.append(o)
        arr = (_lib.Op * len(out))()
        for i, o in enumerate(out):
            arr[i] = o
        self._fwd_keep = out
        return arr

    def _split_pooled(self, o, op):
        """bf16 plans: a node with a pooled input runs as POOLFUSE (pooled input [+ the other non-first input] -> one
        pre-weighted operand `aux`) followed by the node kernel on (input 0, aux).  Rewrites `o` in place and returns the
        POOLFUSE op."""
        n = len(op.ins)
        pi = op.modes.index(_lib.IN_POOL)
        rest = [i for i in range(1, n) if i != pi]
        if pi == 0 or len(rest) > 1 or any(op.modes[i] != _lib.IN_SAME for i in rest):
            raise RuntimeError("internal: unsupported pooled node layout")
        pf = _new_op()
        pf.kind = _lib.OP_POOLFUSE
        pf.train = o.train
        srcs = [pi] + rest
        pf.n_in = len(srcs)
        for k, i in enumerate(srcs):
            pf.inp[k] = _tensor(op.ins[i])
            pf.mode[k] = op.modes[i]
            pf.fw_idx[k] = i
        pf.fw, pf.fw_eps, pf.fw_n = _ptr(op.fw), op.fw_eps, n
        aux = _lib.Tensor(_ref(op.aux), _ref(None), op.out.H, op.out.W, self.Cc, 0)
        pf.out = aux
        pf.pidx[0] = _ref(op.pidx[pi])
        pf.save_d = _ref(op.praw)
        # the node itself: (input 0, aux)
        o.n_in = 2
        o.inp[1] = aux
        o.mode[1] = _lib.IN_SAME
        o.inp[2] = _lib.Tensor(_ref(None), _ref(None), 0, 0, 0, 0)
        o.mode[2] = 0
        o.fw_n = n
        o.fw_idx[0], o.fw_idx[1], o.fw_idx[2] = 0, -1, -1
        for i in range(3):
            o.pidx[i] = _ref(None)
        return pf

    def _cons_of(self, t):
        """MmdCons entries for every consumer edge of tensor `t`."""
        res = []
        for cop, idx in t.consumers:
            c = _new_cons()
            mode = cop.modes[idx]
            if cop.kind == _lib.OP_NODE_FWD:
                c.du = _tensor(cop.du, with_bn=False)
                c.fw, c.fw_k, c.fw_n, c.fw_eps = _ptr(cop.fw), idx, len(cop.ins), cop.fw_eps
            elif cop.kind == _lib.OP_BNAPPLY:
                if cop.glike is None:
                    raise RuntimeError("internal: BNAPPLY consumer without a gradient tensor")
                c.du = _lib.Tensor(_ref(cop.glike), _ref(None), cop.out.H, cop.out.W, self.Cc, 0)
                c.fw = None
            elif cop.kind == _lib.OP_HEAD_GATHER:   # the zero-padded gradient HEAD_SCATTER wrote for this half
                c.du = _lib.Tensor(_ref(cop.gpad[idx]), _ref(None), t.H, t.W, self.Cc, 0)
                c.fw = None
            else:
                raise RuntimeError("internal: unexpected consumer kind")
            c.mode = {_lib.IN_SAME: _lib.CONS_SAME, _lib.IN_UP2: _lib.CONS_UP2, _lib.IN_POOL: _lib.CONS_POOL}[mode]
            c.slot = _ref(cop.slots[idx])
            c.pidx = _ref(cop.pidx[idx])
            res.append(c)
        if len(res) > 3:
            raise RuntimeError("internal: a tensor has %d consumers (max 3)" % len(res))
        return res

    def _galloc(self, param):
        return (B_ZERO, self.grad_off[id(param)][0])

    def _emit_bwd(self):
        max_n = max(self.B * op.out.H * op.out.W * self.Cc for op in self.ops if op.kind == _lib.OP_NODE_FWD)
        gout0 = (self.B_GOUT, 0)
        dd = (B_BWD, self.bwd_arena.alloc(max_n * self.esize))
        out = []
        ext_written = set()

        def new(kind, op):
            o = _new_op()
            o.kind = kind
            o.train = 1
            self._fill_common(o, op)
            o.counter = _ref(op.bwd_counter)
            return o

        def set_cons(o, t):
            cons = self._cons_of(t)
            o.n_cons = len(cons)
            for i, c in enumerate(cons):
                o.cons[i] = c

        for op in reversed(self.ops):
            if op.kind == _lib.OP_ACT_FWD:          # g(bn(x)) = g(alignment) * swish'(bn(x))
                o = new(_lib.OP_ACT_BWD, op)
                o.n_cons = 1
                c = _new_cons()
                c.du = _lib.Tensor(_ref((self.B_GOUT + 1, 0)), _ref(None), op.out.H, op.out.W, self.Cc, 0)
                o.cons[0] = c
                o.dx = _ref(op.dxref)
                out.append(o)
            elif op.kind == _lib.OP_HEAD_GATHER:
                o = new(_lib.OP_HEAD_SCATTER, op)
                o.head_K, o.head_tot, o.head_off, o.head_act = op.head
                o.n_cons = 1
                c = _new_cons()
                c.du = _lib.Tensor(_ref(gout0), _ref(None), 1, op.head[1], op.head[0], 0)
                o.cons[0] = c
                o.du = _ref(op.gpad[0])
                o.dd = _ref(op.gpad[1] if len(op.gpad) > 1 else None)
                out.append(o)
            elif op.kind == _lib.OP_BNAPPLY:
                src = op.ins[0]
                if op.glike is None:   # internal materialisation (P6 / P7 synthesis): gather its gradient first
                    n = self.B * op.out.H * op.out.W * self.Cc
                    op.glike = (B_BWD, self.bwd_arena.alloc(n * self.esize))
                    o = new(_lib.OP_PULL, op)
                    set_cons(o, op.out)
                    o.dx = _ref(op.glike)
                    out.append(o)
                if src.bn is not None:
                    o = new(_lib.OP_SLOT, op)
                    o.n_cons = 1
                    c = _new_cons()
                    c.du = _lib.Tensor(_ref(op.glike), _ref(None), op.out.H, op.out.W, self.Cc, 0)
                    o.cons[0] = c
                    out.append(o)
            elif op.kind == _lib.OP_NODE_FWD:
                o = new(_lib.OP_NODE_BWD, op)
                set_cons(o, op.out)
                o.aux, o.praw = _ref(op.aux), _ref(op.praw)
                o.du = _ref((op.du.base, op.du.off))
                o.dd = _ref(dd)
                o.g_dw = _ref(self._galloc(op.dw.weight))
                if op.gover is not None:   # a header half: no BatchNorm (identity constants), zero-padded weight rows
                    o.out = _lib.Tensor(_ref((op.out.base, op.out.off)), _ref((self.B_CONST, 0)), op.out.H, op.out.W, self.Cc, 0)
                    o.g_pw, o.g_pb = _ref(op.gover["pw"]), _ref(op.gover["pb"])
                    out.append(o)
                    continue
                o.g_pw = _ref(self._galloc(op.conv.weight))
                o.g_pb = _ref(self._galloc(op.conv.bias))
                o.g_bn_w = _ref(self._galloc(op.bn.weight))
                o.g_bn_b = _ref(self._galloc(op.bn.bias))
                if op.fw is not None:
                    o.g_fw = _ref(self._galloc(op.fw))
                out.append(o)
            elif op.kind == _lib.OP_PROJ_FWD:
                o = new(_lib.OP_PROJ_BWD, op)
                set_cons(o, op.out)
                x = op.ins[0]
                xi = x.base - B_EXT
                if self.in_need_grad[xi]:
                    o.dx = _ref((self.B_GIN + xi, 0))
                    o.accumulate_dx = 1 if xi in ext_written else 0
                    ext_written.add(xi)
                o.g_pw = _ref(self._galloc(op.conv.weight))
                o.g_pb = _ref(self._galloc(op.conv.bias))
                o.g_bn_w = _ref(self._galloc(op.bn.weight))
                o.g_bn_b = _ref(self._galloc(op.bn.bias))
                out.append(o)
        # gradients of external pyramid inputs consumed directly by nodes (non-first cells, bare SeparableConvBlock)
        for xi, x in enumerate(self.ext):
            if not self.in_need_grad[xi] or xi in ext_written:
                continue
            if not x.consumers or any(cop.kind == _lib.OP_PROJ_FWD for cop, _ in x.consumers):
                continue
            o = _new_op()
            o.kind = _lib.OP_PULL
            o.train = 1
            o.out = _tensor(x)
            set_cons(o, x)
            o.dx = _ref((self.B_GIN + xi, 0))
            out.append(o)
        arr = (_lib.Op * len(out))()
        for i, o in enumerate(out):
            arr[i] = o
        self._bwd_keep = out
        return arr


def debug_pool_argmax(output):
    """TEST HOOK.  `output`: any tensor returned by a train-mode forward under grad whose backward has not run yet.
    Returns one dict per cell: the window index (uint8 [B,C,Ho,Wo]; 0..8 row-major inside the 3x3 window, 9 = the zero
    padding won) that the forward recorded for every 3x3-s2 max-pool — keyed "p3_out".."p6_out" by the pooled tensor of
    the bottom-up path, "p6_in" / "p7_in" for the first cell's P6 / P7 synthesis.  The parity tests hand these to the
    oracle (oracle.maxpool_same(hint=...)) so that both sides route the pooling gradients through the same elements."""
    fn = output.grad_fn
    plan, saved = getattr(fn, "plan", None), getattr(fn, "saved", None)
    if plan is None or saved is None or not plan.need_grad:
        raise RuntimeError("debug_pool_argmax needs an output of a train-mode forward that recorded a backward")
    arena = saved[1]
    res = {}
    for op in plan.ops:
        if op.tag is None:
            continue
        for ref in op.pidx:
            if ref is None:
                continue
            H, W = op.out.H, op.out.W
            n = plan.B * H * W * plan.Cc
            res.setdefault(op.tag[0], {})[op.tag[1]] = \
                arena.buf[ref[1]: ref[1] + n].view(plan.B, H, W, plan.Cc).permute(0, 3, 1, 2).contiguous().cpu()
    return [res.get(i, {}) for i in range(max(res) + 1 if res else 0)]


def mark_state_changed(modules):
    """Tell the plan caches that parameters / running statistics of these BiFPN cells (or head modules) were changed behind
    PyTorch's back — by a CUDA-graph replay of a training step, whose host-side bookkeeping does not run, or by an
    optimizer kernel writing through raw pointers: eval-mode plans re-fold their packed parameter blocks on next use."""
    for m in modules:
        object.__setattr__(m, _EPOCH_ATTR, getattr(m, _EPOCH_ATTR, 0) + 1)


def forward_multi(items):
    """items = [(BiFPNStack, inputs), ...] (<= 4 fusable stacks sharing batch size and dtype, e.g. the student and its
    three frozen teachers): all forwards are enqueued by ONE mmd_bifpn_run_multi call on the current stream, so that
    nodes of the same pyramid level share a launch.  Returns the per-stack output tuples; a train-mode stack under grad
    mode gets its usual autograd node (the backward is unchanged)."""
    return _forward_multi([(stack, list(stack), tuple(inputs), "cells") for stack, inputs in items])


def forward_multi_heads(items):
    """items = [(Regressor | Classifier, the 5 pyramid tensors), ...] — <= 4 heads of ONE type on the same pyramid geometry,
    e.g. the student's regressor (train) and its three frozen teachers' (eval): like forward_multi(), ONE
    mmd_bifpn_run_multi call, the tower / header nodes of the same level share a launch (blockIdx.y = network), which fills
    the small levels (a P7 tower layer of one network is 32 tiles at B = 32).  Returns [(predictions, alignment), ...]."""
    return _forward_multi([(head, [head], tuple(inputs), "head") for head, inputs in items])


def _forward_multi(specs):
    L = _lib.lib()
    prepared = []
    for owner, mods, inputs, kind in specs:
        plan, params, need_grad = owner._runner._plan_for(mods, inputs, mods[0].training, kind)
        with torch.no_grad():
            bases, outs, saved = owner._runner._forward_prepare(plan, inputs)
        prepared.append((owner, inputs, plan, bases, outs, saved, mods, kind))
    p0 = prepared[0][2]
    if any(p[2].B != p0.B or p[2].dtype != p0.dtype or p[2].device != p0.device for p in prepared):
        raise ValueError("forward_multi: stacks must share batch size, dtype and device")
    n = len(prepared)
    ops = (C.POINTER(_lib.Op) * n)(*[C.cast(p[2].fwd_ops, C.POINTER(_lib.Op)) for p in prepared])
    n_ops = (C.c_int32 * n)(*[len(p[2].fwd_ops) for p in prepared])
    base_arrs = [(C.c_void_p * len(p[3]))(*p[3]) for p in prepared]
    bases = (C.POINTER(C.c_void_p) * n)(*[C.cast(a, C.POINTER(C.c_void_p)) for a in base_arrs])
    n_bases = (C.c_int32 * n)(*[len(p[3]) for p in prepared])
    with torch.cuda.device(p0.device):
        stream = torch.cuda.current_stream().cuda_stream
        rc = L.mmd_bifpn_run_multi(ops, n_ops, bases, n_bases, n, p0.B, p0.Cc,
                                   _lib.MMD_F32 if p0.dtype == torch.float32 else _lib.MMD_BF16, stream)
    _lib.check(rc, "mmd_bifpn_run_multi")
    results = []
    for owner, inputs, plan, _, outs, saved, mods, kind in prepared:
        results.append(owner._runner.run(mods, inputs, mods[0].training, kind, pre=(outs, saved)))
    return results


class _Lease:
    """A pooled device buffer.  It goes back to its plan's pool on release() — called as soon as the work that needs it
    has been enqueued (stream order protects the contents) — or, as a safety net, when the last reference goes away
    (a forward whose backward never runs).  Steady-state steps therefore never touch the CUDA allocator."""
    __slots__ = ("buf", "pool")

    def __init__(self, pool, nbytes, device):
        self.pool = pool
        self.buf = pool.pop() if pool else torch.empty(max(nbytes, _ALIGN), dtype=torch.uint8, device=device)

    def data_ptr(self):
        if self.buf is None:
            raise RuntimeError("mm_distillnet_b200.BiFPN: this forward's workspace was already released (backward twice?)")
        return self.buf.data_ptr()

    def release(self):
        buf, self.buf = self.buf, None
        if buf is not None and len(self.pool) < 4:
            self.pool.append(buf)

    def __del__(self):
        try:
            self.release()
        except Exception:  # interpreter shutdown
            pass


class _StackFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, runner, plan, n_in, pre, *tensors):
        """tensors = inputs + parameters, or (flat-gradient mode) inputs + one fresh anchor leaf: the parameter
        gradients then reach `.grad` through the runner's sink, and the autograd graph has no edge to the parameters'
        (possibly stale, created-on-another-stream) AccumulateGrad nodes, which keeps the backward CUDA-graph capturable."""
        inputs, params = tensors[:n_in], tensors[n_in:]
        outs, saved = pre if pre is not None else runner._forward(plan, inputs)
        ctx.runner, ctx.plan, ctx.saved, ctx.n_in = runner, plan, saved, n_in
        ctx.sink_mode = runner.grad_sink is not None
        ctx.param_list = plan.params if ctx.sink_mode else params
        ctx.n_extra = len(params)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        plan = ctx.plan
        if not plan.need_grad:
            raise RuntimeError("mm_distillnet_b200.BiFPN: backward through an eval-mode (folded BatchNorm) forward is "
                               "not supported; call .train() on the student")
        gin, gflat = ctx.runner._backward(plan, ctx.saved, gouts)
        ctx.saved[1].release()   # the forward arena: every kernel that reads it is enqueued
        grads = [None, None, None, None]
        for i in range(ctx.n_in):
            grads.append(gin[i] if ctx.needs_input_grad[4 + i] else None)
        if ctx.sink_mode:
            # flat-gradient mode (DistillStep): hand over the one contiguous fp32 buffer holding every parameter
            # gradient and make each .grad a view of it, instead of ~360 per-parameter AccumulateGrad kernels
            flat = gflat[:plan.grad_floats]
            for p in ctx.param_list:
                if p.requires_grad:
                    off, n, shape = plan.grad_off[id(p)]
                    p.grad = flat[off // 4: off // 4 + n].view(shape)
            if ctx.runner.grad_sink is not None:
                ctx.runner.grad_sink(flat)
            grads.extend([None] * ctx.n_extra)
            return tuple(grads)
        for j, p in enumerate(ctx.param_list):
            ent = plan.grad_off.get(id(plan.params[j]))
            if ent is None or not ctx.needs_input_grad[4 + ctx.n_in + j]:
                grads.append(None)
            else:
                off, n, shape = ent
                grads.append(gflat[off // 4: off // 4 + n].view(shape))
        return tuple(grads)


class _Runner:
    """Builds / caches plans and runs them through the C ABI."""

    def __init__(self):
        self.plans = {}
        self._param_cache = None
        self.grad_sink = None   # callable(flat_fp32_grad) -> None; see DistillStep

    # Plans hold ctypes op lists full of raw device pointers: they are a cache, never state.  copy.deepcopy(module),
    # torch.save(module) and spawn-based workers therefore get a fresh, empty runner (plans are rebuilt on first use).
    def __getstate__(self):
        return {}

    def __setstate__(self, state):
        self.__init__()

    def __deepcopy__(self, memo):
        return _Runner()

    def _plan_for(self, mods, inputs, training, kind):
        if len(inputs) == 0:
            raise ValueError("BiFPN: empty input tuple")
        x0 = inputs[0]
        if not x0.is_cuda:
            raise RuntimeError("mm_distillnet_b200.BiFPN needs CUDA tensors (there is no CPU fallback)")
        if x0.dtype not in (torch.float32, torch.bfloat16):
            raise TypeError("BiFPN activations must be float32 or bfloat16, got %s" % x0.dtype)
        for x in inputs:
            if x.dim() != 4 or x.shape[0] != x0.shape[0] or x.dtype != x0.dtype or x.device != x0.device:
                raise ValueError("BiFPN: inputs must be [B,C,H,W] tensors sharing batch, dtype and device")
        ck = tuple(id(m) for m in mods)
        if self._param_cache is None or self._param_cache[0] != ck:   # walking 5 cells' modules costs ~1 ms per call
            self._param_cache = (ck, [p for m in mods for p in m.parameters()], [b for m in mods for b in m.buffers()],
                                 [b for m in mods for b in m.modules() if isinstance(b, nn.BatchNorm2d)])
        params, buffers, bns = self._param_cache[1], self._param_cache[2], self._param_cache[3]
        if len(params) == 0:
            raise RuntimeError("mm_distillnet_b200.BiFPN: the module holds no parameters (an nn.DataParallel replica?); "
                               "multi-GPU runs use one process per GPU, see mm_distillnet_b200.DistillStep")
        if any(p.dtype != torch.float32 for p in params):
            raise TypeError("BiFPN parameters must stay float32 (master weights); cast activations, not the module")
        if any(p.device != x0.device for p in params):
            raise RuntimeError("BiFPN: parameters and inputs live on different devices")
        grad_on = torch.is_grad_enabled()
        in_need = [grad_on and x.requires_grad for x in inputs]
        wants_grad = grad_on and (any(in_need) or any(p.requires_grad for p in params))
        if wants_grad and not training:
            # the eval-mode kernels fold the running statistics into the 1x1 weights and keep nothing for a backward;
            # returning detached outputs would silently drop the gradients (reference BiFPN is differentiable in eval mode)
            raise NotImplementedError(
                "mm_distillnet_b200.BiFPN: backward through an eval-mode (folded BatchNorm) forward is not supported; "
                "call .train() on the student, or run frozen / validation forwards under torch.no_grad() "
                "(teachers: train_methods.py:321, validate: :1132-1142)")
        need_grad = training and wants_grad
        Cc = mods[0].num_channels if kind == "cells" else inputs[0].shape[1]
        if Cc != KERNEL_CHANNELS:
            raise NotImplementedError("the sm_100a BiFPN kernels are built for %d channels (EfficientDet-D2), got %d"
                                      % (KERNEL_CHANNELS, Cc))
        if training and x0.shape[0] * min(x.shape[2] * x.shape[3] for x in inputs) < 1:
            raise ValueError("empty batch")
        # the op lists hold the raw data_ptr() of EVERY parameter and BatchNorm buffer: all of them are part of the key
        # (load_state_dict(assign=True), an EMA swap through p.data or a reassigned buffer must miss the cache)
        ptrs = hash(tuple(t.data_ptr() for t in params) + tuple(t.data_ptr() for t in buffers))
        # training plans follow each BatchNorm layer's own mode: a layer in eval() (frozen BatchNorm) normalises with its
        # running statistics and leaves them alone.  The per-layer mask is part of the key, so a mode change between two
        # calls builds or reuses the matching plan (eval plans fold every BatchNorm whatever its flag says)
        mask = tuple(m.training for m in bns) if training else ()
        key = (kind, tuple(tuple(x.shape) for x in inputs), x0.dtype, bool(training), need_grad, tuple(in_need),
               x0.device.index, len(params), ptrs, mask)
        plan = self.plans.get(key)
        if plan is None:
            frozen = [id(m) for m, on in zip(bns, mask) if not on]
            plan = _Plan(mods, kind, [tuple(x.shape) for x in inputs], x0.dtype, bool(training), need_grad, in_need, frozen)
            plan.device = x0.device
            self.plans[key] = plan
            if len(self.plans) > 16:
                self.plans.pop(next(iter(self.plans)))
        return plan, params, need_grad

    def run(self, mods, inputs, training, kind, pre=None):
        """`pre` = (outs, saved) of a forward that forward_multi() has already enqueued for this plan."""
        plan, params, need_grad = self._plan_for(mods, inputs, training, kind)
        if need_grad:
            if self.grad_sink is not None:
                anchor = torch.empty((), dtype=torch.float32, device=plan.device, requires_grad=True)
                outs = _StackFunction.apply(self, plan, len(inputs), pre, *inputs, anchor)
            else:
                outs = _StackFunction.apply(self, plan, len(inputs), pre, *inputs, *params)
        else:
            with torch.no_grad():
                outs, saved = pre if pre is not None else self._forward(plan, inputs)
            saved[1].release()
            outs = tuple(outs)
        return outs

    def _persist_ws(self, plan):
        ws = getattr(plan, "_persist_buf", None)
        if ws is None:
            ws = torch.zeros(max(plan.persist.size, _ALIGN), dtype=torch.uint8, device=plan.device)
            plan._persist_buf = ws
        return ws

    def _call(self, plan, ops, bases):
        arr = (C.c_void_p * len(bases))(*bases)
        with torch.cuda.device(plan.device):
            stream = torch.cuda.current_stream().cuda_stream
            rc = _lib.lib().mmd_bifpn_run(ops, len(ops), arr, len(bases), plan.B, plan.Cc,
                                          _lib.MMD_F32 if plan.dtype == torch.float32 else _lib.MMD_BF16, stream)
        _lib.check(rc, "mmd_bifpn_run")

    def _prep(self, plan, bases):
        """(Re)build the packed parameter blocks when the parameters may have changed: every training forward (the
        optimiser updates the weights between steps); for eval plans (frozen teachers) only when a parameter / buffer
        version or the global running-statistics epoch moved.  Training plans with frozen BatchNorm layers also get
        those layers' (scale, shift, mean, invstd) vectors rewritten here, in fp32 too: gamma and beta move every step."""
        if plan.dtype != torch.bfloat16 and not plan.copies and not plan.frozen:
            return
        if plan.train:
            for m in plan.mods:   # this forward updates running statistics through raw pointers
                object.__setattr__(m, _EPOCH_ATTR, getattr(m, _EPOCH_ATTR, 0) + 1)
        else:
            sig = (tuple(getattr(m, _EPOCH_ATTR, 0) for m in plan.mods), tuple(t._version for t in plan.state_tensors))
            if getattr(plan, "_prep_sig", None) == sig:
                return
            plan._prep_sig = sig
        arr = (C.c_void_p * len(bases))(*bases)
        with torch.cuda.device(plan.device):
            stream = torch.cuda.current_stream().cuda_stream
            rc = _lib.lib().mmd_bifpn_prep(plan.fwd_ops, len(plan.fwd_ops), arr, len(bases), plan.Cc,
                                           _lib.MMD_F32 if plan.dtype == torch.float32 else _lib.MMD_BF16, stream)
        _lib.check(rc, "mmd_bifpn_prep")

    def _forward_prepare(self, plan, inputs):
        """Everything of a forward except the kernel launches: arena lease, outputs, base table, packed parameters."""
        dev = plan.device
        xs = [x.detach().contiguous(memory_format=torch.channels_last) for x in inputs]
        arena = _Lease(plan.pool_fwd, plan.fwd_arena.size, dev)
        outs = [torch.empty(s, dtype=plan.dtype, device=dev, memory_format=torch.channels_last) if len(s) == 4 else
                torch.empty(s, dtype=plan.dtype, device=dev) for s in plan.out_shapes]
        bases = [0] * plan.n_bases
        bases[B_FWD] = arena.data_ptr()
        bases[B_PERSIST] = self._persist_ws(plan).data_ptr()
        for i, x in enumerate(xs):
            bases[B_EXT + i] = x.data_ptr()
        for k, o in enumerate(outs):
            bases[plan.B_OUT + k] = o.data_ptr()
        if plan.const is not None:
            bases[plan.B_CONST] = plan.const.data_ptr()
        self._prep(plan, bases)
        return bases, outs, (xs, arena, outs)

    def _forward(self, plan, inputs):
        bases, outs, saved = self._forward_prepare(plan, inputs)
        self._call(plan, plan.fwd_ops, bases)
        return outs, saved

    def _backward(self, plan, saved, gouts):
        xs, arena, outs = saved
        dev = plan.device
        gs = []
        for g, o in zip(gouts, outs):
            if g is None:
                g = torch.zeros_like(o)
            g = g.detach().to(plan.dtype)
            gs.append(g.contiguous(memory_format=torch.channels_last) if g.dim() == 4 else g.contiguous())
        bwd = _Lease(plan.pool_bwd, plan.bwd_arena.size, dev)
        zero = torch.zeros(max(plan.zero_arena.size, _ALIGN) // 4, dtype=torch.float32, device=dev)
        gin = [torch.empty_like(x) if need else None for x, need in zip(xs, plan.in_need_grad)]
        bases = [0] * plan.n_bases
        bases[B_FWD] = arena.data_ptr()
        bases[B_PERSIST] = self._persist_ws(plan).data_ptr()
        bases[B_BWD] = bwd.data_ptr()
        bases[B_ZERO] = zero.data_ptr()
        for i, x in enumerate(xs):
            bases[B_EXT + i] = x.data_ptr()
            if gin[i] is not None:
                bases[plan.B_GIN + i] = gin[i].data_ptr()
        for k, (o, g) in enumerate(zip(outs, gs)):
            bases[plan.B_OUT + k] = o.data_ptr()
            bases[plan.B_GOUT + k] = g.data_ptr()
        if plan.const is not None:
            bases[plan.B_CONST] = plan.const.data_ptr()
        self._call(plan, plan.bwd_ops, bases)
        bwd.release()
        return gin, zero
