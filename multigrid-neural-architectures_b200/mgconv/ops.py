"""Plan ops: each owns its device buffers and the pre-built C structs of its libmgconv calls.

setup_fwd runs in forward order (allocate activations), setup_bwd in reverse order (so that by
the time a tensor's producer plans its gradient, every consumer has registered the grid it will
write its contribution to).  Gradients are combined in *gather form* (mg_grad_combine): each
tensor reads its consumers' gradient grids through the routing that consumer applied (same /
2x2 arg-max / 2x2 block sum / 3x3-s2 arg-max), so there are no atomics and the summation order
is fixed -- ConcatTable's backward-sum (models/ilsvrc/rnmg.lua:53-82,106,140) without scatter.
"""
import ctypes as C
import os
import torch

from . import ffi
from .ffi import mg_grid, mg_conv_desc, mg_grad_src, mg_bn_fused, mg_dropout, ptr, MG_SEG_SAME, MG_SEG_POOL, MG_SEG_UP, MG_SRC_POOL3, MG_MAX_SRC
from .sched import Unit

# the passes of the engine: forward, backward, and backward in the two halves of the nn protocol -- "update"
# (updateGradInput: data gradients, no parameter gradient) and "acc" (accGradParameters: the parameter gradients)
BWD = ("backward", "update")


def cpad(c):
    return (c + 7) // 8 * 8


def _k(x):
    """dependency key of a device buffer: its base address (torch tensor, mg_grid, raw pointer or None)"""
    if x is None:
        return None
    if isinstance(x, torch.Tensor):
        return x.data_ptr()
    if isinstance(x, mg_grid):
        return x.data
    return int(x)


def _keys(*xs):
    return [k for k in (_k(x) for x in xs) if k]


class TSpec:
    """a materialised NHWC activation tensor of the plan"""

    def __init__(self, idx, N, C, H, W, name, needs_grad=True):
        self.idx, self.N, self.C, self.H, self.W = idx, N, C, H, W
        self.Cp = cpad(C)
        self.name = name
        self.needs_grad = needs_grad
        self.producer = None
        self.pooled = None   # companion TSpec = maxpool2x2_ceil(self)
        self.srcs = []       # Src records registered by consumers (backward)
        self.buf = None
        self.G = None        # mg_grid of the gradient w.r.t. this tensor, set by the producer's backward plan

    def grid(self, buf=None, scale=None, shift=None, relu=0):
        b = self.buf if buf is None else buf
        return mg_grid(b.data_ptr(), None if scale is None else scale.data_ptr(),
                       None if shift is None else shift.data_ptr(), relu, self.N, self.H, self.W, self.C, self.Cp)

    def shape(self):
        return (self.N, self.H, self.W, self.Cp)


class Src:
    """one gradient contribution: grid `buf` [N,H,W,Cp] read at channel offset c_off through `mode`"""

    def __init__(self, buf, H, W, C, Cp, c_off, mode, aux=None):
        self.buf, self.H, self.W, self.C, self.Cp, self.c_off, self.mode, self.aux = buf, H, W, C, Cp, c_off, mode, aux


class Combine:
    """gradient of tensor t = sum of its registered sources (optionally x ReLU mask, + BN sums)"""

    def __init__(self, E, t, relu_mask=False, bn_x=None, sums=None, private=False, pooled_mask=None):
        """pooled_mask: t itself was never stored (stem: BN + ReLU + pool fused); its ReLU mask at an arg-max is the sign of
        the pooled tensor given here (mg_grad_combine relu_mask = 2)"""
        self.E, self.t = E, t
        self.pooled_mask = pooled_mask
        srcs = t.srcs
        if len(srcs) > MG_MAX_SRC:
            raise NotImplementedError(f"{t.name}: {len(srcs)} gradient sources > MG_MAX_SRC")
        s0 = srcs[0] if len(srcs) == 1 else None
        self.noop = False
        self.alias = (s0 is not None and s0.mode == MG_SEG_SAME and s0.c_off == 0 and s0.Cp == t.Cp
                      and not relu_mask and sums is None and not private)
        if self.alias:
            self.buf = s0.buf
            return
        self.buf = E.alloc(t.shape())
        self.noop = len(srcs) == 0  # unused output (e.g. grids dropped by SelectTable(1)): gradient stays zero
        self.x = t.grid() if pooled_mask is None else pooled_mask.grid()
        self.bn_x = bn_x.grid() if bn_x is not None else None
        self.arr = (mg_grad_src * max(1, len(srcs)))()
        for i, s in enumerate(srcs):
            self.arr[i].g = mg_grid(s.buf.data_ptr(), None, None, 0, t.N, s.H, s.W, s.C, s.Cp)
            self.arr[i].c_offset = s.c_off
            self.arr[i].mode = s.mode
            self.arr[i].aux = None if s.aux is None else s.aux.data_ptr()
        self.n = len(srcs)
        self.relu_mask = int(relu_mask) if pooled_mask is None else 2
        self.sums = sums
        self.d = t.grid(self.buf)

    def grid(self):
        return self.t.grid(self.buf)

    def io(self):
        """(buffers read, buffers written) by run()"""
        if self.alias or self.noop:
            return [], []
        r = _keys(self.t.buf if self.pooled_mask is None else self.pooled_mask.buf, self.bn_x, *[sr.buf for sr in self.t.srcs], *[sr.aux for sr in self.t.srcs])
        return r, _keys(self.buf, self.sums)

    def run(self):
        if self.alias or self.noop:
            return
        self.E.ctx.call("mg_grad_combine", C.byref(self.x), self.relu_mask,
                        C.byref(self.bn_x) if self.bn_x is not None else None, self.n, self.arr,
                        C.byref(self.d), ptr(self.sums))

    def run_frozen(self, bn, g, write_d):
        """the same sum, for a tensor that feeds BatchNorm `bn` in evaluation mode: writes g = gamma * invstd_r * d (and d only
        when write_d) and accumulates (sum d, sum d*y) into self.sums (mg_grad_combine_bn_frozen)"""
        if self.noop:
            return
        self.E.ctx.call("mg_grad_combine_bn_frozen", C.byref(self.x), self.relu_mask, C.byref(self.bn_x), self.n, self.arr,
                        ptr(bn.weight), ptr(bn.running_var), bn.eps, C.byref(g), C.byref(self.d) if write_d else None, ptr(self.sums))


def plan_companion_grad(E, x, p):
    """route the gradient of p = maxpool2x2_ceil(x) into x (arg-max recomputed from x in the combine).
    Sources of p that read it at its own resolution compose with the pooling directly; anything else
    (p up-sampled or pooled again by its consumer) needs p's gradient materialised first."""
    if p is None or not p.needs_grad or not x.needs_grad:
        return None
    if all(s.mode == MG_SEG_SAME for s in p.srcs):
        for s in p.srcs:
            x.srcs.append(Src(s.buf, s.H, s.W, s.C, s.Cp, s.c_off, MG_SEG_POOL))
        return None
    comb = Combine(E, p)
    x.srcs.append(Src(comb.buf, p.H, p.W, p.C, p.Cp, 0, MG_SEG_POOL))
    return comb


class Op:
    """Device buffers (reads, writes) of a unit are what the lane scheduler (sched.py) orders across streams; None = unknown:
    the unit then runs on lane 0 behind a full join.  The caller's tensors (InputOp.src, grad_out), bound anew on every call
    and touched by no other unit, are not listed."""
    def setup_fwd(self, E): pass
    def setup_bwd(self, E): pass
    def fwd(self, E): pass
    def io_fwd(self): return None
    def size(self): return getattr(getattr(self, "out", None), "H", 0)

    def forward_unit(self):
        return Unit(self, self.io_fwd(), lambda E, params: self.fwd(E), ("forward",))

    def backward_units(self):
        """the op's work in the backward passes, in execution order, built once after setup_bwd.  run(E, params): params =
        False in updateGradInput, which writes no parameter gradient.  BatchNorm layers add theirs in accGradParameters
        through ApplyOp.param_job (one batched launch of the engine) instead of a unit.  Every op has a unit in backward and
        updateGradInput, if only this empty one: the lane schedules number their events by unit."""
        return [Unit(self, ([], []), lambda E, params: None, BWD)]


def _combine_units(op, comb):
    """the backward of an op whose gradient is a Combine (or nothing, comb = None)"""
    if comb is None:
        return Op.backward_units(op)
    return [Unit(op, comb.io(), lambda E, params: comb.run(), BWD)]


def _merge(*ios):
    r, w = [], []
    for io in ios:
        if io is not None:
            r += io[0]; w += io[1]
    return r, w


class InputOp(Op):
    def __init__(self, out):
        self.out = out
        out.producer = self
        self.src = None   # NCHW fp32 torch tensor, set by the engine per call
        self.comb = None
        self.grad_nchw = None

    def setup_fwd(self, E):
        self.out.buf = E.alloc(self.out.shape())
        self.g = self.out.grid()

    def io_fwd(self):
        return [], _keys(self.out.buf)

    def fwd(self, E):
        E.ctx.call("mg_import_nchw", ptr(self.src), C.byref(self.g))

    def setup_bwd(self, E):
        if self.out.needs_grad:
            self.comb = Combine(E, self.out)
            self.grad_nchw = torch.empty((self.out.N, self.out.C, self.out.H, self.out.W), dtype=torch.float32, device=E.device)
            self.dg = self.comb.grid()

    def backward_units(self):
        if self.comb is None:
            return super().backward_units()
        return [Unit(self, _merge(self.comb.io(), ([], _keys(self.grad_nchw))), self.backward, BWD)]

    def backward(self, E, params):
        self.comb.run()
        E.ctx.call("mg_export_nchw", C.byref(self.dg), ptr(self.grad_nchw))


class AvgPoolOp(Op):
    """cudnn.SpatialAveragePooling(r,r,r,r) of the input image (ilsvrc/rnmg.lua:175-177); backward (needInputGrad): the gradient of
    the pooled image spread over its r x r windows, one more gradient source of the image"""

    def __init__(self, inp, r, out):
        self.inp, self.r, self.out = inp, r, out
        out.producer = self
        self.comb = None

    def setup_fwd(self, E):
        self.out.buf = E.alloc(self.out.shape())
        self.gi, self.go = self.inp.grid(), self.out.grid()

    def io_fwd(self):
        return _keys(self.inp.buf), _keys(self.out.buf)

    def fwd(self, E):
        E.ctx.call("mg_avgpool_forward", C.byref(self.gi), self.r, C.byref(self.go))

    def setup_bwd(self, E):
        if self.inp.needs_grad and self.out.needs_grad:
            t = self.inp
            self.comb = Combine(E, self.out)
            self.din = E.alloc(t.shape())
            self.dg_out, self.dg_in = self.comb.grid(), t.grid(self.din)
            t.srcs.append(Src(self.din, t.H, t.W, t.C, t.Cp, 0, MG_SEG_SAME))

    def backward_units(self):
        if self.comb is None:
            return super().backward_units()
        return [Unit(self, _merge(self.comb.io(), (_keys(self.comb.buf), _keys(self.din))), self.backward, BWD)]

    def backward(self, E, params):
        self.comb.run()
        E.ctx.call("mg_avgpool_backward", C.byref(self.dg_out), self.r, C.byref(self.dg_in))


def _stats(conv):
    """BatchNorm sums a convolution's epilogue reduces: none when the BatchNorm that follows is frozen (it reads running statistics)"""
    return None if conv.apply is not None and conv.apply.frozen else ptr(conv.sums)


class ConvOp(Op):
    """gather(segments) -> k x k convolution (+bias); raw output y and, when a BatchNorm follows,
    the per-channel (sum, sumsq) of y.  ResampleConcat + cudnn.SpatialConvolution
    (ilsvrc/rnmg.lua:41-89 + 26/36)."""

    def __init__(self, b, mod, segs, H, W, name):
        self.mod, self.segs, self.H, self.W, self.name = mod, segs, H, W, name
        self.k, self.stride, self.pad, self.Cout = mod.kW, mod.dW, mod.padW, mod.nOutputPlane
        self.Ho = (H + 2 * self.pad - self.k) // self.stride + 1
        self.Wo = (W + 2 * self.pad - self.k) // self.stride + 1
        self.y = b.new_tensor(self.Cout, self.Ho, self.Wo, name + ".y")
        self.y.producer = self
        self.apply = None
        self.want_stats = False
        self.sums = None
        self.ycomb = None

    def setup_fwd(self, E):
        d = mg_conv_desc()
        d.n_seg = len(self.segs)
        for i, (t, m) in enumerate(self.segs):
            d.seg[i] = t.grid()
            d.seg_mode[i] = m
        d.ksize, d.stride, d.pad, d.Cout, d.H, d.W = self.k, self.stride, self.pad, self.Cout, self.H, self.W
        self.desc = d
        self.y.buf = E.alloc(self.y.shape())
        self.yg = self.y.grid()
        if self.want_stats:
            self.sums = E.alloc_sums(2 * self.Cout, "fwd")
        # Image-fed strided stem (cudnn.SpatialConvolution(3, C, 7,7, 2,2, 3,3), ilsvrc/rnmg.lua:180) on the tensor-core
        # path: im2col once, then a 1x1 convolution over the column tensor with the module's own weight storage
        # ([Cout][3][7][7] flattened IS [Cout][147][1][1]); forward and weight gradient read K = 147 real channels
        # instead of 49 taps x 8 padded ones.  Only when no gradient w.r.t. the image is wanted.  Opt-in (MGCONV_STEM_IM2COL=1):
        # measured on R-MG-34 / B = 256 the conv entry points gain 0.45 ms but the 1.3 GB column tensor costs 1.4 ms.
        t0 = self.segs[0][0]
        self.col = None
        if (E.use_packed and len(self.segs) == 1 and self.segs[0][1] == MG_SEG_SAME and self.stride > 1 and self.k > 1
                and t0.C * self.k * self.k <= 512 and not t0.needs_grad and os.environ.get("MGCONV_STEM_IM2COL", "0") == "1"):
            K = t0.C * self.k * self.k
            Kp = cpad(K)
            self.col = E.alloc((self.y.N, self.Ho, self.Wo, Kp))
            self.col_g = mg_grid(self.col.data_ptr(), None, None, 0, self.y.N, self.Ho, self.Wo, K, Kp)
            self.in_g = t0.grid()
            d1 = mg_conv_desc()
            d1.n_seg = 1
            d1.seg[0] = self.col_g
            d1.seg_mode[0] = MG_SEG_SAME
            d1.ksize, d1.stride, d1.pad, d1.Cout, d1.H, d1.W = 1, 1, 0, self.Cout, self.Ho, self.Wo
            self.desc_direct, self.desc = d, d1
        self.wpack = self.wpack_t = None
        nb = ffi.lib.mg_conv_packed_bytes(C.byref(self.desc), 0) if E.use_packed else 0
        if nb:
            self.wpack = E.alloc((nb,), torch.uint8)
        self.Ccat = sum(t.C for t, _ in self.segs)
        self.CcatP = sum(t.Cp for t, _ in self.segs)

    def pack_jobs(self):
        """(desc, weight, packed image, transposed) of every operand image this convolution needs"""
        jobs = []
        if self.wpack is not None:
            jobs.append((self.desc, self.mod.weight, self.wpack, 0))
        if self.wpack_t is not None:
            jobs.append((self.desc, self.mod.weight, self.wpack_t, 1))
        return jobs

    def _tunable(self):
        return self.wpack is not None and self.k == 3 and self.stride == 1 and self.pad == 1 and 7 <= self.W <= 63

    def _pick(self, E, field, run):
        """time the kernel variants of one direction on this layer's own buffers and keep the fastest
        (cudnn.benchmark = true of the reference, models/ilsvrc/rnmg.lua:230-231)"""
        best, best_t = 0, None
        for algo in (ffi.MG_ALGO_TILE128, ffi.MG_ALGO_TILE256, ffi.MG_ALGO_RESIDENT, ffi.MG_ALGO_TILE128_DEEP, ffi.MG_ALGO_TILE256_DEEP,
                     ffi.MG_ALGO_TILE128_MID, ffi.MG_ALGO_PAIR128, ffi.MG_ALGO_PAIR256, ffi.MG_ALGO_RESIDENT_PAIR):
            setattr(self.desc, field, algo)
            run()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                run()
            e1.record()
            e1.synchronize()
            t = e0.elapsed_time(e1)
            if best_t is None or t < best_t * 0.97:   # a later variant must win by 3 % (timer noise)
                best, best_t = algo, t
        setattr(self.desc, field, best)
        return best

    def tune_fwd(self, E):
        if self._tunable():
            self._pick(E, "algo_fwd", lambda: self.fwd(E))

    def tune_bwd(self, E):
        if self._tunable() and self.needs_dgrad and self.wpack_t is not None:
            g = self.y.G
            self._pick(E, "algo_bwd_data", lambda: E.ctx.call("mg_conv_backward_data", C.byref(self.desc), ptr(self.mod.weight),
                                                              ptr(self.wpack_t), C.byref(g), C.byref(self.dcat_g)))

    def size(self):
        return self.H

    def io_fwd(self):
        return _keys(*[t.buf for t, _ in self.segs]), _keys(self.y.buf, self.sums, self.col)

    def fwd(self, E):
        if self.col is not None:
            E.ctx.call("mg_im2col", C.byref(self.in_g), self.k, self.stride, self.pad, C.byref(self.col_g))
        E.ctx.call("mg_conv_forward", C.byref(self.desc), ptr(self.mod.weight), ptr(self.wpack), ptr(self.mod.bias),
                   C.byref(self.yg), _stats(self))

    def setup_bwd(self, E):
        if self.apply is None:  # plain convolution (Linear head): gradient of y comes straight from its consumers
            self.ycomb = Combine(E, self.y)
            self.y.G = self.ycomb.grid()
        self.needs_dgrad = any(t.needs_grad for t, _ in self.segs)
        self.dcat = None
        if self.needs_dgrad:
            self.dcat = E.alloc((self.y.N, self.H, self.W, self.CcatP))
            self.dcat_g = mg_grid(self.dcat.data_ptr(), None, None, 0, self.y.N, self.H, self.W, self.CcatP, self.CcatP)
            off = 0
            for t, m in self.segs:
                if t.needs_grad:
                    t.srcs.append(Src(self.dcat, self.H, self.W, self.CcatP, self.CcatP, off, m))
                off += t.Cp
            nb = ffi.lib.mg_conv_packed_bytes(C.byref(self.desc), 1) if E.use_packed else 0
            if nb:
                self.wpack_t = E.alloc((nb,), torch.uint8)

    def backward_units(self):
        """dgrad, which the rest of backward waits for, and wgrad, which only the optimiser (and the gradient all-reduce) waits
        for: the lane schedule of backward runs it on a background lane"""
        io_d = _merge(self.ycomb.io() if self.ycomb is not None else None,
                      (_keys(self.y.G), _keys(self.dcat)) if self.needs_dgrad else ([], []))
        io_w = (_keys(self.y.G, self.col, *[t.buf for t, _ in self.segs]), _keys(self.mod.gradWeight, self.mod.gradBias))
        return [Unit(self, io_d, self.dgrad, BWD), Unit(self, io_w, self.wgrad, ("backward", "acc"), "background")]

    def dgrad(self, E, params):
        """gradient of y from its consumers (plain convs), then the gradient of the input"""
        if self.ycomb is not None:
            self.ycomb.run()
        if self.needs_dgrad:
            E.ctx.call("mg_conv_backward_data", C.byref(self.desc), ptr(self.mod.weight), ptr(self.wpack_t),
                       C.byref(self.y.G), C.byref(self.dcat_g))

    def wgrad(self, E, params):
        fused_bias = self.apply is not None and self.apply.bn is not None   # done by mg_bn_backward (from the BatchNorm sums)
        E.ctx.call("mg_conv_backward_weight", C.byref(self.desc), C.byref(self.y.G), ptr(self.mod.gradWeight),
                   None if fused_bias else ptr(self.mod.gradBias), E.gscale)
        E.param_done(self.mod)


class UpConvOp(Op):
    """cudnn.SpatialFullConvolution(nIP, nOP, 2,2,2,2) of U-MG (unmg.lua:35-52); epilogue (BN, ReLU) through
    the same ApplyOp as a convolution"""

    def __init__(self, b, mod, inp, name):
        self.mod, self.inp, self.name = mod, inp, name
        self.Cout, self.Ho, self.Wo = mod.nOutputPlane, 2 * inp.H, 2 * inp.W
        self.segs = [(inp, MG_SEG_SAME)]
        self.k = 2
        self.y = b.new_tensor(self.Cout, self.Ho, self.Wo, name + ".y")
        self.y.producer = self
        self.apply = None
        self.want_stats = False
        self.sums = None
        self.ycomb = None
        self.needs_dgrad = inp.needs_grad

    def setup_fwd(self, E):
        self.y.buf = E.alloc(self.y.shape())
        self.gi, self.yg = self.inp.grid(), self.y.grid()
        if self.want_stats:
            self.sums = E.alloc_sums(2 * self.Cout, "fwd")

    def pack_jobs(self):
        return []

    def size(self):
        return self.Ho

    def io_fwd(self):
        return _keys(self.inp.buf), _keys(self.y.buf, self.sums)

    def fwd(self, E):
        E.ctx.call("mg_upconv2x2_forward", C.byref(self.gi), ptr(self.mod.weight), ptr(self.mod.bias), C.byref(self.yg), _stats(self))

    def setup_bwd(self, E):
        if self.apply is None:
            self.ycomb = Combine(E, self.y)
            self.y.G = self.ycomb.grid()
        self.dx = None
        if self.inp.needs_grad:
            self.dx = E.alloc(self.inp.shape())
            self.dxg = self.inp.grid(self.dx)
            self.inp.srcs.append(Src(self.dx, self.inp.H, self.inp.W, self.inp.C, self.inp.Cp, 0, MG_SEG_SAME))

    def backward_units(self):
        """backward makes one mg_upconv2x2_backward call for dx, dw and dbias (two would launch its shuffle kernel twice);
        updateGradInput makes it for dx alone, accGradParameters for dw and dbias alone"""
        r, w = _keys(self.y.G, self.inp.buf), _keys(self.mod.gradWeight, self.mod.gradBias)
        io = _merge(self.ycomb.io() if self.ycomb is not None else None, (r, w + _keys(self.dx)))
        return [Unit(self, io, self.backward, BWD), Unit(self, (r, w), lambda E, params: self._call(E, False, True), ("acc",))]

    def backward(self, E, params):
        if self.ycomb is not None:
            self.ycomb.run()
        if params or self.dx is not None:
            self._call(E, self.dx is not None, params)

    def _call(self, E, dx, params):
        fused_bias = self.apply is not None and self.apply.bn is not None   # done by mg_bn_backward (from the BatchNorm sums)
        E.ctx.call("mg_upconv2x2_backward", C.byref(self.gi), ptr(self.mod.weight), C.byref(self.y.G), C.byref(self.dxg) if dx else None,
                   ptr(self.mod.gradWeight) if params else None, None if fused_bias or not params else ptr(self.mod.gradBias), E.gscale)
        if params:
            E.param_done(self.mod)


class ApplyOp(Op):
    """epilogue pass of a convolution: out = relu?( BN(y) + shortcut[c < C_s] ), plus the pooled
    companion of out when a coarser neighbour gathers it.  SpatialBatchNormalization -> [ReLU] or
    -> CAddTable(true) with Identity / nn.Padding shortcut -> [ReLU] (ilsvrc/rnmg.lua:13-39,140-154)."""

    def __init__(self, conv, bn, relu, res, out):
        self.conv, self.bn, self.relu, self.res, self.out = conv, bn, relu, res, out
        conv.apply = self
        conv.want_stats = bn is not None
        out.producer = self
        self.pooled = None
        self.pool3 = None    # Pool3Op fused into this pass (fuse_stem_pool3): BN + ReLU + 3x3 / stride-2 max-pool, `out` never stored
        # the BatchNorm runs in evaluation mode (running statistics, no update; backward through the frozen affine): set by the
        # engine before every forward from the model's mode and the module's own train flag (Engine.forward)
        self.frozen = False

    def setup_fwd(self, E):
        t, y = self.out, self.conv.y
        # fused with the stem's pool: the activation is never written -- a one-element stand-in keeps the mg_grid structs valid
        t.buf = E.alloc(t.shape()) if self.pool3 is None else E.alloc((8,))
        self.og = t.grid()
        self.pg = None
        if self.pooled is not None:
            self.pooled.buf = E.alloc(self.pooled.shape())
            self.pg = self.pooled.grid()
        self.rg = self.res.grid() if self.res is not None else None
        if self.bn is not None:
            self.scale, self.shift = E.alloc((y.Cp,), torch.float32), E.alloc((y.Cp,), torch.float32)
            self.mean, self.invstd = E.alloc((y.Cp,), torch.float32), E.alloc((y.Cp,), torch.float32)
            self.zg = y.grid(scale=self.scale, shift=self.shift)
        else:
            self.zg = y.grid()
        self.count = y.N * y.H * y.W
        self.bnf = None   # mg_bn_fused, built on first use (parameter storage may be re-homed by getParameters())

    def _bn_struct(self, E):
        bn = self.bn
        training = not self.frozen
        key = (bn.weight.data_ptr(), bn.bias.data_ptr(), bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
               training, E.bn_sync, float(bn.eps), float(bn.momentum))
        if self.bnf is None or self.bnf_key != key:
            f = mg_bn_fused()
            f.sums = self.conv.sums.data_ptr()
            f.count = self.count * (max(1, E.bn_sync) if training else 1)
            f.gamma, f.beta = bn.weight.data_ptr(), bn.bias.data_ptr()
            f.running_mean, f.running_var = bn.running_mean.data_ptr(), bn.running_var.data_ptr()
            f.eps, f.momentum, f.training = bn.eps, bn.momentum, int(training)
            f.save_mean, f.save_invstd = self.mean.data_ptr(), self.invstd.data_ptr()
            self.bnf, self.bnf_key = f, key
        return self.bnf

    def io_fwd(self):
        r = _keys(self.conv.y.buf, self.conv.sums, None if self.res is None else self.res.buf)
        w = _keys(self.out.buf, None if self.pooled is None else self.pooled.buf)
        if self.pool3 is not None:
            w += _keys(self.pool3.out.buf, self.pool3.code)
        if self.bn is not None:
            w += _keys(self.scale, self.shift, self.mean, self.invstd)
        return r, w

    def fwd(self, E, synced=False):
        """synced: the engine has already all-reduced this layer's statistics together with those of the other scales of the stage"""
        bn = self.bn
        rg = C.byref(self.rg) if self.rg is not None else None
        pg = C.byref(self.pg) if self.pg is not None else None
        if bn is not None:
            if E.bn_sync and not self.frozen and not synced:   # cross-replica statistics: sum (sum y, sum y^2) over the ranks
                E.ctx.call("mg_allreduce_inline", ptr(self.conv.sums), self.conv.sums.numel(), 2)   # int64 limbs of mg_sum
            if self.pool3 is not None:   # stem: + SpatialMaxPooling(3,3,2,2,1,1), arg-max codes for the backward routing
                E.ctx.call("mg_bn_relu_pool3_forward", C.byref(self.zg), C.byref(self._bn_struct(E)), C.byref(self.pool3.go), ptr(self.pool3.code))
                return
            # SpatialBatchNormalization finalisation + CAddTable + ReLU + pooled companion in one pass
            E.ctx.call("mg_bn_residual_forward", C.byref(self.zg), C.byref(self._bn_struct(E)), rg, int(self.relu), C.byref(self.og), pg)
        else:
            E.ctx.call("mg_residual_forward", C.byref(self.zg), rg, int(self.relu), C.byref(self.og), pg)

    def setup_bwd(self, E):
        t, y = self.out, self.conv.y
        self.pc = plan_companion_grad(E, t, self.pooled)
        self.dsums = E.alloc_sums(2 * t.C, "bwd") if self.bn is not None else None
        self.comb = Combine(E, t, relu_mask=self.relu, bn_x=y if self.bn is not None else None, sums=self.dsums,
                            private=self.bn is not None, pooled_mask=None if self.pool3 is None else self.pool3.out)
        D = self.comb.buf
        if self.res is not None and self.res.needs_grad:
            self.res.srcs.append(Src(D, t.H, t.W, t.C, t.Cp, 0, MG_SEG_SAME))
        # frozen BatchNorm: the combine writes G itself, and D only when the shortcut reads it
        self.d_for_res = self.res is not None and self.res.needs_grad
        if self.bn is not None:
            G = E.alloc(t.shape()) if self.res is not None else D   # the shortcut still reads D
            self.G = G   # keep the storage alive: the mg_grid structs below only hold raw pointers
            self.coef = E.alloc((3 * t.Cp,), torch.float32)
            self.dg, self.gg = t.grid(D), t.grid(G)
            self.yraw = y.grid()
            y.G = self.gg
        else:
            y.G = t.grid(D)

    def backward_units(self):
        """one unit: the engine's -bnSync path runs the two halves, bwd_combine and bwd_bn, itself"""
        io = _merge(self.pc.io() if self.pc is not None else None, self.comb.io())
        if self.bn is not None:
            bn = self.bn
            io = _merge(io, (_keys(self.conv.y.buf, self.comb.buf, self.dsums, self.mean, self.invstd),
                             _keys(self.G, bn.gradWeight, bn.gradBias, self.conv.mod.gradBias)))
        return [Unit(self, io, self.backward, BWD)]

    def backward(self, E, params):
        self.bwd_combine(E)
        self.bwd_bn(E, params=params)

    def param_job(self, E, job):
        """fill the mg_bn_param_job of this layer (mg_bn_param_grad): exactly what bwd_bn adds to the parameter gradients, from the
        sums and statistics updateGradInput left behind"""
        bn = self.bn
        job.sums, job.C = _k(self.dsums), self.out.C
        job.gamma, job.dgamma, job.dbeta, job.conv_dbias = _k(bn.weight), _k(bn.gradWeight), _k(bn.gradBias), _k(self.conv.mod.gradBias)
        if self.frozen:
            job.frozen, job.count, job.gscale = 1, 0, E.gscale
            job.running_mean, job.running_var, job.eps = _k(bn.running_mean), _k(bn.running_var), bn.eps
            job.save_mean = job.save_invstd = None
        else:
            job.frozen, job.count, job.gscale = 0, self.count * max(1, E.bn_sync), E.gscale / max(1, E.bn_sync)
            job.save_mean, job.save_invstd = _k(self.mean), _k(self.invstd)
            job.running_mean = job.running_var = None
            job.eps = 0.0

    def bwd_combine(self, E):
        if self.pc is not None:
            self.pc.run()
        if self.frozen:
            self.comb.run_frozen(self.bn, self.gg, self.d_for_res)
        else:
            self.comb.run()

    def bwd_bn(self, E, synced=False, params=True):
        """params = False (updateGradInput): G alone, no parameter gradient; the sums stay for param_job"""
        bn = self.bn
        if bn is not None and self.frozen:
            if not params:   # the combine already wrote G
                return
            # the sums are this rank's own: every rank adds its full share of dgamma / dbeta / gradBias, the gradient all-reduce
            # sums them like any other parameter gradient
            E.ctx.call("mg_bn_backward_frozen", ptr(self.dsums), self.out.C, ptr(bn.weight), ptr(bn.running_mean), ptr(bn.running_var),
                       bn.eps, ptr(bn.gradWeight), ptr(bn.gradBias), E.gscale, ptr(self.conv.mod.gradBias))
            E.param_done(bn)
        elif bn is not None:
            if E.bn_sync and not synced:
                E.ctx.call("mg_allreduce_inline", ptr(self.dsums), self.dsums.numel(), 2)
            pg = ptr if params else (lambda t: None)
            E.ctx.call("mg_bn_backward", C.byref(self.yraw), C.byref(self.dg), C.byref(self.gg), ptr(self.dsums), self.count * max(1, E.bn_sync),
                       ptr(bn.weight), ptr(self.mean), ptr(self.invstd), pg(bn.gradWeight), pg(bn.gradBias),
                       # sync-BN: the sums are already global, every rank adds 1/N of dgamma / dbeta / the conv's gradBias
                       # (all derived from the sums) before the gradient all-reduce
                       E.gscale / max(1, E.bn_sync), ptr(self.coef), pg(self.conv.mod.gradBias))
            if params:
                E.param_done(bn)


class PoolOp(Op):
    """stand-alone SpatialMaxPooling(2,2,2,2):ceil() (mgPool, ilsvrc/rnmg.lua:191-224) when the
    producer of `inp` is not an apply pass that could write the companion itself"""

    def __init__(self, inp, out):
        self.inp, self.out = inp, out
        out.producer = self

    def setup_fwd(self, E):
        self.out.buf = E.alloc(self.out.shape())
        self.gi, self.go = self.inp.grid(), self.out.grid()

    def io_fwd(self):
        return _keys(self.inp.buf), _keys(self.out.buf)

    def fwd(self, E):
        E.ctx.call("mg_pool_forward", C.byref(self.gi), C.byref(self.go), 0, None)

    def setup_bwd(self, E):
        self.pc = plan_companion_grad(E, self.inp, self.out)

    def backward_units(self):
        return _combine_units(self, self.pc)


class Pool3Op(Op):
    """SpatialMaxPooling(3,3,2,2,1,1) of the ImageNet stem (ilsvrc/rnmg.lua:183)"""

    def __init__(self, inp, out):
        self.inp, self.out = inp, out
        out.producer = self
        self.fused = False   # run by the producing ApplyOp (fuse_stem_pool3)

    def setup_fwd(self, E):
        self.out.buf = E.alloc(self.out.shape())
        self.gi, self.go = self.inp.grid(), self.out.grid()
        # arg-max codes for the backward routing (1 byte / element), bf16 mode only
        self.code = E.alloc(self.out.shape(), torch.uint8) if (E.dtype == ffi.MG_BF16 and (self.inp.needs_grad or self.fused)) else None

    def io_fwd(self):
        if self.fused:
            return [], []
        return _keys(self.inp.buf), _keys(self.out.buf, self.code)

    def fwd(self, E):
        if not self.fused:
            E.ctx.call("mg_pool3s2_forward", C.byref(self.gi), C.byref(self.go), ptr(self.code))

    def setup_bwd(self, E):
        t = self.out
        self.comb = None
        if self.inp.needs_grad:
            self.comb = Combine(E, t)
            self.inp.srcs.append(Src(self.comb.buf, t.H, t.W, t.C, t.Cp, 0, MG_SRC_POOL3, aux=self.code))

    def backward_units(self):
        return _combine_units(self, self.comb)


def _tensor_refs(op):
    """TSpec objects an op holds (attributes, lists, (tensor, mode) pairs)"""
    out = []
    def visit(v):
        if isinstance(v, TSpec):
            out.append(v)
        elif isinstance(v, (list, tuple)):
            for e in v:
                visit(e)
    for v in vars(op).values():
        visit(v)
    return out


def fuse_stem_pool3(plan_ops, E):
    """BN -> ReLU -> SpatialMaxPooling(3,3,2,2,1,1) (ilsvrc/rnmg.lua:181-183) as one pass when the activation has no other reader:
    it is then never written (forward) nor read (backward).  bf16 contexts, training graphs (arg-max codes needed)."""
    if E.dtype != ffi.MG_BF16 or os.environ.get("MGCONV_FUSE_POOL3", "1") == "0":
        return
    for P in [o for o in plan_ops if isinstance(o, Pool3Op)]:
        A = P.inp.producer
        if not (isinstance(A, ApplyOp) and A.bn is not None and A.relu and A.res is None and A.pooled is None and A.out is P.inp):
            continue
        if not P.inp.needs_grad or P.inp.pooled is not None:
            continue
        others = [o for o in plan_ops if o is not A and o is not P and any(t is P.inp for t in _tensor_refs(o))]
        if others:
            continue
        A.pool3, P.fused = P, True


class CatOp(Op):
    """JoinTable(2) materialised because a shortcut needs the concatenation as one tensor
    (first residual unit after an isConcat mgPool, ilsvrc/rnmg.lua:133-137,207)"""

    def __init__(self, parts, out):
        self.parts, self.out = parts, out
        out.producer = self

    def setup_fwd(self, E):
        self.out.buf = E.alloc(self.out.shape())
        self.go = self.out.grid()
        self.gp = [p.grid() for p in self.parts]

    def io_fwd(self):
        return _keys(*[p.buf for p in self.parts]), _keys(self.out.buf)

    def fwd(self, E):
        off = 0
        for p, g in zip(self.parts, self.gp):
            E.ctx.call("mg_copy_channels", C.byref(g), C.byref(self.go), off)
            off += p.C

    def setup_bwd(self, E):
        t = self.out
        self.comb = None
        if t.needs_grad:
            self.comb = Combine(E, t)
            off = 0
            for p in self.parts:
                if p.needs_grad:
                    p.srcs.append(Src(self.comb.buf, t.H, t.W, t.C, t.Cp, off, MG_SEG_SAME))
                off += p.C

    def backward_units(self):
        return _combine_units(self, self.comb)


class DropStepOp(Op):
    """device counter of the plan's dropout masks, advanced on the stream once per training forward before the first DropOp:
    a captured step (graph.GraphedStep) draws new masks on every replay"""

    def setup_fwd(self, E):
        self.step = E.alloc((1,), torch.int64)

    def io_fwd(self):
        return [], _keys(self.step)

    def fwd(self, E):
        E.ctx.call("mg_dropout_advance", ptr(self.step))


class DropOp(Op):
    """nn.Dropout(p) in training mode in front of a convolution (models/cifar/pnmg.lua:25-27): the dropped concatenation of
    the conv's segments, materialised as one tensor that the conv reads as its only segment.  Every element of an up-sampled
    pixel has its own mask element, so the dropout cannot ride on the conv's gather.  Backward: the gradient of the dropped
    tensor times the same mask (regenerated, in place), routed to the parts like CatOp's"""

    def __init__(self, segs, p, ordinal, step_op, out):
        self.segs, self.p, self.ordinal, self.step_op, self.out = segs, p, ordinal, step_op, out
        out.producer = self

    def setup_fwd(self, E):
        self.out.buf = E.alloc(self.out.shape())
        self.go = self.out.grid()
        n = len(self.segs)
        self.sg = (mg_grid * n)(*[t.grid() for t, _ in self.segs])
        self.sm = (C.c_int32 * n)(*[m for _, m in self.segs])
        self.dp = mg_dropout(self.p, self.ordinal, E.dropout_rank, E.dropout_seed, self.step_op.step.data_ptr())

    def io_fwd(self):
        return _keys(self.step_op.step, *[t.buf for t, _ in self.segs]), _keys(self.out.buf)

    def fwd(self, E):
        E.ctx.call("mg_dropout_forward", C.byref(self.dp), len(self.segs), self.sg, self.sm, C.byref(self.go))

    def setup_bwd(self, E):
        t = self.out
        self.comb = None
        if t.needs_grad:
            self.comb = Combine(E, t)   # usually an alias of the consuming conv's dcat
            self.dg = self.comb.grid()
            off = 0
            for p, m in self.segs:
                if p.needs_grad:
                    p.srcs.append(Src(self.comb.buf, t.H, t.W, t.C, t.Cp, off, m))
                off += p.C

    def backward_units(self):
        if self.comb is None:
            return super().backward_units()
        return [Unit(self, _merge(self.comb.io(), (_keys(self.step_op.step, self.comb.buf), _keys(self.comb.buf))), self.backward, BWD)]

    def backward(self, E, params):
        self.comb.run()
        E.ctx.call("mg_dropout_backward", C.byref(self.dp), C.byref(self.dg))


class GlobalAvgOp(Op):
    """SelectTable(1) -> cudnn.SpatialAveragePooling(7,7,1,1) on the 7x7 grid (ilsvrc/rnmg.lua:281-282)"""

    def __init__(self, inp, out):
        self.inp, self.out = inp, out
        out.producer = self

    def setup_fwd(self, E):
        self.out.buf = E.alloc(self.out.shape())
        self.gi, self.go = self.inp.grid(), self.out.grid()

    def io_fwd(self):
        return _keys(self.inp.buf), _keys(self.out.buf)

    def fwd(self, E):
        E.ctx.call("mg_global_avgpool_forward", C.byref(self.gi), C.byref(self.go))

    def setup_bwd(self, E):
        self.comb = Combine(E, self.out)
        self.din = E.alloc(self.inp.shape())
        self.dg_out, self.dg_in = self.comb.grid(), self.inp.grid(self.din)
        self.inp.srcs.append(Src(self.din, self.inp.H, self.inp.W, self.inp.C, self.inp.Cp, 0, MG_SEG_SAME))

    def backward_units(self):
        return [Unit(self, _merge(self.comb.io(), (_keys(self.comb.buf), _keys(self.din))), self.backward, BWD)]

    def backward(self, E, params):
        self.comb.run()
        E.ctx.call("mg_global_avgpool_backward", C.byref(self.dg_out), C.byref(self.dg_in))


class LogSoftMaxOp(Op):
    def __init__(self, inp):
        self.inp = inp

    def setup_fwd(self, E):
        self.result = torch.empty((self.inp.N, self.inp.C), dtype=torch.float32, device=E.device)
        self.gi = self.inp.grid()

    def size(self):
        return self.inp.H

    def io_fwd(self):
        return _keys(self.inp.buf), _keys(self.result)

    def fwd(self, E):
        E.ctx.call("mg_logsoftmax_forward", C.byref(self.gi), ptr(self.result))

    def setup_bwd(self, E):
        self.dl = E.alloc(self.inp.shape())
        self.dlg = self.inp.grid(self.dl)
        self.inp.srcs.append(Src(self.dl, 1, 1, self.inp.C, self.inp.Cp, 0, MG_SEG_SAME))
        self.grad_out = None

    def backward_units(self):
        return [Unit(self, (_keys(self.result), _keys(self.dl)), self.backward, BWD)]

    def backward(self, E, params):
        E.ctx.call("mg_logsoftmax_backward", ptr(self.result), ptr(self.grad_out), C.byref(self.dlg))


class SigmoidOp(Op):
    def __init__(self, inp):
        self.inp = inp

    def setup_fwd(self, E):
        t = self.inp
        self.result = torch.empty((t.N, t.C, t.H, t.W), dtype=torch.float32, device=E.device)
        self.gi = t.grid()

    def size(self):
        return self.inp.H

    def io_fwd(self):
        return _keys(self.inp.buf), _keys(self.result)

    def fwd(self, E):
        E.ctx.call("mg_sigmoid_forward", C.byref(self.gi), ptr(self.result))

    def setup_bwd(self, E):
        t = self.inp
        self.dx = E.alloc(t.shape())
        self.dxg = t.grid(self.dx)
        t.srcs.append(Src(self.dx, t.H, t.W, t.C, t.Cp, 0, MG_SEG_SAME))
        self.grad_out = None

    def backward_units(self):
        return [Unit(self, (_keys(self.result), _keys(self.dx)), self.backward, BWD)]

    def backward(self, E, params):
        E.ctx.call("mg_sigmoid_backward", ptr(self.result), ptr(self.grad_out), C.byref(self.dxg))


class ExportOp(Op):
    """a raw activation grid returned at the Torch boundary as NCHW fp32 (unit tests of single
    mg stages; whole networks end in LogSoftMax / Sigmoid)"""

    def __init__(self, inp):
        self.inp = inp

    def setup_fwd(self, E):
        t = self.inp
        self.result = torch.empty((t.N, t.C, t.H, t.W), dtype=torch.float32, device=E.device)
        self.gi = t.grid()

    def size(self):
        return self.inp.H

    def io_fwd(self):
        return _keys(self.inp.buf), _keys(self.result)

    def fwd(self, E):
        E.ctx.call("mg_export_nchw", C.byref(self.gi), ptr(self.result))

    def setup_bwd(self, E):
        t = self.inp
        self.dx = E.alloc(t.shape())
        self.dxg = t.grid(self.dx)
        t.srcs.append(Src(self.dx, t.H, t.W, t.C, t.Cp, 0, MG_SEG_SAME))
        self.grad_out = None

    def backward_units(self):
        return [Unit(self, ([], _keys(self.dx)), self.backward, BWD)]

    def backward(self, E, params):
        E.ctx.call("mg_import_nchw", ptr(self.grad_out), C.byref(self.dxg))
