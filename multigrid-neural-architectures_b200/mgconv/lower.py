"""Symbolic lowering of a Torch7-style module graph (nn.py) to a flat plan of fused ops (ops.py).

Values flowing through the trace:
  TVal     a materialised NHWC tensor (TSpec)
  UpVal    SpatialUpSamplingNearest(2) of a TVal -- never materialised, becomes an UP segment
  CatVal   JoinTable(2) of values -- never materialised unless a shortcut needs it as one tensor
  NodeVal  output of a convolution whose epilogue (BN, ReLU, shortcut add, ReLU) is still being
           collected; `seal` turns it into a TVal by emitting the apply pass
  PadVal   nn.Padding(1, p, 3) of a value (only meaningful as the shortcut operand of CAddTable)
  DropVal  nn.Dropout(p) of a value in training mode -- materialised by a DropOp (the dropped concatenation of the value's
           segments) the first time a convolution or shortcut consumes it
  OutVal   fp32 network output at the Torch boundary (log-probabilities / probabilities)

max-pool 2x2/ceil of a tensor is its *pooled companion*: written by the producer's apply pass
(one extra quarter-size store) so that every convolution gathers by pure copies; pool and
up-sample distribute over JoinTable, so ResampleConcat (models/ilsvrc/rnmg.lua:41-89), mgPool
with isConcat (191-224) and ConcatUnet + MapTable(JoinTable) (unmg.lua:219-220) all reduce to
segment lists of the consuming convolution.
"""
from . import ops as O
from .ffi import MG_SEG_SAME, MG_SEG_UP, MG_MAX_SEG


class Val:
    pass


class TVal(Val):
    def __init__(self, spec):
        self.spec = spec
    C = property(lambda s: s.spec.C)
    H = property(lambda s: s.spec.H)
    W = property(lambda s: s.spec.W)


class UpVal(Val):
    def __init__(self, src):
        self.src = src  # TVal
    C = property(lambda s: s.src.C)
    H = property(lambda s: 2 * s.src.H)
    W = property(lambda s: 2 * s.src.W)


class CatVal(Val):
    def __init__(self, parts):
        self.parts = parts
        h, w = parts[0].H, parts[0].W
        for p in parts:
            if (p.H, p.W) != (h, w):
                raise ValueError(f"JoinTable(2): inconsistent tensor sizes {[(q.H, q.W) for q in parts]}")
    C = property(lambda s: sum(p.C for p in s.parts))
    H = property(lambda s: s.parts[0].H)
    W = property(lambda s: s.parts[0].W)


class NodeVal(Val):
    """copy-on-extend: attaching an epilogue stage returns a NEW NodeVal and retires this one, so a
    value that two consumers try to continue differently is detected instead of silently fused"""

    def __init__(self, conv, bn=None, relu1=False, res=None, relu2=False):
        self.conv, self.bn, self.relu1, self.res, self.relu2 = conv, bn, relu1, res, relu2
        self.out = None      # TVal once sealed
        self.retired = False

    def extend(self, **kw):
        if self.retired or self.out is not None:
            raise NotImplementedError("a convolution output is continued by two different consumers "
                                      "(BN/ReLU/CAddTable after it was already used): not a pattern of the builders")
        self.retired = True
        d = dict(bn=self.bn, relu1=self.relu1, res=self.res, relu2=self.relu2)
        d.update(kw)
        return NodeVal(self.conv, **d)
    C = property(lambda s: s.conv.Cout)
    H = property(lambda s: s.conv.Ho)
    W = property(lambda s: s.conv.Wo)


class PadVal(Val):
    def __init__(self, src, pad):
        self.src, self.pad = src, pad
    C = property(lambda s: s.src.C + s.pad)
    H = property(lambda s: s.src.H)
    W = property(lambda s: s.src.W)


class DropVal(Val):
    def __init__(self, src, p):
        self.src, self.p = src, p
        self.out = None      # TVal once materialised
    C = property(lambda s: s.src.C)
    H = property(lambda s: s.src.H)
    W = property(lambda s: s.src.W)


class OutVal(Val):
    def __init__(self, op, shape):
        self.op, self.shape = op, shape


class Builder:
    """trace context: owns the plan (tensor specs + op list)"""

    def __init__(self, N):
        self.N = N
        self.tensors = []
        self.ops = []
        self.drops = []      # DropOps in plan order: their index is the `op` word of the mask counter
        self.drop_step = None

    # ---- tensors ------------------------------------------------------------------------
    def new_tensor(self, C, H, W, name, needs_grad=True):
        t = O.TSpec(len(self.tensors), self.N, C, H, W, name, needs_grad)
        self.tensors.append(t)
        return t

    def emit(self, op):
        self.ops.append(op)
        return op

    def input(self, C, H, W):
        t = self.new_tensor(C, H, W, "input", needs_grad=False)
        self.emit(O.InputOp(t))
        return TVal(t)

    # ---- value normalisation ----------------------------------------------------------------
    def seal(self, node):
        if node.out is not None:
            return node.out
        if node.retired:
            raise NotImplementedError("a convolution output is used both raw and through its BN/ReLU epilogue")
        conv = node.conv
        plain = node.bn is None and not node.relu1 and node.res is None and not node.relu2
        if plain:
            conv.y.name = conv.name + ".out"
            node.out = TVal(conv.y)
            return node.out
        if node.res is not None and node.relu1:
            raise NotImplementedError("ReLU between BatchNorm and CAddTable is not a pattern of the builders")
        out = self.new_tensor(conv.Cout, conv.Ho, conv.Wo, conv.name + ".act")
        relu = node.relu2 if node.res is not None else node.relu1
        self.emit(O.ApplyOp(conv, node.bn, relu, node.res.spec if node.res is not None else None, out))
        node.out = TVal(out)
        return node.out

    def resolve(self, v):
        return self.seal(v) if isinstance(v, NodeVal) else v

    def seal_all(self, x):
        if isinstance(x, (list, tuple)):
            return [self.seal_all(e) for e in x]
        return self.resolve(x)

    def as_tensor(self, v):
        """a single materialised tensor holding v (shortcut operands, pool3, heads)"""
        v = self.resolve(v)
        if isinstance(v, TVal):
            return v
        if isinstance(v, DropVal):
            return self.drop(v)
        if isinstance(v, CatVal):
            segs = self.segments(v)
            if any(m != MG_SEG_SAME for _, m in segs):
                raise NotImplementedError("materialising an up-sampled tensor is not needed by the builders")
            out = self.new_tensor(v.C, v.H, v.W, "cat", needs_grad=any(t.needs_grad for t, _ in segs))
            self.emit(O.CatOp([t for t, _ in segs], out))
            return TVal(out)
        raise NotImplementedError(f"cannot materialise {type(v).__name__}")

    def segments(self, v):
        v = self.resolve(v)
        if isinstance(v, TVal):
            return [(v.spec, MG_SEG_SAME)]
        if isinstance(v, UpVal):
            return [(v.src.spec, MG_SEG_UP)]
        if isinstance(v, DropVal):
            return [(self.drop(v).spec, MG_SEG_SAME)]
        if isinstance(v, CatVal):
            out = []
            for p in v.parts:
                out.extend(self.segments(p))
            return out
        raise NotImplementedError(f"{type(v).__name__} cannot feed a convolution")

    def drop(self, v):
        """the dropped concatenation of v's segments as one tensor (one mask shared by every consumer, like the output of
        a Torch7 nn.Dropout); the plan's step counter is advanced right before its first DropOp"""
        if v.out is None:
            segs = self.segments(v.src)
            if len(segs) > MG_MAX_SEG:
                raise NotImplementedError(f"nn.Dropout of {len(segs)} segments > MG_MAX_SEG")
            if self.drop_step is None:
                self.drop_step = self.emit(O.DropStepOp())
            out = self.new_tensor(v.C, v.H, v.W, f"drop{len(self.drops)}", needs_grad=any(t.needs_grad for t, _ in segs))
            self.drops.append(self.emit(O.DropOp(segs, v.p, len(self.drops), self.drop_step, out)))
            v.out = TVal(out)
        return v.out

    # ---- ops called by the modules ---------------------------------------------------------
    def dropout(self, v, p):
        v = self.resolve(v)
        if isinstance(v, (DropVal, PadVal, OutVal)):
            raise NotImplementedError(f"nn.Dropout of {type(v).__name__}: not a pattern of the builders")
        return DropVal(v, p)

    def cat(self, parts):
        parts = [self.resolve(p) for p in parts]
        return parts[0] if len(parts) == 1 else CatVal(parts)

    def pool2(self, v):
        v = self.resolve(v)
        if isinstance(v, TVal):
            return TVal(self.companion(v.spec))
        if isinstance(v, CatVal):
            return CatVal([self.pool2(p) for p in v.parts])
        if isinstance(v, UpVal):
            return v.src  # max over a 2x2 block of identical values
        raise NotImplementedError(f"max-pool of {type(v).__name__}")

    def companion(self, t):
        """maxpool2x2_ceil(t), materialised once per tensor"""
        if t.pooled is None:
            p = self.new_tensor(t.C, (t.H + 1) // 2, (t.W + 1) // 2, t.name + ".pool", needs_grad=t.needs_grad)
            t.pooled = p
            if isinstance(t.producer, O.ApplyOp) and t.producer.out is t:
                t.producer.pooled = p   # fused into the apply pass
                p.producer = t.producer
            else:
                self.emit(O.PoolOp(t, p))
        return t.pooled

    def up2(self, v):
        v = self.resolve(v)
        if isinstance(v, TVal):
            return UpVal(v)
        if isinstance(v, CatVal):
            return CatVal([self.up2(p) for p in v.parts])
        raise NotImplementedError(f"up-sampling of {type(v).__name__}")

    def pool3(self, v):
        t = self.as_tensor(v).spec
        out = self.new_tensor(t.C, (t.H - 1) // 2 + 1, (t.W - 1) // 2 + 1, t.name + ".pool3", needs_grad=t.needs_grad)
        self.emit(O.Pool3Op(t, out))
        return TVal(out)

    def avgpool(self, v, k, d):
        t = self.as_tensor(v).spec
        if k == d:  # image pyramid (ilsvrc/rnmg.lua:175-177): carries a gradient when the image does (needInputGrad)
            out = self.new_tensor(t.C, t.H // k, t.W // k, f"{t.name}.avg{k}", needs_grad=t.needs_grad)
            self.emit(O.AvgPoolOp(t, k, out))
            return TVal(out)
        if d == 1 and k == t.H and k == t.W:  # classifier head Avg(7,7,1,1) on the 7x7 grid (rnmg.lua:282)
            out = self.new_tensor(t.C, 1, 1, t.name + ".gap")
            self.emit(O.GlobalAvgOp(t, out))
            return TVal(out)
        raise NotImplementedError(f"SpatialAveragePooling({k},{k},{d},{d}) on a {t.H}x{t.W} grid")

    def conv(self, mod, v):
        segs = self.segments(v)
        if len(segs) > MG_MAX_SEG:
            raise NotImplementedError(f"{len(segs)} input segments > MG_MAX_SEG")
        v = self.resolve(v)
        cin = sum(t.C for t, _ in segs)
        if cin != mod.nInputPlane:
            raise ValueError(f"{mod.typename}: {cin} input planes, expected {mod.nInputPlane}")
        op = O.ConvOp(self, mod, segs, v.H, v.W, f"conv{len([o for o in self.ops if isinstance(o, O.ConvOp)])}")
        self.emit(op)
        return NodeVal(op)

    def upconv(self, mod, v):
        t = self.as_tensor(v).spec
        if t.C != mod.nInputPlane:
            raise ValueError(f"SpatialFullConvolution: {t.C} input planes, expected {mod.nInputPlane}")
        op = O.UpConvOp(self, mod, t, f"upconv{len([o for o in self.ops if isinstance(o, O.UpConvOp)])}")
        self.emit(op)
        return NodeVal(op)

    def batchnorm(self, mod, v):
        if not (isinstance(v, NodeVal) and v.out is None and v.bn is None and not v.relu1 and v.res is None):
            raise NotImplementedError("SpatialBatchNormalization must directly follow a convolution")
        return v.extend(bn=mod)

    def relu(self, v):
        if not (isinstance(v, NodeVal) and v.out is None):
            raise NotImplementedError("ReLU must follow a convolution / BatchNorm / CAddTable epilogue")
        return v.extend(relu2=True) if v.res is not None else v.extend(relu1=True)

    def add(self, a, b):
        if not (isinstance(a, NodeVal) and a.out is None) and isinstance(b, NodeVal) and b.out is None:
            a, b = b, a
        if not (isinstance(a, NodeVal) and a.out is None and a.res is None):
            raise NotImplementedError("CAddTable: one operand must be an open convolution branch")
        pad = 0
        if isinstance(b, PadVal):
            pad, b = b.pad, b.src
        s = self.as_tensor(b)
        if s.C + pad != a.C or (s.H, s.W) != (a.H, a.W):
            raise ValueError(f"CAddTable: shortcut {s.C}+{pad}x{s.H}x{s.W} vs branch {a.C}x{a.H}x{a.W}")
        return a.extend(res=s)

    def logsoftmax(self, v):
        t = self.as_tensor(v).spec
        assert t.H == 1 and t.W == 1
        op = self.emit(O.LogSoftMaxOp(t))
        return OutVal(op, (self.N, t.C))

    def sigmoid(self, v):
        t = self.as_tensor(v).spec
        op = self.emit(O.SigmoidOp(t))
        return OutVal(op, (self.N, t.C, t.H, t.W))


def trace_model(model, shapes, need_input_grad=False):
    """lower `model` for NCHW input shape(s) (a tuple, or a list of tuples for a table input).
    Pure host logic -- no device needed.  Returns (builder, output structure of Vals)."""
    table = isinstance(shapes, list)
    shp = shapes if table else [shapes]
    b = Builder(shp[0][0])
    vals = []
    for (n, c, h, w) in shp:
        v = b.input(c, h, w)
        v.spec.needs_grad = need_input_grad
        vals.append(v)
    out = model.trace(vals if table else vals[0], b)
    return b, b.seal_all(out)


def plan_summary(b):
    """structural facts of a lowered plan (used by the CPU tests against README.md:85-92,109)"""
    convs = [o for o in b.ops if isinstance(o, O.ConvOp)]
    macs = sum(sum(t.C for t, _ in o.segs) * o.Cout * o.k * o.k * o.Ho * o.Wo for o in convs)
    return {"convs": len(convs), "macs": macs, "ops": len(b.ops), "tensors": len(b.tensors),
            "max_segs": max(len(o.segs) for o in convs),
            "act_bytes_bf16": sum(t.N * t.H * t.W * t.Cp * 2 for t in b.tensors)}
