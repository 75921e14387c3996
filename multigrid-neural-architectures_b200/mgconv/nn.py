"""Torch7-`nn`-shaped module vocabulary of the reference's model builders, backed by libmgconv.

The reference assembles its multigrid networks from stock Torch7 containers and layers
(models/ilsvrc/rnmg.lua:41-224, models/cifar/*.lua, models/mnist-cluttered/*.lua,
layers/ConcatUnet.lua).  This module offers the same constructors, so the builder code in
mgconv/builders.py reads like the Lua it mirrors -- but a model built from them is *lowered*:
on the first forward() the module graph is traced symbolically (lower.py) into a flat plan of
fused C-ABI calls (engine.py).  Max-pool / up-sample / JoinTable never materialise a
concatenated tensor: they become segment descriptors of the consuming convolution; BN, ReLU,
the zero-padded shortcut and CAddTable become the conv's epilogue pass.

Module protocol kept from Torch7 (SURVEY.md section 8b): forward(input), backward(input,
gradOutput), parameters(), getParameters(), zeroGradParameters(), training(), evaluate(),
findModules(typename), listModules(), apply(fn), cuda(), clearState(); fields .output,
.gradInput, .train.  Tensors at the boundary are torch CUDA tensors, NCHW fp32, as the
reference's put2GPU leaves them (utils/utilfuncs.lua:3-30).
"""
import math
import torch

from . import lower as L

MAX_ENGINES = 3   # lowered plans (with their activation buffers) kept per top-level module, one per input shape


# ------------------------------------------------------------------------------------
class Module:
    typename = "nn.Module"

    def __init__(self):
        self.train = True
        self.output = None
        self.gradInput = None
        self._engine = None
        self._dropouts = None

    # ---- graph walking ----------------------------------------------------------------
    def children(self):
        return []

    def listModules(self):
        out = [self]
        for c in self.children():
            out.extend(c.listModules())
        return out

    def findModules(self, typename):
        return [m for m in self.listModules() if m.typename == typename]

    def apply(self, fn):
        for m in self.listModules():
            fn(m)
        return self

    def training(self):
        return self.apply(lambda m: setattr(m, "train", True))

    def evaluate(self):
        return self.apply(lambda m: setattr(m, "train", False))

    # ---- parameters -------------------------------------------------------------------
    def own_parameters(self):
        """[(name, tensor, grad tensor)] of this module only"""
        return []

    def parameters(self):
        ws, gs = [], []
        for m in self.listModules():
            for _, w, g in m.own_parameters():
                ws.append(w)
                gs.append(g)
        return ws, gs

    def getParameters(self):
        """Flatten every parameter into one storage and re-point the modules at views of it,
        like Torch7's Module:getParameters() (pipelines/standard/train.lua:115)."""
        mods = [m for m in self.listModules() if m.own_parameters()]
        total = sum(w.numel() for m in mods for _, w, _ in m.own_parameters())
        ws, _ = self.parameters()
        dev = ws[0].device if ws else torch.device("cpu")
        flat = torch.zeros(total, dtype=torch.float32, device=dev)
        gflat = torch.zeros(total, dtype=torch.float32, device=dev)
        off = 0
        for m in mods:
            for name, w, g in m.own_parameters():
                n = w.numel()
                flat[off:off + n].copy_(w.reshape(-1))
                gflat[off:off + n].copy_(g.reshape(-1))
                setattr(m, name, flat[off:off + n].view(w.shape))
                setattr(m, "grad" + name[0].upper() + name[1:], gflat[off:off + n].view(w.shape))
                off += n
        self._flat = (flat, gflat)
        self.clearState()  # raw pointers changed: plans are rebuilt lazily
        return flat, gflat

    def zeroGradParameters(self):
        if getattr(self, "_flat", None) is not None:
            self._flat[1].zero_()
        else:
            for g in self.parameters()[1]:
                g.zero_()

    def _move(self, fn):
        for m in self.listModules():
            for k, v in list(vars(m).items()):
                if isinstance(v, torch.Tensor):
                    setattr(m, k, fn(v))
        self._flat = None
        self.clearState()
        return self

    def cuda(self, device=None):
        dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        return self._move(lambda t: t.to(dev))

    def float(self):
        return self._move(lambda t: t.cpu())

    def clearState(self):
        for m in self.listModules():
            m._engine = None
            m._engines = None
            m._dropouts = None
            m.output = None
            m.gradInput = None
        return self

    # ---- execution (top-level module only) ----------------------------------------------
    def _get_engine(self, input):
        from .engine import Engine
        from .engine import engine_key
        if self._dropouts is None:   # found once: the key is computed on every forward
            self._dropouts = self.findModules("nn.Dropout")
        key = engine_key(input, self._dropouts)
        if self._engine is None or self._engine.key != key:
            # plans are kept per input shape (most recent MAX_ENGINES): the reference's loop alternates between the training
            # batch and the partial last batch of the test pass (pipelines/standard/test.lua:40-44) every epoch
            cache = getattr(self, "_engines", None)
            if cache is None:
                cache = self._engines = {}
            eng = cache.pop(key, None)
            if eng is None:
                eng = Engine(self, input)
                while len(cache) >= MAX_ENGINES:
                    cache.pop(next(iter(cache)))
            cache[key] = eng      # most recently used last
            self._engine = eng
        return self._engine

    def forward(self, input):
        eng = self._get_engine(input)
        self.output = eng.forward(input, self.train)
        return self.output

    updateOutput = forward

    def backward(self, input, gradOutput, scale=1.0):
        eng = self._engine if input is None else self._get_engine(input)
        self.gradInput = eng.backward(gradOutput, scale)
        return self.gradInput

    # ---- symbolic trace ---------------------------------------------------------------
    def trace(self, x, b):
        raise NotImplementedError(f"{self.typename}: not lowerable")


# ------------------------------------------------------------------------------------ containers
class Container(Module):
    def __init__(self):
        super().__init__()
        self.modules = []

    def add(self, m):
        self.modules.append(m)
        return self

    def get(self, i):  # 1-based like Lua
        return self.modules[i - 1]

    def size(self):
        return len(self.modules)

    def children(self):
        return self.modules


class Sequential(Container):
    typename = "nn.Sequential"

    def trace(self, x, b):
        for m in self.modules:
            x = m.trace(x, b)
        return x


class ConcatTable(Container):
    """same input to every branch; backward sums the branches' gradInputs"""
    typename = "nn.ConcatTable"

    def trace(self, x, b):
        return [m.trace(x, b) for m in self.modules]


class ParallelTable(Container):
    typename = "nn.ParallelTable"

    def trace(self, x, b):
        assert len(x) == len(self.modules), f"ParallelTable: {len(x)} inputs for {len(self.modules)} modules"
        return [m.trace(x[i], b) for i, m in enumerate(self.modules)]


class MapTable(Container):
    typename = "nn.MapTable"

    def __init__(self, m=None):
        super().__init__()
        if m is not None:
            self.add(m)

    def trace(self, x, b):
        return [self.modules[0].trace(e, b) for e in x]


class SelectTable(Module):
    typename = "nn.SelectTable"

    def __init__(self, index):
        super().__init__()
        self.index = index

    def trace(self, x, b):
        return x[self.index - 1] if self.index > 0 else x[self.index]


class JoinTable(Module):
    typename = "nn.JoinTable"

    def __init__(self, dimension, nInputDims=None):
        super().__init__()
        assert dimension == 2, "only the channel concat JoinTable(2) of the builders is lowered"

    def trace(self, x, b):
        return b.cat(list(x))


class FlattenTable(Module):
    typename = "nn.FlattenTable"

    def trace(self, x, b):
        out = []

        def rec(t):
            if isinstance(t, (list, tuple)):
                for e in t:
                    rec(e)
            else:
                out.append(t)
        rec(x)
        return out


class CAddTable(Module):
    typename = "nn.CAddTable"

    def __init__(self, inplace=False):
        super().__init__()

    def trace(self, x, b):
        assert len(x) == 2, "CAddTable: the builders only add {conv branch, shortcut}"
        return b.add(x[0], x[1])


class Identity(Module):
    typename = "nn.Identity"

    def trace(self, x, b):
        return x


class Padding(Module):
    """nn.Padding(1, pad, 3): zero channels appended after the last one (ilsvrc/rnmg.lua:16)"""
    typename = "nn.Padding"

    def __init__(self, dim, pad, nInputDim):
        super().__init__()
        assert dim == 1 and nInputDim == 3 and pad > 0
        self.pad = pad

    def trace(self, x, b):
        return L.PadVal(x, self.pad)


class View(Module):
    typename = "nn.View"

    def __init__(self, *sizes):
        super().__init__()
        self.sizes = sizes

    def trace(self, x, b):
        v = b.resolve(x)
        assert v.H == 1 and v.W == 1 and self.sizes[-1] == v.C, "View: only the (-1, nFeatures) flatten of the classifier"
        return v


class ConcatUnet(Module):
    """layers/ConcatUnet.lua:1-37: {shortcut{t1..tn}, subnet{p1..pm}}, m <= n
    -> {{t1,p1}, ..., {tm,pm}, {t(m+1)}, ...}; pure table reshuffle, gradients zip back."""
    typename = "nn.ConcatUnet"

    def trace(self, x, b):
        assert len(x) == 2, "ConcatUnet expects {shortcut table, subnet table}"
        shortcut, subnet = x
        assert len(shortcut) >= len(subnet), "ConcatUnet: subnet table longer than shortcut table"
        out = []
        for i, t in enumerate(shortcut):
            e = [t]
            if i < len(subnet):
                e.append(subnet[i])
            out.append(e)
        return out


# ------------------------------------------------------------------------------------ layers
class SpatialConvolution(Module):
    typename = "cudnn.SpatialConvolution"  # what model:findModules() is asked for (ilsvrc/rnmg.lua:302)

    def __init__(self, nInputPlane, nOutputPlane, kW, kH, dW=1, dH=1, padW=0, padH=0):
        super().__init__()
        assert kW == kH and dW == dH and padW == padH, "square kernels only (all builders)"
        self.nInputPlane, self.nOutputPlane = nInputPlane, nOutputPlane
        self.kW = self.kH = kW
        self.dW = self.dH = dW
        self.padW = self.padH = padW
        self.weight = torch.empty(nOutputPlane, nInputPlane, kH, kW)
        self.bias = torch.empty(nOutputPlane)
        self.gradWeight = torch.zeros_like(self.weight)
        self.gradBias = torch.zeros_like(self.bias)
        self.reset()

    def reset(self, stdv=None):  # torch7 SpatialConvolution:reset()
        stdv = stdv or 1.0 / math.sqrt(self.kW * self.kH * self.nInputPlane)
        self.weight.uniform_(-stdv, stdv)
        self.bias.uniform_(-stdv, stdv)

    def own_parameters(self):
        return [("weight", self.weight, self.gradWeight), ("bias", self.bias, self.gradBias)]

    def trace(self, x, b):
        return b.conv(self, x)


class SpatialFullConvolution(Module):
    """cudnn.SpatialFullConvolution(nIP, nOP, 2,2, 2,2, 0,0): learned 2x up-sampling (unmg.lua:35-41)"""
    typename = "cudnn.SpatialFullConvolution"

    def __init__(self, nInputPlane, nOutputPlane, kW, kH, dW, dH, padW=0, padH=0):
        super().__init__()
        assert (kW, kH, dW, dH, padW, padH) == (2, 2, 2, 2, 0, 0), "only the 2x2 stride-2 up-convolution of U-MG is lowered"
        self.nInputPlane, self.nOutputPlane = nInputPlane, nOutputPlane
        self.kW = self.kH = 2
        self.weight = torch.empty(nInputPlane, nOutputPlane, 2, 2)
        self.bias = torch.empty(nOutputPlane)
        self.gradWeight = torch.zeros_like(self.weight)
        self.gradBias = torch.zeros_like(self.bias)
        stdv = 1.0 / math.sqrt(kW * kH * nInputPlane)   # torch7 SpatialFullConvolution:reset()
        self.weight.uniform_(-stdv, stdv)
        self.bias.uniform_(-stdv, stdv)

    def own_parameters(self):
        return [("weight", self.weight, self.gradWeight), ("bias", self.bias, self.gradBias)]

    def trace(self, x, b):
        return b.upconv(self, x)


class Linear(Module):
    typename = "nn.Linear"

    def __init__(self, inputSize, outputSize):
        super().__init__()
        self.weight = torch.empty(outputSize, inputSize)
        self.bias = torch.empty(outputSize)
        self.gradWeight = torch.zeros_like(self.weight)
        self.gradBias = torch.zeros_like(self.bias)
        self.reset()
        # a Linear on N x C x 1 x 1 is a 1x1 convolution
        self.nInputPlane, self.nOutputPlane = inputSize, outputSize
        self.kW = self.kH = 1
        self.dW = self.dH = 1
        self.padW = self.padH = 0

    def reset(self, stdv=None):  # torch7 Linear:reset()
        stdv = stdv or 1.0 / math.sqrt(self.weight.shape[1])
        self.weight.uniform_(-stdv, stdv)
        self.bias.uniform_(-stdv, stdv)

    def own_parameters(self):
        return [("weight", self.weight, self.gradWeight), ("bias", self.bias, self.gradBias)]

    def trace(self, x, b):
        return b.conv(self, x)


class SpatialBatchNormalization(Module):
    typename = "nn.SpatialBatchNormalization"

    def __init__(self, nOutput, eps=1e-5, momentum=0.1, affine=True):
        super().__init__()
        assert affine
        self.eps, self.momentum = eps, momentum
        self.weight = torch.empty(nOutput).uniform_(0, 1)  # torch7 reset(): gamma ~ U(0,1), beta = 0
        self.bias = torch.zeros(nOutput)
        self.gradWeight = torch.zeros(nOutput)
        self.gradBias = torch.zeros(nOutput)
        self.running_mean = torch.zeros(nOutput)
        self.running_var = torch.ones(nOutput)

    def reset(self):  # torch7 BatchNormalization:reset()
        self.weight.uniform_(0, 1)
        self.bias.zero_()
        self.running_mean.zero_()
        self.running_var.fill_(1)

    def own_parameters(self):
        return [("weight", self.weight, self.gradWeight), ("bias", self.bias, self.gradBias)]

    def trace(self, x, b):
        return b.batchnorm(self, x)


class ReLU(Module):
    typename = "nn.ReLU"

    def __init__(self, inplace=False):
        super().__init__()

    def trace(self, x, b):
        return b.relu(x)


class Dropout(Module):
    typename = "nn.Dropout"

    def __init__(self, p=0.5):
        super().__init__()
        self.p = p

    def trace(self, x, b):
        """training: y = x * mask / (1 - p), a fresh mask per forward (the lowered plan's DropOp); evaluate(): y = x"""
        if not 0 <= self.p < 1:
            raise ValueError(f"nn.Dropout: p = {self.p} is outside [0, 1)")
        if self.p > 0 and self.train:
            return b.dropout(x, self.p)
        return x


class SpatialMaxPooling(Module):
    typename = "nn.SpatialMaxPooling"

    def __init__(self, kW, kH, dW, dH, padW=0, padH=0):
        super().__init__()
        self.cfg = (kW, kH, dW, dH, padW, padH)
        self.ceil_mode = False

    def ceil(self):
        self.ceil_mode = True
        return self

    def trace(self, x, b):
        if self.cfg == (2, 2, 2, 2, 0, 0) and self.ceil_mode:
            return b.pool2(x)
        if self.cfg == (3, 3, 2, 2, 1, 1) and not self.ceil_mode:
            return b.pool3(x)
        raise NotImplementedError(f"SpatialMaxPooling{self.cfg} ceil={self.ceil_mode}: not used by the builders")


class SpatialAveragePooling(Module):
    typename = "cudnn.SpatialAveragePooling"

    def __init__(self, kW, kH, dW=1, dH=1, padW=0, padH=0):
        super().__init__()
        assert kW == kH and dW == dH and padW == 0 and padH == 0
        self.k, self.d = kW, dW

    def trace(self, x, b):
        return b.avgpool(x, self.k, self.d)


class SpatialUpSamplingNearest(Module):
    typename = "nn.SpatialUpSamplingNearest"

    def __init__(self, scale):
        super().__init__()
        assert scale == 2
        self.scale_factor = scale

    def trace(self, x, b):
        return b.up2(x)


class LogSoftMax(Module):
    typename = "nn.LogSoftMax"

    def trace(self, x, b):
        return b.logsoftmax(x)


class Sigmoid(Module):
    typename = "nn.Sigmoid"

    def trace(self, x, b):
        return b.sigmoid(x)


# ------------------------------------------------------------------------------------ criteria
class Criterion:
    def __init__(self):
        self.output = 0.0
        self.gradInput = None


class ClassNLLCriterion(Criterion):
    """mean NLL on log-probabilities; targets are 1-based like Lua (dataset labels 1..nClass)"""

    def __init__(self):
        super().__init__()
        self._loss = None

    def forward(self, input, target):
        from .engine import criterion_ctx
        from .ffi import ptr
        ctx = criterion_ctx(input)
        if self._loss is None or self._loss.device != input.device:
            self._loss = torch.zeros(1, dtype=torch.float32, device=input.device)
        self._t0 = (target.to(input.device, non_blocking=True).to(torch.int32) - 1).contiguous()
        ctx.call("mg_memset_zero", ptr(self._loss), 4)
        ctx.call("mg_nll_criterion", ptr(input), ptr(self._t0), input.shape[0], input.shape[1], ptr(self._loss), None, 1.0)
        self.output = self._loss
        return self.output

    def backward(self, input, target, gscale=1.0):
        from .engine import criterion_ctx
        from .ffi import ptr
        ctx = criterion_ctx(input)
        if self.gradInput is None or self.gradInput.shape != input.shape:
            self.gradInput = torch.empty_like(input)
        t0 = (target.to(input.device, non_blocking=True).to(torch.int32) - 1).contiguous()
        ctx.call("mg_nll_criterion", ptr(input), ptr(t0), input.shape[0], input.shape[1], None, ptr(self.gradInput), float(gscale))
        return self.gradInput


class BCECriterion(Criterion):
    def __init__(self):
        super().__init__()
        self._loss = None

    def forward(self, input, target):
        from .engine import criterion_ctx
        from .ffi import ptr
        ctx = criterion_ctx(input)
        if self._loss is None or self._loss.device != input.device:
            self._loss = torch.zeros(1, dtype=torch.float32, device=input.device)
        t = target.to(input.device, torch.float32).contiguous()
        ctx.call("mg_memset_zero", ptr(self._loss), 4)
        ctx.call("mg_bce_criterion", ptr(input), ptr(t), input.numel(), ptr(self._loss), None, 1.0)
        self.output = self._loss
        return self.output

    def backward(self, input, target, gscale=1.0):
        from .engine import criterion_ctx
        from .ffi import ptr
        ctx = criterion_ctx(input)
        if self.gradInput is None or self.gradInput.shape != input.shape:
            self.gradInput = torch.empty_like(input)
        t = target.to(input.device, torch.float32).contiguous()
        ctx.call("mg_bce_criterion", ptr(input), ptr(t), input.numel(), None, ptr(self.gradInput), float(gscale))
        return self.gradInput


class MultiCriterion(Criterion):
    """weighted sum of criteria (model.lua:39-44 wraps the net's criterion with weight 1/iterSize)"""

    def __init__(self):
        super().__init__()
        self.criterions, self.weights = [], []

    def add(self, criterion, weight=1.0):
        self.criterions.append(criterion)
        self.weights.append(weight)
        return self

    def forward(self, input, target):
        self.output = sum(w * c.forward(input, target) for c, w in zip(self.criterions, self.weights))
        return self.output

    def backward(self, input, target):
        assert len(self.criterions) == 1, "MultiCriterion: the reference only ever wraps one criterion"
        self.gradInput = self.criterions[0].backward(input, target, self.weights[0])
        return self.gradInput
