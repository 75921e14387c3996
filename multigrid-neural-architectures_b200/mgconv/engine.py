"""Plan executor: lowers a module graph for one input shape, owns every device buffer, and
replays the plan's C-ABI calls for forward and backward on the caller's CUDA stream.

PyTorch is used for device memory (torch.zeros as the allocator), streams and, in
dataparallel.py, torch.distributed rendezvous -- all arithmetic is libmgconv's.
"""
import ctypes as C
import os
import torch

from . import ffi, lower, ops, sched

_PRECISION = {"bf16": (ffi.MG_BF16, torch.bfloat16), "fp32": (ffi.MG_F32, torch.float32)}
_IMPL = {"auto": ffi.MG_IMPL_AUTO, "simt": ffi.MG_IMPL_SIMT, "tcgen05": ffi.MG_IMPL_TCGEN05}
_crit_ctx = {}


def criterion_ctx(t):
    """context used by the criteria (dtype independent kernels), one per device"""
    if not t.is_cuda:
        raise ffi.MGError("criterion inputs must be CUDA tensors: the multigrid hot path has no CPU fallback")
    dev = t.device.index
    if dev not in _crit_ctx:
        _crit_ctx[dev] = ffi.Context(dev, 0, ffi.MG_F32)
    _crit_ctx[dev].set_stream(torch.cuda.current_stream(dev).cuda_stream)
    return _crit_ctx[dev]


def _flatten(x):
    if isinstance(x, (list, tuple)):
        out = []
        for e in x:
            out.extend(_flatten(e))
        return out
    return [x]


def engine_key(input, dropouts=(), batchnorms=(), training=True):
    """plans are kept per input shape and device; a model with an active nn.Dropout (`dropouts`: its nn.Dropout modules) also
    gets one plan per mode (training plans hold the dropout ops, evaluation plans are those of the same model without them).
    A training model whose BatchNorm modules (`batchnorms`) do not all train -- some frozen by bn:evaluate() -- gets one plan per
    pattern of frozen layers; models in one mode keep the key of their input alone."""
    ts = _flatten(input)
    key = (tuple(input.shape) if isinstance(input, torch.Tensor) else tuple(tuple(t.shape) for t in ts),
           ts[0].device.index)
    active = [m for m in dropouts if m.p > 0]
    if active:
        key += (any(m.train for m in active),)
    if training and not all(m.train for m in batchnorms):
        key += (("frozen_bn",) + tuple(i for i, m in enumerate(batchnorms) if not m.train),)
    return key


class Engine:
    def __init__(self, model, input):
        inputs = _flatten(input)
        for t in inputs:
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dim() == 4):
                raise ffi.MGError("forward() needs 4-D CUDA tensors (NCHW); there is no CPU fallback -- "
                                  "call model:cuda() and move the inputs with put2GPU first")
        self.model = model
        self.device = inputs[0].device
        self.key = engine_key(input, model.findModules("nn.Dropout"), model.findModules("nn.SpatialBatchNormalization"), model.train)
        precision = getattr(model, "precision", os.environ.get("MGCONV_PRECISION", "bf16"))
        self.dtype, self.elt = _PRECISION[precision]
        self.ctx = ffi.Context(self.device.index, torch.cuda.current_stream(self.device).cuda_stream, self.dtype)
        impl = getattr(model, "impl", os.environ.get("MGCONV_IMPL", "auto"))
        self.ctx.set_impl(_IMPL[impl])
        self.use_packed = self.dtype == ffi.MG_BF16 and impl != "simt"
        self.training = True
        self.bn_sync = 0   # 0 = per-replica BatchNorm statistics (the reference's DataParallelTable); N = sync over N ranks
        self.gscale = 1.0
        self.bytes = 0
        self.on_param_done = None
        # BatchNorm sums of the whole plan (mg_sum: deterministic fixed-point pairs of int64, see mgconv.h) live in two arenas
        # (forward: sum y, sum y^2; backward: sum d, sum d*y), each zeroed by ONE memset per pass instead of one per convolution
        self._sums = {"fwd": [torch.zeros(1 << 18, dtype=torch.int64, device=self.device), 0],
                      "bwd": [torch.zeros(1 << 18, dtype=torch.int64, device=self.device), 0]}
        self._pack_cache = None
        # per-layer choice of the 3x3 kernel variant by timing (cudnn.benchmark of the reference); MGCONV_AUTOTUNE=0 keeps the heuristics
        self.autotune = os.environ.get("MGCONV_AUTOTUNE", "1") != "0"
        self._tuned_fwd = self._tuned_bwd = False
        # per-scale chains of a stage on separate CUDA streams (sched.py); MGCONV_LANES=1 runs the serial plan
        self.n_lanes = max(1, min(4, int(os.environ.get("MGCONV_LANES", "3"))))
        self._units = {}    # pass -> its sched.Units in execution order (ops.Op.forward_unit / backward_units), built once per plan
        self._scheds = {}   # (pass, n_lanes) -> its lane schedule
        # split backward (updateGradInput / accGradParameters): forwards run so far, and the forward the last update_grad_input
        # differentiated -- acc_grad_parameters reads what that call left in the plan's buffers
        self.generation = 0
        self.grad_input_generation = None
        self._bn_jobs = None
        for m in model.listModules():
            for _, w, _ in m.own_parameters():
                if w.device != self.device:
                    raise ffi.MGError(f"{m.typename} parameters live on {w.device}, inputs on {self.device}: call model:cuda()")

        shapes = [tuple(t.shape) for t in inputs]
        b, out = lower.trace_model(model, shapes if isinstance(input, (list, tuple)) else shapes[0],
                                   bool(getattr(model, "needInputGrad", False)))
        self.out_struct = self._wrap_outputs(out, b)
        self.plan = b
        # Philox key of the plan's dropout masks, drawn from torch's default generator (torch.manual_seed fixes every mask)
        self.dropout_seed = 0
        if b.drops:
            lo, hi = torch.randint(0, 1 << 32, (2,), dtype=torch.int64).tolist()
            self.dropout_seed = lo | hi << 32
        self._dropout_rank = 0
        self.input_ops = [o for o in b.ops if isinstance(o, ops.InputOp)]
        self.conv_ops = [o for o in b.ops if isinstance(o, ops.ConvOp)]
        self.bn_ops = [o for o in b.ops if isinstance(o, ops.ApplyOp) and o.bn is not None]
        ops.fuse_stem_pool3(b.ops, self)
        for o in b.ops:
            o.setup_fwd(self)
        self._units["forward"] = [o.forward_unit() for o in b.ops]
        self._bwd_ready = False

    def _wrap_outputs(self, out, b):
        if isinstance(out, (list, tuple)):
            return [self._wrap_outputs(e, b) for e in out]
        if isinstance(out, lower.OutVal):
            return out.op
        if isinstance(out, lower.CatVal):
            out = b.as_tensor(out)
        if isinstance(out, lower.TVal):
            return b.emit(ops.ExportOp(out.spec))
        raise NotImplementedError(f"model output of kind {type(out).__name__}")

    def alloc(self, shape, dtype=None):
        t = torch.zeros(shape, dtype=dtype or self.elt, device=self.device)
        self.bytes += t.numel() * t.element_size()
        return t

    def alloc_sums(self, n, which):
        """n deterministic sums (mg_sum = two int64 each)"""
        arena = self._sums[which]
        n2 = 2 * n
        n8 = (n2 + 7) // 8 * 8
        if arena[1] + n8 > arena[0].numel():
            raise ffi.MGError("BatchNorm statistics arena exhausted")
        v = arena[0][arena[1]:arena[1] + n2]
        arena[1] += n8
        return v

    def zero_sums(self, which):
        arena = self._sums[which]
        if arena[1]:
            self.ctx.call("mg_memset_zero", ffi.ptr(arena[0]), arena[1] * 8)

    def param_done(self, mod):
        if self.on_param_done is not None:
            self.on_param_done(mod)

    def _report_tuning(self, field):
        if os.environ.get("MGCONV_VERBOSE"):
            import collections
            names = {0: "heuristic", 1: "tile128", 2: "tile256", 3: "resident", 4: "tile128deep", 5: "tile256deep", 6: "tile128mid"}
            cnt = collections.Counter((o.H, o.CcatP, o.Cout, names[getattr(o.desc, field)]) for o in self.conv_ops if o._tunable())
            print(f"[mgconv] autotune {field}: " + ", ".join(f"{h}x{h} {ci}->{co}: {a} x{n}" for (h, ci, co, a), n in sorted(cnt.items())), flush=True)

    def set_bn_sync(self, nranks):
        """0 = per-replica BatchNorm statistics (the reference's DataParallelTable), N = statistics over N equal shards"""
        self.bn_sync = int(nranks)

    @property
    def dropout_rank(self):
        """data-parallel rank: a word of the dropout mask counter, so that shards draw different masks"""
        return self._dropout_rank

    @dropout_rank.setter
    def dropout_rank(self, rank):
        self._dropout_rank = int(rank)
        for o in self.plan.drops:
            o.dp.rank = self._dropout_rank

    def _use_lanes(self):
        # cross-replica BatchNorm issues NCCL calls from inside the chains: those must stay on one stream
        return self.n_lanes > 1 and not self.bn_sync

    def _bind_stream(self):
        self.ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- execution ------------------------------------------------------------------------
    def pack_weights(self):
        """fp32 master weights -> bf16 operand images of every convolution, one launch for the whole plan"""
        jobs = [j for o in self.conv_ops for j in o.pack_jobs()]
        if not jobs:
            return
        key = tuple((id(d), w.data_ptr(), wp.data_ptr(), t) for d, w, wp, t in jobs)
        if self._pack_cache is None or self._pack_cache[0] != key:
            n = len(jobs)
            descs = (C.POINTER(ffi.mg_conv_desc) * n)(*[C.pointer(d) for d, _, _, _ in jobs])
            ws = (C.c_void_p * n)(*[w.data_ptr() for _, w, _, _ in jobs])
            wps = (C.c_void_p * n)(*[wp.data_ptr() for _, _, wp, _ in jobs])
            tr = (C.c_int32 * n)(*[t for _, _, _, t in jobs])
            self._pack_cache = (key, n, descs, ws, wps, tr)
        _, n, descs, ws, wps, tr = self._pack_cache
        self.ctx.call("mg_conv_pack_weights_batched", n, descs, ws, wps, tr)

    def forward(self, input, training=True):
        self._bind_stream()
        self.training = training
        self.generation += 1
        # a BatchNorm trains only when the model trains and its own module does (Torch7: bn:evaluate() inside model:training());
        # a frozen one normalises with its running statistics, leaves them alone, and is differentiated as that fixed affine
        for o in self.bn_ops:
            o.frozen = not (training and o.bn.train)
        for op, t in zip(self.input_ops, _flatten(input)):
            op.src = t.contiguous().float()
        self.pack_weights()
        if self.autotune and not self._tuned_fwd and self.use_packed and not torch.cuda.is_current_stream_capturing():
            self._tuned_fwd = True
            for o in self.conv_ops:
                o.tune_fwd(self)
            self._report_tuning("algo_fwd")
        self.zero_sums("fwd")
        self._run("forward")
        return self._results(self.out_struct)

    def _run(self, name):
        """run pass `name` ("forward", "backward", "update" or "acc") from its units: on the lanes, else serially, under
        -bnSync with one all-reduce of the BatchNorm sums per run of consecutive ApplyOps"""
        units, params = self._units[name], name != "update"
        if self._use_lanes():
            s = self._scheds.get((name, self.n_lanes))
            if s is None:
                # weight gradients (nothing but the optimiser waits for them) fill a background lane beside the chains of
                # backward; in accGradParameters they are all there is, and spread over the lanes by size
                bg = self.n_lanes if name == "backward" and self.n_lanes < 4 else None
                base = 0 if name == "forward" else len(self.plan.ops) + 16   # backward event ids follow the forward's
                s = self._scheds[name, self.n_lanes] = sched.Schedule(units, lambda u: u.io, lambda u: u.run, self.n_lanes, base, bg)
            s.run(self, params)
        elif self.bn_sync:
            self._run_sync_bn(units, name == "forward", params)
        else:
            for u in units:
                u.run(self, params)

    # ---- cross-replica BatchNorm: one all-reduce per STAGE ----------------------------------------------------------
    # The plan lists a stage as [conv of every scale ..., apply of every scale ...] and the statistics of consecutive layers
    # are consecutive slices of one arena, so the sums of all scales of a stage travel in ONE in-stream all-reduce instead of
    # one per BatchNorm layer (R-MG-34: 2 x 27 collectives per step instead of 2 x 75).
    def _allreduce_sums(self, tensors):
        """all-reduce the arena range spanned by `tensors` (int64 limbs of mg_sum); False if they are not one compact range"""
        if not tensors:
            return True
        lo = min(t.data_ptr() for t in tensors)
        hi = max(t.data_ptr() + t.numel() * 8 for t in tensors)
        padded = sum((t.numel() + 7) // 8 * 8 for t in tensors)
        if (hi - lo) // 8 > padded:
            return False
        self.ctx.call("mg_allreduce_inline", C.c_void_p(lo), (hi - lo) // 8, 2)
        return True

    def _run_sync_bn(self, units, fwd, params):
        """params = False: the backward of update_grad_input (no parameter gradients).  An evaluate() forward all-reduces
        nothing: every BatchNorm is frozen."""
        i, n = 0, len(units)
        while i < n:
            if not isinstance(units[i].op, ops.ApplyOp):
                units[i].run(self, params)
                i += 1
                continue
            j = i
            while j < n and isinstance(units[j].op, ops.ApplyOp):
                j += 1
            run = [u.op for u in units[i:j]]
            if fwd:
                synced = self._allreduce_sums([a.conv.sums for a in run if a.bn is not None and not a.frozen])
                for a in run:
                    a.fwd(self, synced=synced)
            else:
                for a in run:
                    a.bwd_combine(self)
                synced = self._allreduce_sums([a.dsums for a in run if a.bn is not None and not a.frozen])
                for a in run:
                    a.bwd_bn(self, synced=synced, params=params)
            i = j

    def _results(self, s):
        if isinstance(s, list):
            return [self._results(e) for e in s]
        return s.result

    def _setup_bwd(self):
        for o in reversed(self.plan.ops):
            o.setup_bwd(self)
        units = [u for o in reversed(self.plan.ops) for u in o.backward_units()]
        for name in ("backward", "update", "acc"):
            self._units[name] = [u for u in units if name in u.passes]
        self._bwd_ready = True

    def _begin_backward(self, gradOutput):
        self._bind_stream()
        if not self._bwd_ready:
            self._setup_bwd()
            self.pack_weights()  # transposed images for dgrad were allocated just now
        for op, g in zip(_flatten(self.out_struct), _flatten(gradOutput)):
            op.grad_out = g.contiguous().float()
        if self.autotune and not self._tuned_bwd and self.use_packed and not torch.cuda.is_current_stream_capturing():
            self._tuned_bwd = True
            for o in self.conv_ops:
                o.tune_bwd(self)
            self._report_tuning("algo_bwd_data")
        self.zero_sums("bwd")

    def _grad_input(self):
        gi = [op.grad_nchw for op in self.input_ops]
        if all(g is None for g in gi):
            return None
        return gi if len(gi) > 1 else gi[0]

    def backward(self, gradOutput, scale=1.0):
        self.gscale = float(scale)
        self._begin_backward(gradOutput)
        self.grad_input_generation = None   # the buffers now hold this backward's gradient
        self._run("backward")
        return self._grad_input()

    # ---- backward in the two phases of the nn protocol --------------------------------------------------------------
    # update_grad_input runs everything backward() runs except the parameter gradients: the data gradients, the dgrad half of
    # every convolution, BatchNorm with no dgamma / dbeta / gradBias output.  The BatchNorm sums (the "bwd" arena) and every
    # gradient grid stay where they are, and acc_grad_parameters turns them into the parameter gradients: one batched BatchNorm
    # launch (mg_bn_param_grad), then the wgrad half of every convolution.  Each buffer gets the same writes in the same order
    # as in backward(), so the pair leaves backward's bits.
    def update_grad_input(self, gradOutput):
        self._begin_backward(gradOutput)
        # under -bnSync the data gradient needs the global (sum d, sum d*y): the all-reduce of the sums belongs to this phase
        self._run("update")
        self.grad_input_generation = self.generation
        return self._grad_input()

    def acc_grad_parameters(self, scale=1.0):
        if self.grad_input_generation != self.generation:
            raise ffi.MGError("accGradParameters: no updateGradInput since the last forward -- it adds the parameter gradients "
                              "of the gradOutput given to the last updateGradInput of the current forward")
        self._bind_stream()
        self.gscale = float(scale)
        if self.bn_ops:
            n = len(self.bn_ops)
            if self._bn_jobs is None:
                self._bn_jobs = (ffi.mg_bn_param_job * n)()
            for o, j in zip(self.bn_ops, self._bn_jobs):
                o.param_job(self, j)
            self.ctx.call("mg_bn_param_grad", n, self._bn_jobs)
            for o in self.bn_ops:
                self.param_done(o.bn)
        # a lane schedule starts behind everything on lane 0 (the update phase joined its lanes there, then the BatchNorm launch)
        self._run("acc")
