"""Data parallelism: the four global helpers of multigpu.lua (makeDataParallel:81,
saveDataParallel:105, loadDataParallel:137, loadAndRemoveDPT:150) on a process-per-GPU design.

The reference wraps the model in nn.DataParallelTable(1, true, true): one process, one Lua
thread per GPU, batch split ceil(B/nGPU) along dim 1, nccl.reduce of the flat gradient to GPU 1
after backward, SGD on GPU 1, nccl.bcast of the parameters (pipelines/standard/train.lua:163-169).
Here every rank owns a full replica and its shard of the batch; the flat gradient is cut into
buckets in reverse layer order and each bucket is all-reduced (ncclAllReduce through libmgconv,
over NVLink) on a side stream as soon as the last wgrad that writes into it has been enqueued,
overlapping the rest of backward; every rank then applies the same SGD step, so no broadcast is
needed after initialisation.  BN statistics stay per replica, as in the reference (multigpu.lua:38-41).
"""
import ctypes as C
import os
import torch
import torch.distributed as dist

from . import ffi
from .ffi import ptr

BUCKET_BYTES = int(os.environ.get("MGCONV_BUCKET_MB", "16")) << 20


def shard_range(B, nGPU, rank):
    """rows of a global batch owned by `rank`: DataParallelTable splits dim 1 into ceil(B/nGPU) chunks"""
    per = -(-B // nGPU)
    lo = min(B, rank * per)
    return lo, min(B, lo + per)


def plan_buckets(sizes, bucket_bytes=BUCKET_BYTES, elt=4):
    """cut the flat vector (parameter sizes in module order) into contiguous buckets, built from the
    END of the vector because backward produces gradients in reverse module order.
    Returns [(offset, count, first_param_index)] in launch order; a bucket is complete when the
    gradient of parameter `first_param_index` (its lowest-indexed member) has been written."""
    buckets, end, count = [], sum(sizes), 0
    off = end
    for i in range(len(sizes) - 1, -1, -1):
        off -= sizes[i]
        count += sizes[i]
        if count * elt >= bucket_bytes or i == 0:
            buckets.append((off, count, i))
            count = 0
    return buckets


class DataParallel:
    """stands where nn.DataParallelTable stood: same module protocol, local shard in, local
    outputs out; gradients are global sums divided by nothing -- the criterion already averages
    over the *global* batch through gscale = 1/nranks (equal shards)."""
    typename = "nn.DataParallelTable"

    def __init__(self, model, nGPU, group=None, bnSync=False):
        self.model = model
        self.bnSync = bool(bnSync)
        self.nGPU = nGPU
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        if self.world != nGPU:
            raise ffi.MGError(f"makeDataParallel: -nGPU {nGPU} but {self.world} ranks were launched "
                              "(one process per GPU: torchrun --nproc-per-node nGPU)")
        self.flat = self.gflat = None
        self.buckets = []
        self._comm = None          # ffi.Context that OWNS the NCCL communicator; engines borrow it (mg_comm_share)
        self._owner = {}
        self.needsSync = False
        self.train = True
        self._grads_clean = False  # True right after zeroGradParameters(): backward may all-reduce gflat in place
        self._gprev = None         # stash of the already reduced micro-batch gradients (-iterSize > 1)
        self._shards = {}          # local batch size -> (global batch size) agreed on by all ranks

    # ---- module protocol passthrough ----------------------------------------------------
    def __getattr__(self, name):
        return getattr(self.__dict__["model"], name)

    def listModules(self):
        return self.model.listModules()

    # methods of the wrapped model that return `self` must return the WRAPPER (model = model:cuda() keeps the DPT)
    def cuda(self, device=None):
        self.model.cuda(device)
        self.flat = self.gflat = None
        return self

    def float(self):
        self.model.float()
        self.flat = self.gflat = None
        return self

    def clearState(self):
        self.model.clearState()
        return self

    def zeroGradParameters(self):
        self.model.zeroGradParameters()
        self._grads_clean = True

    def training(self):
        self.train = True
        self.model.training()
        return self

    def evaluate(self):
        self.train = False
        self.model.evaluate()
        return self

    def getParameters(self):
        self.flat, self.gflat = self.model.getParameters()
        sizes, self._owner, idx = [], {}, 0
        for m in self.model.listModules():
            for name, w, _ in m.own_parameters():
                sizes.append(w.numel())
                self._owner.setdefault(id(m), []).append(idx)
                idx += 1
        self.sizes = sizes
        self.buckets = plan_buckets(sizes)
        self._trigger = {first: (off, cnt) for off, cnt, first in self.buckets}
        self.syncParameters()
        return self.flat, self.gflat

    def syncParameters(self):
        """nccl.bcast(root = GPU 1) of the flat parameter vector (train.lua:166-168): needed once,
        after initialisation / checkpoint load; afterwards every rank takes identical steps"""
        if self.world > 1 and self.flat is not None:
            if self.flat.is_cuda and dist.get_backend(self.group) == "gloo":
                tmp = self.flat.cpu()
                dist.broadcast(tmp, 0, group=self.group)
                self.flat.copy_(tmp)
            else:
                dist.broadcast(self.flat, 0, group=self.group)
        self.needsSync = False

    def _init_comm(self, eng):
        """one NCCL communicator per DataParallel, owned by a context of its own: engines are rebuilt whenever the
        input shape changes (the partial last batch of pipelines/standard/test.lua:40-44), the communicator is not"""
        if self.world == 1:
            return
        if self._comm is not None:
            if not getattr(eng, "_comm_shared", False):
                eng.ctx.call("mg_comm_share", self._comm.h)
                eng._comm_shared = True
            return
        self._comm = ffi.Context(eng.device.index, 0, ffi.MG_F32)
        uid = torch.zeros(128, dtype=torch.uint8)
        if self.rank == 0:
            ffi_rc = ffi.lib.mg_comm_unique_id(C.c_void_p(uid.data_ptr()))
            if ffi_rc != 0:
                raise ffi.MGError("mg_comm_unique_id failed (libnccl.so.2 not loadable?)")
        if dist.get_backend(self.group) == "nccl":
            u = uid.cuda()
            dist.broadcast(u, 0, group=self.group)
            uid = u.cpu()
        else:
            dist.broadcast(uid, 0, group=self.group)
        self._comm.call("mg_comm_init", self.rank, self.world, C.c_void_p(uid.data_ptr()))
        eng.ctx.call("mg_comm_share", self._comm.h)
        eng._comm_shared = True

    def _agree_on_shards(self, local_B):
        """DataParallelTable splits dim 1 into ceil(B/nGPU) chunks (multigpu.lua:87): shards may be unequal (B = 10 on 4 GPUs
        gives 3,3,3,1).  The criterion averages over the LOCAL shard, so a rank's gradient weighs local_B / global_B of the
        global-mean loss; cross-replica BatchNorm needs the global element count.  An empty shard cannot run."""
        if local_B not in self._shards:
            sizes = [torch.zeros(1, dtype=torch.int64) for _ in range(self.world)]
            mine = torch.tensor([local_B], dtype=torch.int64)
            if self.world > 1:
                if dist.get_backend(self.group) == "nccl":
                    dev = torch.device("cuda", torch.cuda.current_device())
                    sizes = [t.to(dev) for t in sizes]
                    dist.all_gather(sizes, mine.to(dev), group=self.group)
                else:
                    dist.all_gather(sizes, mine, group=self.group)
            else:
                sizes = [mine]
            sizes = [int(t.item()) for t in sizes]
            if min(sizes) <= 0:
                raise ffi.MGError(f"makeDataParallel: shard sizes {sizes}: a rank without images cannot take part in the step "
                                  "(global batch smaller than ceil(B/nGPU) * (nGPU-1) + 1)")
            self._shards[local_B] = (sum(sizes), len(set(sizes)) == 1)
        return self._shards[local_B]

    def _attach(self, eng, input):
        """bind a (new or cached) engine to this wrapper BEFORE it runs: dropout rank, bucket triggers, communicator, shard weights"""
        eng.dropout_rank = self.rank
        if self.world == 1:
            return
        ts = input
        while isinstance(ts, (list, tuple)):
            ts = ts[0]
        local_B = int(ts.shape[0])
        global_B, equal = self._agree_on_shards(local_B)
        if self.bnSync and not equal:
            # the BatchNorm backward mixes the gradients of all ranks; with unequal shards the criteria's 1/local_B
            # weights differ per rank and the mixed sums would be wrong
            raise ffi.MGError("-bnSync needs equal shards on every rank (global batch divisible by nGPU)")
        eng.shard = (local_B, global_B)
        self._init_comm(eng)
        if self.gflat is not None:
            eng.on_param_done = self._param_done
        eng.set_bn_sync(self.world if self.bnSync else 0)

    def forward(self, input):
        # -bnSync: BatchNorm statistics over the GLOBAL batch (one tiny all-reduce of the per-channel sums per BN
        # layer, forward and backward) -- equals the single-device result on the whole batch.  The engine is bound
        # before it runs, so the first forward already uses global statistics (no second running-statistics update).
        eng = self.model._get_engine(input)
        self._attach(eng, input)
        return self.model.forward(input)

    def backward(self, input, gradOutput, scale=1.0):
        eng = self.model._engine if input is None else self.model._get_engine(input)
        if self.world == 1 or self.gflat is None:
            return self.model.backward(input, gradOutput, scale)
        self._reset_buckets()
        # Gradient accumulation (-iterSize, model.lua:39-44; pipelines/standard/train.lua:147-169 zeroes the gradients only
        # before the first micro-batch): backward ACCUMULATES into gflat, so all-reducing gflat in place would sum the
        # already reduced earlier micro-batches once more per rank.  Unless the gradients were zeroed since the last
        # backward, set the reduced part aside, reduce only what this backward produces, and add it back.
        stash = not self._grads_clean
        self._grads_clean = False
        if stash:
            if self._gprev is None:
                self._gprev = torch.empty_like(self.gflat)
            self._gprev.copy_(self.gflat)
            self.gflat.zero_()
        local_B, global_B = getattr(eng, "shard", (1, self.world))
        gi = self.model.backward(input, gradOutput, scale * local_B / global_B)
        for b, (off, cnt, _) in enumerate(self.buckets):   # parameters the plan never touched
            if b not in self.launched:
                eng.ctx.call("mg_allreduce_launch", ptr(self.gflat[off:off + cnt]), cnt, 0)
        eng.ctx.call("mg_allreduce_wait")
        if stash:
            self.gflat.add_(self._gprev)
        return gi

    def _param_done(self, mod):
        """called by the engine right after the wgrad / BN-backward of `mod` was enqueued: a bucket whose
        last missing gradient this was is all-reduced now, overlapping the rest of backward"""
        eng = self.model._engine
        for idx in self._owner.get(id(mod), ()):
            if idx in self._done:
                continue
            self._done.add(idx)
            b = self._bucket_of[idx]
            self._missing[b] -= 1
            if self._missing[b] == 0:
                off, cnt, _ = self.buckets[b]
                eng.ctx.call("mg_allreduce_launch", ptr(self.gflat[off:off + cnt]), cnt, 0)
                self.launched.append(b)

    def _reset_buckets(self):
        self._done = set()
        self.launched = []
        firsts = sorted((f, i) for i, (_, _, f) in enumerate(self.buckets))
        self._bucket_of = {}
        self._missing = [0] * len(self.buckets)
        for k, (f, b) in enumerate(firsts):
            end = firsts[k + 1][0] if k + 1 < len(firsts) else len(self.sizes)
            for idx in range(f, end):
                self._bucket_of[idx] = b
                self._missing[b] += 1


def makeDataParallel(model, nGPU, net=None, bnSync=False):
    """multigpu.lua:81-103"""
    if nGPU > 1:
        if not dist.is_initialized():
            raise ffi.MGError("makeDataParallel(nGPU > 1) needs torch.distributed to be initialised: launch one "
                              "process per GPU (python -m torch.distributed.run --nproc-per-node nGPU ...)")
        return DataParallel(model, nGPU, bnSync=bnSync)
    return model


_BUFFERS = ("running_mean", "running_var")


def _state(model):
    """what a checkpoint holds per module: its parameters and BatchNorm running statistics -- saveDataParallel clears
    output / gradInput of every module before saving (multigpu.lua:110-131), so no activation is ever stored"""
    m = model.model if isinstance(model, DataParallel) else model
    st = []
    for mod in m.listModules():
        d = {name: w.detach().cpu().clone() for name, w, _ in mod.own_parameters()}
        for k in _BUFFERS:
            v = getattr(mod, k, None)
            if isinstance(v, torch.Tensor):
                d[k] = v.detach().cpu().clone()
        st.append((mod.typename, d))
    return st


def saveDataParallel(filename, model):
    """multigpu.lua:105-135: persist replica 1 with its buffers cleared.  The module graph is
    rebuilt by the builder; what is stored are the per-module tensors in listModules() order."""
    if not dist.is_initialized() or dist.get_rank() == 0:
        if str(filename).endswith(".t7"):      # the reference's own container: torch.save of the module tree (mgconv/t7.py)
            from . import t7
            t7.save_model(filename, model)
        else:
            torch.save({"format": "mgconv-b200/1", "modules": _state(model)}, filename)


def _load_into(model, filename):
    if str(filename).endswith(".t7"):          # a Torch7 checkpoint (model_<epoch>.t7, possibly an nn.DataParallelTable)
        from . import t7
        return t7.load_into(model, filename)
    blob = torch.load(filename, map_location="cpu")
    mods = (model.model if isinstance(model, DataParallel) else model).listModules()
    if len(mods) != len(blob["modules"]):
        raise ffi.MGError(f"{filename}: {len(blob['modules'])} modules stored, model has {len(mods)}")
    for mod, (tn, d) in zip(mods, blob["modules"]):
        if tn != mod.typename:
            raise ffi.MGError(f"{filename}: module type {tn} does not match {mod.typename}")
        for k, v in d.items():
            dst = getattr(mod, k, None)
            if not isinstance(dst, torch.Tensor):
                if k in ("output", "gradInput"):     # files written before the state was restricted to parameters
                    continue
                raise ffi.MGError(f"{filename}: {tn} has no tensor field '{k}'")
            if tuple(dst.shape) != tuple(v.shape):
                raise ffi.MGError(f"{filename}: {tn}.{k} is {tuple(v.shape)} in the file, {tuple(dst.shape)} in the model")
            dst.copy_(v)
    return model


def loadDataParallel(filename, nGPU, net, opt):
    """multigpu.lua:137-148: rebuild through the net's createModel, load, wrap for nGPU"""
    o = type(opt)(opt)
    o["nGPU"] = 1
    model = _load_into(net.createModel(o), filename)
    bn_sync = bool(opt.get("bnSync", False)) if hasattr(opt, "get") else bool(getattr(opt, "bnSync", False))
    return makeDataParallel(model, nGPU, net, bnSync=bn_sync)


def loadAndRemoveDPT(filename, net, opt):
    """multigpu.lua:150-160: load a checkpoint as a plain single-GPU module"""
    o = type(opt)(opt)
    o["nGPU"] = 1
    return _load_into(net.createModel(o), filename)
