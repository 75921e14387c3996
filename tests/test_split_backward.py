"""backward() in the two halves of the Torch7 nn protocol: updateGradInput(input, gradOutput) and accGradParameters(input,
gradOutput, scale) (include/mgconv.h: mg_bn_param_grad, mg_stage_update_grad_input / mg_stage_acc_grad_parameters;
mgconv/engine.py: update_grad_input / acc_grad_parameters).

CPU: the header and the ctypes signatures, the misuse rules of nn.Module on a stub engine.
GPU: the batched BatchNorm parameter-gradient launch against mg_bn_backward / mg_bn_backward_frozen bit for bit; whole networks:
updateGradInput + accGradParameters(scale) leaves the bits of backward(scale); updateGradInput alone writes no parameter gradient
and launches fewer tensor-core kernels; repeated accumulation; lanes and CUDA-graph replay; the plan-level ABI from plain C; two
GPUs.
"""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from mgconv import builders as B, ffi, nn
from mgconv.ffi import ptr
from util import Grid, bf16_round

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mgconv.h")
LIB = os.path.join(ROOT, "multigrid-neural-architectures_b200", "mgconv", "libmgconv.so")
NEW = ("mg_bn_param_grad", "mg_stage_update_grad_input", "mg_stage_acc_grad_parameters")


# ------------------------------------------------------------------------------------------------ CPU
def test_header_declares_the_split_in_ffi_cdef_syntax():
    import cffi
    f = cffi.FFI()
    lines = [l for l in open(HEADER).read().split("\n")
             if not l.strip().startswith("#") and not l.startswith('extern "C"') and l.strip() != "}"]
    f.cdef("\n".join(lines).replace("size_t", "unsigned long"))
    lib = f.dlopen(LIB)
    for name in NEW:
        assert hasattr(lib, name)
    assert f.sizeof("mg_bn_param_job") == C.sizeof(ffi.mg_bn_param_job) == 96
    for name, _ in ffi.mg_bn_param_job._fields_:
        assert f.offsetof("mg_bn_param_job", name) == getattr(ffi.mg_bn_param_job, name).offset, name


def test_signatures_match_the_header():
    assert ffi.SIGNATURES["mg_bn_param_grad"] == (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(ffi.mg_bn_param_job)])
    P = C.POINTER(ffi.mg_stage_params)
    assert ffi.SIGNATURES["mg_stage_update_grad_input"] == (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), P, C.POINTER(C.c_void_p)])
    assert ffi.SIGNATURES["mg_stage_acc_grad_parameters"] == (C.c_int, [C.c_void_p, C.c_void_p, P, C.c_float])


class _StubEngine:
    """the engine's side of the protocol without a device: forward generations, the generation updateGradInput recorded"""

    def __init__(self):
        self.generation, self.grad_input_generation, self.acc = 0, None, []

    def forward(self):
        self.generation += 1

    def update_grad_input(self, gradOutput):
        self.grad_input_generation = self.generation
        return "gradInput"

    def acc_grad_parameters(self, scale):
        self.acc.append(scale)


def test_misuse_raises_on_a_stub_engine():
    m = nn.Module()
    go, other = torch.zeros(4, 10), torch.zeros(4, 10)
    with pytest.raises(ffi.MGError, match="no forward"):
        m.updateGradInput(None, go)                          # no plan yet
    m._engine = eng = _StubEngine()
    eng.forward()
    with pytest.raises(ffi.MGError, match="no updateGradInput"):
        m.accGradParameters(None, go)                        # forward without updateGradInput
    assert m.updateGradInput(None, go) == "gradInput"
    m.accGradParameters(None, go, 0.5)                       # the very tensor
    m.accGradParameters(None, None)                          # or None
    m.accGradParameters(None, go, 2)                         # accumulates again
    assert eng.acc == [0.5, 1.0, 2]
    for wrong in (other, go[:2], go.view(40)):               # another storage, another shape
        with pytest.raises(ffi.MGError, match="not the tensor"):
            m.accGradParameters(None, wrong)
    eng.forward()                                            # a new forward
    with pytest.raises(ffi.MGError, match="no updateGradInput"):
        m.accGradParameters(None, go)
    m.updateGradInput(None, [go, other])                     # tables of tensors
    m.accGradParameters(None, [go, other])
    with pytest.raises(ffi.MGError, match="not the tensor"):
        m.accGradParameters(None, [go, go])
    m.clearState()                                           # plan rebuild (getParameters calls clearState too)
    with pytest.raises(ffi.MGError, match="no updateGradInput"):
        m.accGradParameters(None, None)
    assert eng.acc == [0.5, 1.0, 2, 1.0]


# ------------------------------------------------------------------------------------------------ GPU, kernel
DT = {"fp32": ffi.MG_F32, "bf16": ffi.MG_BF16}


def _random_sums(rng, C_):
    """2*C mg_sum values (hi * 2^-10 + lo * 2^-54) of plausible magnitude"""
    s = np.zeros((2 * C_, 2), np.int64)
    s[:, 0] = rng.integers(-(1 << 24), 1 << 24, 2 * C_)
    s[:, 1] = rng.integers(0, 1 << 44, 2 * C_)
    return torch.from_numpy(s.reshape(-1)).cuda()


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("scale", [1.0, 0.25])
def test_batched_parameter_gradients_equal_the_fused_backward(precision, scale):
    """several layers in one launch -- unaligned channel counts, training and frozen layers, one wider than the bf16 one-pass
    kernel takes -- against the dgamma / dbeta / gradBias mg_bn_backward and mg_bn_backward_frozen add, bit for bit"""
    dtype = DT[precision]
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, dtype)
    rng = np.random.default_rng(3)
    N, H = 2, 5
    layers = [(5, False), (13, True), (24, False), (3, True), (37, False), (2056, False), (8, False)]
    jobs = (ffi.mg_bn_param_job * len(layers))()
    fused, split, keep = [], [], []
    for (Cc, frozen), j in zip(layers, jobs):
        sums = _random_sums(rng, Cc)
        gamma, mean = (torch.from_numpy(rng.uniform(a, b, Cc).astype(np.float32)).cuda() for a, b in ((0.5, 1.5), (-0.3, 0.3)))
        invstd = torch.from_numpy(rng.uniform(0.5, 3.0, Cc).astype(np.float32)).cuda()
        rvar = torch.from_numpy(rng.uniform(0.5, 2.0, Cc).astype(np.float32)).cuda()
        start = torch.from_numpy(rng.standard_normal(3 * Cc).astype(np.float32)).cuda()
        a, b = start.clone(), start.clone()
        keep += [sums, gamma, mean, invstd, rvar]
        if frozen:
            ctx.call("mg_bn_backward_frozen", ptr(sums), Cc, ptr(gamma), ptr(mean), ptr(rvar), 1e-5, ptr(a[:Cc]), ptr(a[Cc:2 * Cc]), scale,
                     ptr(a[2 * Cc:]))
        else:
            Y = Grid(dtype, N, Cc, H, H, bf16_round(rng.standard_normal((N, Cc, H, H))))
            D = Grid(dtype, N, Cc, H, H, bf16_round(rng.standard_normal((N, Cc, H, H))))
            G = Grid(dtype, N, Cc, H, H)
            coef = torch.zeros(3 * Y.Cp, device="cuda")
            keep += [Y, D, G, coef]
            ctx.call("mg_bn_backward", C.byref(Y.g()), C.byref(D.g()), C.byref(G.g()), ptr(sums), N * H * H, ptr(gamma), ptr(mean),
                     ptr(invstd), ptr(a[:Cc]), ptr(a[Cc:2 * Cc]), scale, ptr(coef), ptr(a[2 * Cc:]))
        j.sums, j.C, j.frozen, j.gamma, j.eps, j.gscale = sums.data_ptr(), Cc, int(frozen), gamma.data_ptr(), 1e-5, scale
        j.count = 0 if frozen else N * H * H
        if frozen:
            j.running_mean, j.running_var = mean.data_ptr(), rvar.data_ptr()
        else:
            j.save_mean, j.save_invstd = mean.data_ptr(), invstd.data_ptr()
        j.dgamma, j.dbeta, j.conv_dbias = b[:Cc].data_ptr(), b[Cc:2 * Cc].data_ptr(), b[2 * Cc:].data_ptr()
        fused.append(a); split.append(b)
    ctx.call("mg_bn_param_grad", len(layers), jobs)
    torch.cuda.synchronize()
    for (Cc, frozen), a, b in zip(layers, fused, split):
        assert torch.equal(a, b), (Cc, frozen)


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_bn_backward_without_parameter_outputs_writes_the_same_gradient(precision):
    """the update phase calls mg_bn_backward with dgamma / dbeta / conv_dbias NULL: G must not change"""
    dtype = DT[precision]
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, dtype)
    rng = np.random.default_rng(5)
    N, H, Cc = 3, 6, 13
    sums = _random_sums(rng, Cc)
    gamma, mean, invstd = (torch.from_numpy(rng.uniform(0.5, 1.5, Cc).astype(np.float32)).cuda() for _ in range(3))
    Y = Grid(dtype, N, Cc, H, H, bf16_round(rng.standard_normal((N, Cc, H, H))))
    D = Grid(dtype, N, Cc, H, H, bf16_round(rng.standard_normal((N, Cc, H, H))))
    outs = []
    for with_params in (True, False):
        G, coef, pg = Grid(dtype, N, Cc, H, H), torch.zeros(3 * Y.Cp, device="cuda"), torch.zeros(3 * Cc, device="cuda")
        p = (ptr(pg[:Cc]), ptr(pg[Cc:2 * Cc]), ptr(pg[2 * Cc:])) if with_params else (None, None, None)
        ctx.call("mg_bn_backward", C.byref(Y.g()), C.byref(D.g()), C.byref(G.g()), ptr(sums), N * H * H, ptr(gamma), ptr(mean), ptr(invstd),
                 p[0], p[1], 0.5, ptr(coef), p[2])
        outs.append(G)
    torch.cuda.synchronize()
    assert torch.equal(outs[0].t, outs[1].t)


# ------------------------------------------------------------------------------------------------ GPU, networks
PNMG_OPT = dict(nLayer=1, blocks=B.CIFAR_RNMG_BLOCKS)
R10_BLOCKS = [([16, 8, 8], [3, 3, 3], False), ([32, 16, 16], [3, 3, 3], True), ([64, 32], [3, 3], True), ([128], [3], False)]
R10_OPT = dict(nClass=10, inputBlock=[16, 8, 8], cfg=[1, 1, 1, 1], avg=2, blocks=R10_BLOCKS)
# name, network, options, input shape, mode
NETS = [
    ("R-MG-34 224x224", "ilsvrc/rnmg", dict(depth=34), (2, 3, 224, 224), "train"),
    ("PR-NMG-30", "cifar/prnmg", dict(nLayer=2), (4, 3, 32, 32), "train"),
    ("prnmg.mnist", "mnist-cluttered/prnmg.mnist", dict(dataset="mnist-seg"), (2, 1, 64, 64), "train"),
    ("U-MG", "mnist-cluttered/unmg", dict(dataset="mnist-seg"), (2, 1, 64, 64), "train"),
    ("P-NMG-11 isDropout", "cifar/pnmg", dict(isDropout=True, **PNMG_OPT), (8, 3, 32, 32), "train"),
    ("P-NMG-11 quarter frozen", "cifar/pnmg", PNMG_OPT, (8, 3, 32, 32), "quarter-frozen"),
    ("R-MG-10 evaluate needInputGrad", "ilsvrc/rnmg", R10_OPT, (4, 3, 64, 64), "evaluate"),
]


def _model(net, opt, precision, mode, seed=7):
    torch.manual_seed(seed)
    m = B.load_net(net).createModel(B.Opt(nGPU=1, **opt))
    m.precision = precision
    m.needInputGrad = mode == "evaluate"
    m.cuda()
    if mode == "evaluate":
        m.evaluate()
    elif mode == "quarter-frozen":
        bns = m.findModules("nn.SpatialBatchNormalization")
        for b in bns[:max(1, len(bns) // 4)]:
            b.evaluate()
    return m


def _state(m, grads, gi):
    bns = m.findModules("nn.SpatialBatchNormalization")
    gi = [] if gi is None else (gi if isinstance(gi, list) else [gi])
    return [g.clone() for g in gi] + [grads.clone()] + [t.clone() for b in bns for t in (b.running_mean, b.running_var)]


def _run(net, opt, shape, precision, mode, split, scale, seed=7):
    m = _model(net, opt, precision, mode, seed)
    params, grads = m.getParameters()
    g = torch.Generator().manual_seed(11)
    x = torch.randn(*shape, generator=g).cuda()
    torch.manual_seed(seed + 1)   # dropout key of the plan
    out = m.forward(x)
    go = torch.randn(*out.shape, generator=g).cuda()
    if split:
        gi = m.updateGradInput(x, go)
        m.accGradParameters(x, go, scale)
    else:
        gi = m.backward(x, go, scale)
    torch.cuda.synchronize()
    return m, _state(m, grads, gi)


def _equal(a, b):
    assert len(a) == len(b)
    for i, (u, v) in enumerate(zip(a, b)):
        assert torch.equal(u, v), i


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("case", range(len(NETS)), ids=[n[0] for n in NETS])
def test_split_equals_backward(monkeypatch, case, precision):
    """gradInput, the flat gradient vector and the running statistics, bit for bit"""
    monkeypatch.setenv("MGCONV_AUTOTUNE", "0")
    name, net, opt, shape, mode = NETS[case]
    scale = 0.25 if case % 2 else 1.0
    _, ref = _run(net, opt, shape, precision, mode, False, scale)
    m, got = _run(net, opt, shape, precision, mode, True, scale)
    if mode == "evaluate":
        assert m.gradInput is not None
    _equal(got, ref)


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_update_grad_input_alone(monkeypatch, precision):
    """image gradients (evaluate() + needInputGrad): the gradient vector keeps its sentinel, the image gradient is backward's,
    and no weight-gradient kernel runs"""
    monkeypatch.setenv("MGCONV_AUTOTUNE", "0")
    name, net, opt, shape, _ = NETS[-1]
    res = {}
    for split in (False, True):
        m = _model(net, opt, precision, "evaluate")
        _, grads = m.getParameters()
        sentinel = torch.arange(grads.numel(), dtype=torch.float32, device="cuda").remainder_(977).mul_(0.125)
        grads.copy_(sentinel)
        x = torch.randn(*shape, generator=torch.Generator().manual_seed(3)).cuda()
        out = m.forward(x)
        go = torch.randn(*out.shape, generator=torch.Generator().manual_seed(4)).cuda()
        m.updateGradInput(x, go) if split else m.backward(x, go)   # first call: plans the backward, tunes nothing (autotune off)
        torch.cuda.synchronize()
        ctx = m._engine.ctx
        # bf16 convolutions run on the tcgen05 kernels, fp32 ones on CUDA cores: count those, or every launch
        count = ctx.tc_launches if precision == "bf16" else ctx.launches
        m.forward(x)
        n0 = count()
        gi = m.updateGradInput(x, go) if split else m.backward(x, go)
        torch.cuda.synchronize()
        res[split] = (gi.clone(), count() - n0, torch.equal(grads, sentinel))
    assert res[True][2], "updateGradInput wrote a parameter gradient"
    assert not res[False][2]
    assert torch.equal(res[True][0], res[False][0])
    assert 0 < res[True][1] < res[False][1], (res[True][1], res[False][1])
    what = "tcgen05 launches" if precision == "bf16" else "launches"
    print(f"[measured] {name} {precision}: {what} of updateGradInput {res[True][1]}, of backward {res[False][1]}")


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_accumulation_and_misuse(monkeypatch, precision):
    """two accGradParameters(1) equal two backward(1) of the same forward bit for bit; every misuse raises"""
    monkeypatch.setenv("MGCONV_AUTOTUNE", "0")
    name, net, opt, shape, mode = NETS[5]
    res = []
    for split in (False, True):
        m = _model(net, opt, precision, mode)
        _, grads = m.getParameters()
        x = torch.randn(*shape, generator=torch.Generator().manual_seed(3)).cuda()
        out = m.forward(x)
        go = torch.randn(*out.shape, generator=torch.Generator().manual_seed(4)).cuda()
        if split:
            with pytest.raises(ffi.MGError, match="no updateGradInput"):
                m.accGradParameters(x, go)
            m.updateGradInput(x, go)
            with pytest.raises(ffi.MGError, match="not the tensor"):
                m.accGradParameters(x, go.clone())
            m.accGradParameters(x, go, 1.0)
            m.accGradParameters(x, None, 1.0)
        else:
            m.backward(x, go, 1.0)
            m.backward(x, go, 1.0)
        torch.cuda.synchronize()
        res.append(grads.clone())
        if split:
            m.forward(x)                                           # a new forward
            with pytest.raises(ffi.MGError, match="no updateGradInput"):
                m.accGradParameters(x, go)
            m.updateGradInput(x, go)
            m.clearState()                                         # plan rebuilt
            with pytest.raises(ffi.MGError, match="no updateGradInput"):
                m.accGradParameters(x, go)
            m.forward(x)
            m.updateGradInput(x, go)
            m.getParameters()                                      # parameters re-homed: plan rebuilt
            with pytest.raises(ffi.MGError, match="no updateGradInput"):
                m.accGradParameters(x, go)
    assert torch.equal(res[0], res[1])


@gpu
def test_lanes_and_graph_replay_of_the_split_step(monkeypatch):
    """P-NMG-11 bf16 with a quarter of its BatchNorm layers frozen: the split step on three lanes and replayed as one CUDA graph
    equals the serial eager split step, which equals the serial backward step"""
    from mgconv.graph import GraphedStep
    monkeypatch.setenv("MGCONV_AUTOTUNE", "0")
    name, net, opt, shape, mode = NETS[5]
    g = torch.Generator().manual_seed(3)
    x = torch.randn(*shape, generator=g).cuda()
    t = torch.randint(1, 101, (shape[0],), generator=g).cuda()
    res = {}
    for variant in ("backward", "serial", "lanes", "graph"):
        monkeypatch.setenv("MGCONV_LANES", "1" if variant in ("backward", "serial") else "3")
        m = _model(net, opt, "bf16", mode)
        params, grads = m.getParameters()
        crit = B.load_net(net).createCriterion()
        st = {}

        def step():
            m.zeroGradParameters()
            out = m.forward(x)
            crit.forward(out, t)
            go = crit.backward(out, t)
            if variant == "backward":
                m.backward(x, go)
            else:
                m.updateGradInput(x, go)
                m.accGradParameters(x, go, 0.5)
                m.accGradParameters(x, go, 0.5)
            st["out"] = out
        step()
        torch.cuda.synchronize()
        run = GraphedStep(step) if variant == "graph" else step
        run()
        torch.cuda.synchronize()
        res[variant] = (st["out"].clone(), grads.clone())
    for v in ("lanes", "graph"):
        assert torch.equal(res[v][0], res["serial"][0]) and torch.equal(res[v][1], res["serial"][1]), v
    assert torch.equal(res["serial"][0], res["backward"][0])


def _build_cabi_split():
    src, binary = os.path.join(ROOT, "tests", "cabi_split.c"), os.path.join(ROOT, "tests", "cabi_split")
    if os.path.exists(binary) and os.path.getmtime(binary) >= max(os.path.getmtime(src), os.path.getmtime(LIB)):
        return binary
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.run(["gcc", "-std=c99", "-O1", src, "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(cuda, "include"), "-o", binary, LIB,
                    "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + os.path.dirname(LIB), "-Wl,-rpath," + os.path.join(cuda, "lib64")],
                   check=True)
    return binary


def test_cabi_split_compiles_as_c99():
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    assert os.path.exists(_build_cabi_split())


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("scale", ["1", "0.25"])
def test_stage_split_through_the_c_abi(precision, scale):
    r = subprocess.run([_build_cabi_split(), precision, scale], capture_output=True, text=True, timeout=300)
    print(r.stdout)
    assert r.returncode == 0 and "cabi_split ok" in r.stdout, r.stdout + r.stderr


@gpu
@pytest.mark.parametrize("variant", ["local-bn", "bnSync", "iterSize2"])
def test_two_gpu_split_equals_backward(variant):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "tests", "dp_split_worker.py"), variant]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "dp-split ok rank 0" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
