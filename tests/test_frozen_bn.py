"""BatchNorm in evaluation mode under backpropagation: model:evaluate() + backward, and bn:evaluate() inside a training model
(include/mgconv.h: mg_grad_combine_bn_frozen, mg_bn_backward_frozen; mgconv/engine.py: per-module BatchNorm mode).

CPU: the plan keys (models in one mode keep theirs) and the oracle (oracle/frozen_bn.py) against PyTorch autograd.
GPU: the frozen combine and parameter-gradient kernels against numpy in fp32 and bf16, whole networks against the fp64 oracle,
running statistics of frozen layers left alone, the evaluate() forward unchanged by skipping the statistics, lanes / graph replay
against the serial eager step, and the plan-level ABI after mg_stage_forward(training = 0).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import builders as OB, frozen_bn as OF, nn_ops as NO
from mgconv import builders as B, ffi, ops as O
from mgconv.ffi import mg_grad_src, ptr
from util import Grid, copy_params_from_oracle, rel_err, bf16_round, emulate_bf16_storage

gpu = pytest.mark.gpu
SHAPE = (8, 3, 32, 32)
PNMG = (lambda: OB.cifar_pnmg(1, blocks=OB.CIFAR_RNMG_NARROW), B.cifar_pnmg, dict(nLayer=1, blocks=B.CIFAR_RNMG_BLOCKS))


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def _first_quarter(n):
    return list(range(max(1, n // 4)))


# ------------------------------------------------------------------------------------------------ CPU
def test_plan_keys_change_only_for_mixed_modes():
    from mgconv.engine import engine_key
    m = B.cifar_pnmg.createModel(B.Opt(nGPU=1, **PNMG[2]))
    x = torch.zeros(SHAPE)
    drops, bns = m.findModules("nn.Dropout"), m.findModules("nn.SpatialBatchNormalization")
    base = engine_key(x, drops)
    assert engine_key(x, drops, bns, m.train) == base            # training(): every BatchNorm trains
    m.evaluate()
    assert engine_key(x, drops, bns, m.train) == base            # evaluate(): every BatchNorm frozen, same plan
    m.training()
    bns[0].evaluate(); bns[2].evaluate()
    k = engine_key(x, drops, bns, m.train)
    assert k != base and k[-1] == ("frozen_bn", 0, 2)
    bns[2].training()
    assert engine_key(x, drops, bns, m.train) not in (base, k)


def test_oracle_eval_backward_matches_autograd():
    rng = np.random.default_rng(0)
    N, Cc, H = 3, 5, 6
    x, go = rng.standard_normal((N, Cc, H, H)), rng.standard_normal((N, Cc, H, H))
    g, b = rng.uniform(0.5, 1.5, Cc), rng.normal(0, 0.2, Cc)
    rm, rv = rng.normal(0, 0.3, Cc), rng.uniform(0.5, 2.0, Cc)
    tx, tg, tb = _t(x).requires_grad_(), _t(g).requires_grad_(), _t(b).requires_grad_()
    y = torch.nn.functional.batch_norm(tx, _t(rm), _t(rv), tg, tb, training=False, eps=1e-5)
    y.backward(_t(go))
    assert np.allclose(OF.bn_forward_eval(x, g, b, rm, rv), y.detach().numpy(), rtol=1e-12, atol=1e-12)
    gi, gw, gb = OF.bn_backward_eval(x, go, g, rm, rv)
    for a, ref in ((gi, tx.grad), (gw, tg.grad), (gb, tb.grad)):
        assert np.allclose(a, ref.numpy(), rtol=1e-12, atol=1e-12)


def test_oracle_freeze_leaves_running_statistics_alone():
    om = PNMG[0]().double()
    frozen = OF.freeze(om, [0, 1])
    before = [(m.running_mean.clone(), m.running_var.clone()) for m in OF.batchnorms(om)]
    om(torch.randn(4, 3, 32, 32, dtype=torch.float64))
    after = [(m.running_mean, m.running_var) for m in OF.batchnorms(om)]
    for i, ((m0, v0), (m1, v1)) in enumerate(zip(before, after)):
        assert torch.equal(m0, m1) == (i < 2) and torch.equal(v0, v1) == (i < 2)
    assert all(not m.training for m in frozen)


def test_oracle_stem_and_pyramid_backward_match_autograd():
    """oracle.nn_ops: data gradient of the 7x7 / stride-2 / pad-3 stem and SpatialAveragePooling(r,r,r,r) backward (floor mode,
    sizes that leave rows / columns outside every window)"""
    rng = np.random.default_rng(1)
    x, w = rng.standard_normal((2, 3, 23, 21)), rng.standard_normal((16, 3, 7, 7))
    tx = _t(x).requires_grad_()
    y = torch.nn.functional.conv2d(tx, _t(w), stride=2, padding=3)
    go = rng.standard_normal(tuple(y.shape))
    y.backward(_t(go))
    assert np.allclose(NO.conv_backward(x, w, go, s=2, p=3)[0], tx.grad.numpy(), rtol=1e-12, atol=1e-12)
    for r in (2, 4):
        tx = _t(x).requires_grad_()
        y = torch.nn.functional.avg_pool2d(tx, r, r)
        go = rng.standard_normal(tuple(y.shape))
        y.backward(_t(go))
        assert np.allclose(NO.avgpool_backward(go, x.shape, r), tx.grad.numpy(), rtol=1e-12, atol=1e-12)


def test_lowering_gives_the_pyramid_a_gradient_only_with_needInputGrad():
    from mgconv import lower as L
    for need in (False, True):
        m = B.ilsvrc_rnmg.createModel(B.Opt(nGPU=1, **NETS[2][3]))
        b, _ = L.trace_model(m, (2, 3, 64, 64), need)
        pools = [o for o in b.ops if isinstance(o, O.AvgPoolOp)]
        assert pools and all(o.out.needs_grad == need for o in pools)
        stem = [o for o in b.ops if isinstance(o, O.ConvOp) and o.stride == 2]
        assert stem and all(o.k == 7 and o.segs[0][0].C == 3 and o.segs[0][0].needs_grad == need for o in stem)   # one per pyramid level


# ------------------------------------------------------------------------------------------------ GPU, kernels
DT = {"fp32": ffi.MG_F32, "bf16": ffi.MG_BF16}


def _rnd(a, precision):
    return bf16_round(a) if precision == "bf16" else np.asarray(a, np.float32).astype(np.float64)


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("Cc", [5, 24], ids=["unaligned", "aligned"])
@pytest.mark.parametrize("write_d", [False, True], ids=["G-only", "residual-reads-D"])
def test_frozen_combine_and_parameter_gradients(precision, Cc, write_d):
    """sources: the same-resolution gradient of a consumer and the up-sampled one of a finer consumer; ReLU mask of x"""
    dtype = DT[precision]
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, dtype)
    rng = np.random.default_rng(Cc + 7 * write_d)
    N, H = 2, 6
    x = _rnd(rng.standard_normal((N, Cc, H, H)), precision)
    y = _rnd(rng.standard_normal((N, Cc, H, H)), precision)
    g0 = _rnd(rng.standard_normal((N, Cc, H, H)), precision)
    g1 = _rnd(rng.standard_normal((N, Cc, 2 * H, 2 * H)), precision)
    gamma, rm = rng.uniform(0.5, 1.5, Cc).astype(np.float32), rng.normal(0, 0.3, Cc).astype(np.float32)
    rv = rng.uniform(0.5, 2.0, Cc).astype(np.float32)
    eps = 1e-5
    X, Y, S0, S1 = (Grid(dtype, N, Cc, H, H, x), Grid(dtype, N, Cc, H, H, y), Grid(dtype, N, Cc, H, H, g0), Grid(dtype, N, Cc, 2 * H, 2 * H, g1))
    src = (mg_grad_src * 2)()
    for i, (S, mode) in enumerate(((S0, ffi.MG_SEG_SAME), (S1, ffi.MG_SEG_UP))):
        src[i].g, src[i].c_offset, src[i].mode, src[i].aux = S.g(), 0, mode, None
    tg, trm, trv = (torch.from_numpy(a).cuda() for a in (gamma, rm, rv))
    dg, db, cb = (torch.full((Cc,), 0.5, device="cuda") for _ in range(3))

    def run():
        G, D = Grid(dtype, N, Cc, H, H), Grid(dtype, N, Cc, H, H)
        sums = torch.zeros(4 * Cc, dtype=torch.int64, device="cuda")
        ctx.call("mg_grad_combine_bn_frozen", C.byref(X.g()), 1, C.byref(Y.g()), 2, src, ptr(tg), ptr(trv), eps, C.byref(G.g()),
                 C.byref(D.g()) if write_d else None, ptr(sums))
        ctx.call("mg_bn_backward_frozen", ptr(sums), Cc, ptr(tg), ptr(trm), ptr(trv), eps, ptr(dg), ptr(db), 0.75, ptr(cb))
        torch.cuda.synchronize()
        return G, D

    G, D = run()
    d = (g0 + g1.reshape(N, Cc, H, 2, H, 2).sum(axis=(3, 5))) * (x > 0)
    if precision == "bf16":
        d = bf16_round(d)   # the sum is taken in fp32 and stored once
    gi, gw, gb = OF.bn_backward_eval(y, d, gamma, rm, rv, eps, scale=0.75)
    A = (gamma.astype(np.float64) / np.sqrt(rv.astype(np.float64) + eps)).astype(np.float32).astype(np.float64)
    tol = {"fp32": 1e-4, "bf16": 2e-2}[precision]
    assert rel_err(G.nchw(), gi) <= tol
    assert not G.pad_channels().any()
    if write_d:
        assert rel_err(D.nchw(), d) <= tol
    else:
        assert not D.t.any()
    assert rel_err(dg.cpu().numpy() - 0.5, gw) <= tol
    assert rel_err(db.cpu().numpy() - 0.5, gb) <= tol
    assert rel_err(cb.cpu().numpy() - 0.5, 0.75 * A * d.sum(axis=(0, 2, 3))) <= tol
    # deterministic: a second run writes the same bits
    first = [a.clone() for a in (dg, db, cb)]
    for a in (dg, db, cb):
        a.fill_(0.5)
    G2, _ = run()
    assert torch.equal(G.t, G2.t)
    assert all(torch.equal(a, f) for a, f in zip((dg, db, cb), first))


# ------------------------------------------------------------------------------------------------ GPU, networks
R10_BLOCKS = [([16, 8, 8], [3, 3, 3], False), ([32, 16, 16], [3, 3, 3], True), ([64, 32], [3, 3], True), ([128], [3], False)]
NETS = [
    ("R-NMG-12 cifar/rnmg nLayer=1", lambda: OB.cifar_rnmg(1), B.cifar_rnmg, dict(nLayer=1), (8, 3, 32, 32), 100),
    ("P-NMG-11 cifar/pnmg nLayer=1 narrow", PNMG[0], PNMG[1], PNMG[2], (8, 3, 32, 32), 100),
    ("R-MG-10 ilsvrc/rnmg reduced 64x64", lambda: OB.ilsvrc_rnmg(18, 10, [16, 8, 8], R10_BLOCKS, [1, 1, 1, 1], 2), B.ilsvrc_rnmg,
     dict(nClass=10, inputBlock=[16, 8, 8], cfg=[1, 1, 1, 1], avg=2, blocks=R10_BLOCKS), (4, 3, 64, 64), 10),
    ("R-MG-34 ilsvrc/rnmg depth 34 224x224", lambda: OB.ilsvrc_rnmg(34), B.ilsvrc_rnmg, dict(depth=34), (2, 3, 224, 224), 1000),
]
# the fp32 whole-network bars of test_models_gpu.FP32_GRAD_BAR (1e-4 elsewhere): R-NMG-12 normalises its 1x1 grids over a
# handful of values in its training-mode layers; R-MG-34 at batch 2 sums 34 layers deep, where an activation within fp32
# rounding of zero flips its ReLU mask against the fp64 oracle (measured 2.6e-4 in evaluate(), 7.4e-4 with a quarter frozen)
FP32_GRAD_BAR = {"R-NMG-12 cifar/rnmg nLayer=1": 2e-2, "R-MG-34 ilsvrc/rnmg depth 34 224x224": 1e-2}


def _random_running_statistics(om, rng):
    with torch.no_grad():
        for m in OF.batchnorms(om):
            m.running_mean.copy_(_t(rng.normal(0, 0.2, m.num_features)))
            m.running_var.copy_(_t(rng.uniform(0.5, 2.0, m.num_features)))


def _all_grads(olist, plist):
    og = np.concatenate([np.concatenate([o.weight.grad.numpy().ravel(), o.bias.grad.numpy().ravel()]) for o in olist])
    pg = np.concatenate([np.concatenate([p.gradWeight.cpu().numpy().ravel(), p.gradBias.cpu().numpy().ravel()]) for p in plist])
    return og, pg


@gpu
@pytest.mark.parametrize("mode", ["evaluate", "first-quarter-frozen"])
@pytest.mark.parametrize("case", range(len(NETS)), ids=[n[0] for n in NETS])
def test_network_gradients_follow_the_oracle(case, mode):
    """fp32 (the 1e-4 parity path): log-probabilities, every parameter gradient and the image gradient (needInputGrad: through the
    strided stem and the SpatialAveragePooling pyramid where the network has them) against the fp64 oracle in the same modes"""
    name, octor, net, opt, shape, nclass = NETS[case]
    torch.manual_seed(2)
    rng = np.random.default_rng(5)
    om = octor().double()
    _random_running_statistics(om, rng)
    pm = net.createModel(B.Opt(nGPU=1, **opt))
    pm.precision = "fp32"
    pm.needInputGrad = True
    olist, plist = copy_params_from_oracle(om, pm)
    pm.cuda()
    plist = [m for m in pm.listModules() if m.own_parameters()]
    pbns = pm.findModules("nn.SpatialBatchNormalization")
    if mode == "evaluate":
        om.eval(); pm.evaluate()
        frozen = list(range(len(pbns)))
    else:
        frozen = _first_quarter(len(pbns))
        OF.freeze(om, frozen)
        for i in frozen:
            pbns[i].evaluate()
    x = bf16_round(rng.standard_normal(shape))
    t = rng.integers(1, nclass + 1, shape[0])
    ox = _t(x).requires_grad_()
    olp = om(ox)
    torch.nn.functional.nll_loss(olp, _t(t - 1)).backward()
    rs = [(b.running_mean.clone(), b.running_var.clone()) for b in pbns]
    outputs, err = net.ftrain(_t(x).float().cuda(), _t(t).cuda(), pm, net.createCriterion())
    torch.cuda.synchronize()
    assert all(pm._engine.bn_ops[i].frozen == (i in frozen) for i in range(len(pbns)))
    e = rel_err(outputs.cpu().numpy(), olp.detach().numpy())
    og, pg = _all_grads(olist, plist)
    eg = rel_err(pg, og)
    ei = rel_err(pm.gradInput.cpu().numpy(), ox.grad.numpy())
    print(f"[measured] {name} fp32 {mode}: log-prob {e:.2e}, gradient {eg:.2e}, image gradient {ei:.2e}")
    assert e <= 1e-4, ("log-probabilities", e)
    assert eg <= FP32_GRAD_BAR.get(name, 1e-4), ("parameter gradients", eg)
    assert ei <= FP32_GRAD_BAR.get(name, 1e-4), ("image gradient", ei)
    for i, (b, (m0, v0)) in enumerate(zip(pbns, rs)):
        if i in frozen:
            assert torch.equal(b.running_mean, m0) and torch.equal(b.running_var, v0), i
        else:
            assert not torch.equal(b.running_var, v0), i


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_residual_unit_input_gradient_in_evaluation_mode(precision):
    """model:evaluate(), needInputGrad: the gradient of the inputs of a residual multigrid unit (models/ilsvrc/rnmg.lua:91-159)"""
    torch.manual_seed(1)
    rng = np.random.default_rng(3)
    cin, cout, hs, N = [8, 4, 4], [16, 8, 4], [8, 4, 2], 3
    om = OB.res_mgConv(list(cin), list(cout), [3, 3, 3]).double()
    with torch.no_grad():
        for m in OF.batchnorms(om):
            m.weight.uniform_(0.5, 1.5); m.bias.normal_(0, 0.1)
    _random_running_statistics(om, rng)
    om.eval()
    pm = B.mgConv(list(cin), list(cout), [3, 3, 3])
    pm.precision = precision
    pm.needInputGrad = True
    olist, _ = copy_params_from_oracle(om, pm, bf16_weights=precision == "bf16")
    if precision == "bf16":
        emulate_bf16_storage(om)
    pm.cuda()
    pm.evaluate()
    plist = [m for m in pm.listModules() if m.own_parameters()]
    xs = [bf16_round(rng.standard_normal((N, c, h, h))) for c, h in zip(cin, hs)]
    oxs = [_t(x).requires_grad_() for x in xs]
    oy = om(oxs)
    gos = [bf16_round(rng.standard_normal(tuple(y.shape))) for y in oy]
    torch.autograd.backward(oy, [_t(g) for g in gos])
    py = pm.forward([_t(x).float().cuda() for x in xs])
    gi = pm.backward(None, [_t(g).float().cuda() for g in gos])
    torch.cuda.synchronize()
    tol = {"fp32": 1e-4, "bf16": 2e-2}[precision]
    for i in range(3):
        assert rel_err(py[i].cpu().numpy(), oy[i].detach().numpy()) <= tol, ("out", i)
        assert rel_err(gi[i].cpu().numpy(), oxs[i].grad.numpy()) <= tol, ("gradInput", i)
    og, pg = _all_grads(olist, plist)
    assert rel_err(pg, og) <= tol


def _bf16_model(frozen=True, seed=11):
    torch.manual_seed(seed)
    pm = PNMG[1].createModel(B.Opt(nGPU=1, **PNMG[2]))
    pm.precision = "bf16"
    pm.cuda()
    if frozen:
        bns = pm.findModules("nn.SpatialBatchNormalization")
        for i in _first_quarter(len(bns)):
            bns[i].evaluate()
    return pm


def _batch(seed=3):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(*SHAPE, generator=g).cuda(), torch.randint(1, 101, (SHAPE[0],), generator=g).cuda()


@gpu
def test_evaluate_forward_is_unchanged_by_skipping_the_statistics(monkeypatch):
    """evaluate(): the convolutions no longer reduce BatchNorm statistics; the output is bit for bit the one of a plan that does"""
    monkeypatch.setenv("MGCONV_AUTOTUNE", "0")
    outs = []
    for skip in (True, False):
        if not skip:   # what the plan did before: every convolution feeding a BatchNorm reduces its sums
            monkeypatch.setattr(O, "_stats", lambda conv: ptr(conv.sums))
        for name, octor, net, opt, shape, _ in (NETS[0], NETS[2]):
            torch.manual_seed(4)
            pm = net.createModel(B.Opt(nGPU=1, **opt))
            pm.cuda()
            x = torch.randn(*shape, generator=torch.Generator().manual_seed(1)).cuda()
            pm.forward(x)              # one training forward: running statistics away from (0, 1)
            pm.evaluate()
            outs.append(pm.forward(x).clone())
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[2]) and torch.equal(outs[1], outs[3])


@gpu
def test_lanes_and_graph_replay_equal_the_serial_eager_step(monkeypatch):
    from mgconv.graph import GraphedStep
    monkeypatch.setenv("MGCONV_AUTOTUNE", "0")
    x, t = _batch()
    res = {}
    for variant in ("serial", "lanes", "graph"):
        monkeypatch.setenv("MGCONV_LANES", "1" if variant == "serial" else "3")
        pm = _bf16_model()
        params, grads = pm.getParameters()
        crit = PNMG[1].createCriterion()
        out = {}

        def step():
            pm.zeroGradParameters()
            out["o"], _ = PNMG[1].ftrain(x, t, pm, crit)
        step()
        torch.cuda.synchronize()
        run = GraphedStep(step) if variant == "graph" else step
        run()
        torch.cuda.synchronize()
        assert any(o.frozen for o in pm._engine.bn_ops) and not all(o.frozen for o in pm._engine.bn_ops)
        res[variant] = (out["o"].clone(), grads.clone())
    for v in ("lanes", "graph"):
        assert torch.equal(res[v][0], res["serial"][0]) and torch.equal(res[v][1], res["serial"][1]), v


@gpu
def test_frozen_training_steps_are_bit_identical_and_keep_running_statistics():
    x, t = _batch()
    res = []
    for _ in range(2):
        pm = _bf16_model()
        bns = pm.findModules("nn.SpatialBatchNormalization")
        frozen = _first_quarter(len(bns))
        rs = [(b.running_mean.clone(), b.running_var.clone()) for b in bns]
        params, grads = pm.getParameters()
        crit = PNMG[1].createCriterion()
        st = dict(learningRate=0.05, momentum=0.9, weightDecay=5e-4, dampening=0.0)
        for _ in range(2):
            pm.zeroGradParameters()

            def feval(_p):
                PNMG[1].ftrain(x, t, pm, crit)
                return 0.0, grads
            PNMG[1].btrain(params, feval, st)
        torch.cuda.synchronize()
        for i, (b, (m0, v0)) in enumerate(zip(bns, rs)):
            assert (torch.equal(b.running_mean, m0) and torch.equal(b.running_var, v0)) == (i in frozen), i
        res.append(params.clone())
    assert torch.equal(res[0], res[1])


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_stage_backward_after_evaluation_forward(precision):
    """plan-level ABI: mg_stage_forward(training = 0) then mg_stage_backward differentiates the evaluation-mode unit"""
    dtype = DT[precision]
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, dtype)
    rng = np.random.default_rng(9)
    torch.manual_seed(9)
    cin, cout, hs, N = [16, 8], [16, 16], [8, 4], 2
    n = len(cin)
    om = OB.res_mgConv(list(cin), list(cout), [3] * n).double()
    convs = [m for m in om.modules() if isinstance(m, torch.nn.Conv2d)]
    bns = OF.batchnorms(om)
    with torch.no_grad():
        for c in convs:
            if precision == "bf16":
                c.weight.copy_(c.weight.to(torch.bfloat16).to(c.weight.dtype))
            c.bias.normal_(0, 0.1)
        for b in bns:
            b.weight.uniform_(0.5, 1.5); b.bias.normal_(0, 0.2)
    _random_running_statistics(om, rng)
    om.eval()
    if precision == "bf16":
        emulate_bf16_storage(om)
    xs = [bf16_round(rng.standard_normal((N, c, h, h))) for c, h in zip(cin, hs)]
    oxs = [_t(x).requires_grad_() for x in xs]
    oy = om(oxs)
    gos = [bf16_round(rng.standard_normal(tuple(y.shape))) for y in oy]
    torch.autograd.backward(oy, [_t(g) for g in gos])

    d = ffi.mg_stage_desc()
    d.n_scales, d.residual, d.no_final_relu, d.eps, d.momentum = n, 1, 0, 1e-5, 0.1
    for i in range(n):
        d.C_in[i], d.C_out[i], d.H[i], d.W[i], d.ksize[i] = cin[i], cout[i], hs[i], hs[i], 3
    plan = C.c_void_p()
    ctx.call("mg_plan_create", C.byref(d), N, C.byref(plan))
    ws = torch.zeros(ffi.lib.mg_plan_workspace_bytes(plan) // 4 + 64, dtype=torch.float32, device="cuda")
    keep = []

    def dev(t_):
        a = t_.detach().float().contiguous().cuda()
        keep.append(a)
        return a.data_ptr()
    prm = ffi.mg_stage_params()
    for k, (c, b) in enumerate(zip(convs, bns)):
        prm.conv_w[k], prm.conv_b[k], prm.bn_g[k], prm.bn_b[k] = dev(c.weight), dev(c.bias), dev(b.weight), dev(b.bias)
        prm.bn_rm[k], prm.bn_rv[k] = dev(b.running_mean), dev(b.running_var)
        for f, ref in (("conv_gw", c.weight), ("conv_gb", c.bias), ("bn_gg", b.weight), ("bn_gb", b.bias)):
            getattr(prm, f)[k] = dev(torch.zeros_like(ref))
    by_ptr = {a.data_ptr(): a for a in keep}
    running = [(by_ptr[prm.bn_rm[k]], by_ptr[prm.bn_rv[k]]) for k in range(len(bns))]
    running_before = [(m.clone(), v.clone()) for m, v in running]
    x_d = [dev(_t(x)) for x in xs]
    y_t = [torch.zeros(tuple(y.shape), device="cuda") for y in oy]
    dy_d = [dev(_t(g)) for g in gos]
    dx_t = [torch.zeros(tuple(x.shape), device="cuda") for x in xs]
    arr = lambda ps: (C.c_void_p * n)(*ps)
    # the stage calls take the plan, not the context: errors are read from the context the plan was created on
    for rc in (ffi.lib.mg_stage_forward(plan, C.c_void_p(ws.data_ptr()), arr(x_d), C.byref(prm), arr([y.data_ptr() for y in y_t]), 0),
               ffi.lib.mg_stage_backward(plan, C.c_void_p(ws.data_ptr()), arr(dy_d), C.byref(prm), arr([t_.data_ptr() for t_ in dx_t]), 1.0)):
        assert rc == 0, ffi.lib.mg_last_error(ctx.h).decode()
    torch.cuda.synchronize()
    ffi.lib.mg_plan_destroy(plan)
    tol = {"fp32": 1e-4, "bf16": 2e-2}[precision]
    for a, ref in zip(y_t, oy):
        assert rel_err(a.cpu().numpy(), ref.detach().numpy()) <= tol
    for a, ref in zip(dx_t, oxs):
        assert rel_err(a.cpu().numpy(), ref.grad.numpy()) <= tol
    for k, (c, b) in enumerate(zip(convs, bns)):
        for f, ref in (("conv_gw", c.weight.grad), ("conv_gb", c.bias.grad), ("bn_gg", b.weight.grad), ("bn_gb", b.bias.grad)):
            assert rel_err(by_ptr[getattr(prm, f)[k]].cpu().numpy(), ref.numpy()) <= 2 * tol, (f, k)
        assert torch.equal(running[k][0], running_before[k][0]) and torch.equal(running[k][1], running_before[k][1])


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", [(2, 3, 24, 24), (1, 3, 23, 21)], ids=["even", "odd"])
def test_stem_data_gradient_and_avgpool_backward(precision, shape):
    """mg_conv_backward_data on the strided stem descriptor and mg_avgpool_backward against oracle.nn_ops; same bits twice"""
    from util import conv_desc
    dtype = DT[precision]
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, dtype)
    rng = np.random.default_rng(4)
    N, Ci, H, W = shape
    Cout = 64
    x = _rnd(rng.standard_normal(shape), precision)
    w = bf16_round(rng.standard_normal((Cout, Ci, 7, 7)) * 0.1)
    Ho, Wo = (H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1
    g = _rnd(rng.standard_normal((N, Cout, Ho, Wo)), precision)
    X, Gg = Grid(dtype, N, Ci, H, W, x), Grid(dtype, N, Cout, Ho, Wo, g)
    d = conv_desc([X], [ffi.MG_SEG_SAME], 7, 2, 3, Cout, H, W)
    tw = torch.from_numpy(w.astype(np.float32)).cuda()
    tol = {"fp32": 1e-4, "bf16": 2e-2}[precision]
    outs = []
    for _ in range(2):
        DX = Grid(dtype, N, Ci, H, W)
        ctx.call("mg_conv_backward_data", C.byref(d), ptr(tw), None, C.byref(Gg.g()), C.byref(DX.g()))
        outs.append(DX)
    ref = NO.conv_backward(x, w, g, s=2, p=3)[0]
    assert rel_err(outs[0].nchw(), ref) <= tol
    assert not outs[0].pad_channels().any()
    assert torch.equal(outs[0].t, outs[1].t)
    for r in (2, 4):
        gp = _rnd(rng.standard_normal((N, Ci, H // r, W // r)), precision)
        GP, DI = Grid(dtype, N, Ci, H // r, W // r, gp), Grid(dtype, N, Ci, H, W)
        ctx.call("mg_avgpool_backward", C.byref(GP.g()), r, C.byref(DI.g()))
        assert rel_err(DI.nchw(), NO.avgpool_backward(gp, x.shape, r)) <= tol
        assert not DI.pad_channels().any()


@gpu
def test_two_gpu_syncbn_with_frozen_layers_equals_single_gpu():
    """-bnSync with the first quarter of the BatchNorm layers frozen: the two-GPU step equals the single-GPU step on the whole batch"""
    import os, subprocess, sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(root, "tests", "dp_frozen_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "dp-frozen ok rank 0" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
