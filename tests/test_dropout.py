"""nn.Dropout in training mode (include/mgconv.h: mg_dropout; models/cifar/pnmg.lua:25-27 with -isDropout).

CPU: the oracle's numpy Philox4x32-10 (oracle/dropout.py) reproduces the published known-answer vectors, and the lowering places one DropOp per
active nn.Dropout (training plans only; evaluation plans and models without dropout are unchanged).
GPU: the kernels against the numpy mask bit for bit, the keep fraction, mask independence across steps / ops / ranks, the
P-NMG-11 network against the fp64 oracle given the engine's masks, and the training step's reproducibility (two seeded runs,
lanes vs one lane, CUDA-graph replays vs eager steps).
"""
import copy
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import builders as OB, dropout as OD
from mgconv import builders as B, ffi, lower as L, ops as O
from util import Grid, copy_params_from_oracle, rel_err, bf16_round, emulate_bf16_storage

gpu = pytest.mark.gpu
PNMG_OPT = dict(nGPU=1, nLayer=1, blocks=B.CIFAR_RNMG_BLOCKS)
SHAPE = (16, 3, 32, 32)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_numpy_philox_known_answers(ctr, key, want):
    """Random123 kat_vectors, philox4x32 with 10 rounds"""
    got = OD.philox4x32_10(np.array(ctr, dtype=np.uint64), key)
    assert " ".join(f"{int(v):08x}" for v in got) == want


def test_mask_threshold_and_scale():
    assert OD.threshold(0.0) == 0 and OD.threshold(0.5) == 1 << 31
    assert OD.scale(0.2) == np.float32(1.0 / (1.0 - float(np.float32(0.2))))
    assert OD.keep_flat(1000, 0.0, 7, 0, 1, 0).all()


def _plan(train, dropout=True):
    m = B.cifar_pnmg.createModel(B.Opt(isDropout=dropout, **PNMG_OPT))
    if not train:
        m.evaluate()
    b, _ = L.trace_model(m, SHAPE)
    return m, b


def _signature(b):
    return [(type(o).__name__, [(t.name, t.C, t.H, t.W, m) for t, m in getattr(o, "segs", [])]) for o in b.ops]


def test_pnmg_dropout_training_plan():
    m, b = _plan(True)
    drops = [o for o in b.ops if isinstance(o, O.DropOp)]
    mods = [d for d in m.findModules("nn.Dropout") if d.p > 0]
    assert len(drops) == len(mods) == 11
    assert [o.ordinal for o in drops] == list(range(len(drops)))
    assert sorted({o.p for o in drops}) == [0.1, 0.2, 0.3, 0.4]
    assert sum(isinstance(o, O.DropStepOp) for o in b.ops) == 1
    assert b.ops.index(b.drop_step) < b.ops.index(drops[0])
    for d in drops:
        consumers = [o for o in b.ops if isinstance(o, O.ConvOp) and any(t is d.out for t, _ in o.segs)]
        assert len(consumers) == 1 and len(consumers[0].segs) == 1, d.out.name
        assert consumers[0].segs[0][1] == ffi.MG_SEG_SAME
        assert d.out.C == sum(t.C for t, _ in d.segs)
        assert {mo for _, mo in d.segs} <= {ffi.MG_SEG_SAME, ffi.MG_SEG_UP}
    # the 1x1 convolutions on the coarsest grids of blocks 4 and 5 are behind a dropout too
    assert any(c.k == 1 and c.segs[0][0].producer.__class__ is O.DropOp for c in b.ops if isinstance(c, O.ConvOp))


def test_oracle_places_dropouts_like_the_product():
    m, b = _plan(True)
    om = OD.cifar_pnmg(1, blocks=OB.CIFAR_RNMG_NARROW)
    assert [d.p for d in om.modules() if isinstance(d, OD.Dropout)] == [d.p for d in b.drops]
    with torch.no_grad():
        om(torch.zeros(2, 3, 32, 32))
    assert [d.last_shape[1:] for d in om.modules() if isinstance(d, OD.Dropout)] == [(d.out.C, d.out.H, d.out.W) for d in b.drops]


def test_pnmg_dropout_evaluation_plan_is_the_plain_plan():
    _, be = _plan(False)
    _, b0 = _plan(True, dropout=False)
    assert not be.drops and be.drop_step is None
    assert _signature(be) == _signature(b0)


def test_plan_key_depends_on_train_only_with_dropout():
    from mgconv.engine import engine_key
    x = torch.zeros(SHAPE)
    m, _ = _plan(True)
    drops = m.findModules("nn.Dropout")
    k_train = engine_key(x, drops)
    m.evaluate()
    assert engine_key(x, drops) != k_train
    for name, opt in (("ilsvrc/rnmg", dict(depth=34)), ("cifar/prnmg", dict(nLayer=2)), ("cifar/pnmg", dict(nLayer=1))):
        net = B.load_net(name)
        mm = net.createModel(B.Opt(nGPU=1, **opt))
        shape = (2, 3, 224, 224) if name == "ilsvrc/rnmg" else SHAPE
        b, _ = L.trace_model(mm, shape)
        assert not b.drops and b.drop_step is None
        assert not any(isinstance(o, (O.DropOp, O.DropStepOp)) for o in b.ops)
        xs = torch.zeros(shape)
        k = engine_key(xs, mm.findModules("nn.Dropout"))
        mm.evaluate()
        assert engine_key(xs, mm.findModules("nn.Dropout")) == k == engine_key(xs)


def test_dropout_rejects_p_outside_unit_interval():
    from mgconv import nn
    for p in (-0.1, 1.0):
        seq = nn.Sequential().add(nn.Dropout(p)).add(nn.SpatialConvolution(8, 8, 3, 3, 1, 1, 1, 1))
        with pytest.raises(ValueError):
            L.trace_model(seq, (2, 8, 4, 4))


# ------------------------------------------------------------------------------------------------ GPU, kernels
DT = {"fp32": ffi.MG_F32, "bf16": ffi.MG_BF16}


def _ctx(dtype):
    return ffi.Context(0, torch.cuda.current_stream().cuda_stream, dtype)


def _dp(p, op, rank, seed, step):
    return ffi.mg_dropout(p, op, rank, seed, step.data_ptr())


def _round(a, dtype):
    return bf16_round(a) if dtype == ffi.MG_BF16 else np.asarray(a, dtype=np.float32).astype(np.float64)


def _segments(ctx, dtype, rng, N, H, cs):
    """SAME (C cs[0]) + SAME pooled companion of an odd (2H-1)x(2H-1) grid (C cs[1]) + UP of an (H/2)x(H/2) grid (C cs[2])"""
    a = Grid(dtype, N, cs[0], H, H, nchw=rng.standard_normal((N, cs[0], H, H)))
    fine = Grid(dtype, N, cs[1], 2 * H - 1, 2 * H - 1, nchw=rng.standard_normal((N, cs[1], 2 * H - 1, 2 * H - 1)))
    pooled = Grid(dtype, N, cs[1], H, H)
    ctx.call("mg_pool_forward", C.byref(fine.g()), C.byref(pooled.g()), 0, None)
    up = Grid(dtype, N, cs[2], H // 2, H // 2, nchw=rng.standard_normal((N, cs[2], H // 2, H // 2)))
    cat = np.concatenate([a.nchw(), pooled.nchw(), up.nchw().repeat(2, 2).repeat(2, 3)], 1)
    return [a, pooled, up], [ffi.MG_SEG_SAME, ffi.MG_SEG_SAME, ffi.MG_SEG_UP], cat


def _forward(ctx, dp, segs, modes, out):
    n = len(segs)
    ctx.call("mg_dropout_forward", C.byref(dp), n, (ffi.mg_grid * n)(*[s.g() for s in segs]), (C.c_int32 * n)(*modes), C.byref(out.g()))


def _expect(x, keep, p, dtype):
    s = OD.scale(p)
    return _round(np.where(keep, (np.asarray(x, np.float32) * s).astype(np.float64), 0.0), dtype)


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("cs", [(5, 3, 6), (8, 16, 8)], ids=["unaligned", "aligned"])
def test_dropout_forward_backward_bit_exact(precision, cs):
    dtype = DT[precision]
    ctx = _ctx(dtype)
    rng = np.random.default_rng(1)
    N, H, p, seed, op, rank = 3, 6, 0.3, 0x1234_5678_9abc_def0, 2, 1
    segs, modes, cat = _segments(ctx, dtype, rng, N, H, cs)
    Ct = sum(cs)
    out = Grid(dtype, N, Ct, H, H)
    out.t.fill_(7.0)   # every element, pad channels included, must be written
    step = torch.tensor([5], dtype=torch.int64, device="cuda")
    dp = _dp(p, op, rank, seed, step)
    _forward(ctx, dp, segs, modes, out)
    keep = OD.keep_nchw(N, Ct, H, H, p, seed, op, 5, rank)
    assert np.array_equal(out.nchw(), _expect(cat, keep, p, dtype))
    assert not out.pad_channels().any()
    g = Grid(dtype, N, Ct, H, H, nchw=rng.standard_normal((N, Ct, H, H)))
    g0 = g.nchw()
    ctx.call("mg_dropout_backward", C.byref(dp), C.byref(g.g()))
    assert np.array_equal(g.nchw(), _expect(g0, keep, p, dtype))
    assert not g.pad_channels().any()


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("p", [0.1, 0.4])
def test_dropout_keep_fraction(precision, p):
    dtype = DT[precision]
    ctx = _ctx(dtype)
    N, Cc, H = 64, 64, 32          # 4.19M elements
    x = Grid(dtype, N, Cc, H, H)
    x.t[..., :Cc] = 1.0
    out = Grid(dtype, N, Cc, H, H)
    step = torch.tensor([1], dtype=torch.int64, device="cuda")
    _forward(ctx, _dp(p, 0, 0, 99, step), [x], [ffi.MG_SEG_SAME], out)
    torch.cuda.synchronize()
    n = N * Cc * H * H
    kept = int((out.t[..., :Cc] != 0).sum())
    sigma = math.sqrt(p * (1 - p) / n)
    assert abs(kept / n - (1 - p)) <= 5 * sigma, (kept / n, 1 - p, sigma)
    vals = out.t[..., :Cc][out.t[..., :Cc] != 0].float().unique().cpu().numpy()
    assert np.array_equal(vals, [float(_round(OD.scale(p), dtype))])


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_masks_differ_between_steps_ops_and_ranks(precision):
    dtype = DT[precision]
    ctx = _ctx(dtype)
    N, Cc, H = 4, 24, 8
    x = Grid(dtype, N, Cc, H, H)
    x.t[..., :Cc] = 1.0
    step = torch.tensor([0], dtype=torch.int64, device="cuda")

    def mask(op, rank):
        out = Grid(dtype, N, Cc, H, H)
        _forward(ctx, _dp(0.5, op, rank, 42, step), [x], [ffi.MG_SEG_SAME], out)
        return out.nchw() != 0
    ctx.call("mg_dropout_advance", ffi.ptr(step))
    m1 = mask(0, 0)
    ctx.call("mg_dropout_advance", ffi.ptr(step))
    torch.cuda.synchronize()
    assert int(step.item()) == 2
    m2 = mask(0, 0)
    assert np.array_equal(m1, OD.keep_nchw(N, Cc, H, H, 0.5, 42, 0, 1, 0))
    assert np.array_equal(m2, OD.keep_nchw(N, Cc, H, H, 0.5, 42, 0, 2, 0))
    for a, b in ((m1, m2), (m2, mask(1, 0)), (m2, mask(0, 1))):     # step, op, rank
        assert not np.array_equal(a, b)
        assert 0.3 < (a == b).mean() < 0.7   # independent masks of p = 0.5 agree on about half the elements


@gpu
@pytest.mark.parametrize("p", [-0.1, 1.0, 1.5, float("nan")])
def test_dropout_rejects_bad_p(p):
    ctx = _ctx(ffi.MG_BF16)
    x = Grid(ffi.MG_BF16, 1, 8, 2, 2)
    out = Grid(ffi.MG_BF16, 1, 8, 2, 2)
    step = torch.zeros(1, dtype=torch.int64, device="cuda")
    with pytest.raises(ffi.MGError, match="outside"):
        _forward(ctx, _dp(p, 0, 0, 1, step), [x], [ffi.MG_SEG_SAME], out)
    with pytest.raises(ffi.MGError, match="outside"):
        ctx.call("mg_dropout_backward", C.byref(_dp(p, 0, 0, 1, step)), C.byref(x.g()))


# ------------------------------------------------------------------------------------------------ GPU, network
def _set_oracle_masks(om, eng):
    """give the oracle's Dropout modules the engine's (seed, op, step, rank); module order = plan order of the DropOps"""
    mods = [m for m in om.modules() if isinstance(m, OD.Dropout)]
    drops = eng.plan.drops
    assert len(mods) == len(drops)
    step = int(eng.plan.drop_step.step.item())
    for m, d in zip(mods, drops):
        m.seed, m.op, m.step, m.rank = eng.dropout_seed, d.ordinal, step, eng.dropout_rank
    return mods, drops


@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_pnmg_dropout_network_follows_the_oracle(precision):
    """P-NMG-11 narrow with -isDropout, one training step, against the fp64 oracle drawing the engine's masks"""
    torch.manual_seed(2)
    rng = np.random.default_rng(5)
    om = OD.cifar_pnmg(1, blocks=OB.CIFAR_RNMG_NARROW).double()
    pm = B.cifar_pnmg.createModel(B.Opt(isDropout=True, **PNMG_OPT))
    pm.precision = precision
    olist, plist = copy_params_from_oracle(om, pm, bf16_weights=precision == "bf16")
    pm.cuda()
    plist = [m for m in pm.listModules() if m.own_parameters()]
    x = bf16_round(rng.standard_normal(SHAPE))
    t = rng.integers(1, 101, SHAPE[0])
    crit = B.cifar_pnmg.createCriterion()
    xd, td = _t(x).float().cuda(), _t(t).cuda()
    outputs, err = B.cifar_pnmg.ftrain(xd, td, pm, crit)
    torch.cuda.synchronize()
    eng = pm._engine
    assert int(eng.plan.drop_step.step.item()) == 1
    mods, drops = _set_oracle_masks(om, eng)
    loss_fn = lambda m: torch.nn.functional.nll_loss(m(_t(x)), _t(t - 1))
    olp = om(_t(x))
    oloss = torch.nn.functional.nll_loss(olp, _t(t - 1))
    oloss.backward()
    for m, d in zip(mods, drops):
        assert m.last_shape == (d.out.N, d.out.C, d.out.H, d.out.W)
    e_storage = 0.0
    if precision == "bf16":
        # the dropped tensor is one more bf16 storage point of the product
        def extra(m16):
            for m in m16.modules():
                if isinstance(m, OD.Dropout):
                    m.register_forward_hook(lambda _m, _i, o: o.to(torch.bfloat16).to(o.dtype))
        om16 = emulate_bf16_storage(copy.deepcopy(om))
        extra(om16)
        for m in om16.modules():
            for p_ in m.parameters(recurse=False):
                p_.grad = None
        loss_fn(om16).backward()
        o16 = [m for m in om16.modules() if isinstance(m, (torch.nn.Conv2d, torch.nn.BatchNorm2d, torch.nn.Linear))]
        g16, g64 = [], []
        for a, b16 in zip(olist, o16):
            g64.append(a.weight.grad.numpy().ravel()); g16.append(b16.weight.grad.numpy().ravel())
            if not isinstance(a, torch.nn.Conv2d):
                g64.append(a.bias.grad.numpy().ravel()); g16.append(b16.bias.grad.numpy().ravel())
        e_storage = rel_err(np.concatenate(g16), np.concatenate(g64))
    tol = {"fp32": 1e-4, "bf16": 2e-2}[precision]
    e = rel_err(outputs.cpu().numpy(), olp.detach().numpy())
    assert e <= tol, ("log-probabilities", e)
    assert abs(float(err) - oloss.item()) <= tol * max(1.0, abs(oloss.item())), "loss"
    og, pg = [], []
    for o, p in zip(olist, plist):
        og.append(o.weight.grad.numpy().ravel()); pg.append(p.gradWeight.cpu().numpy().ravel())
        if p.typename != "cudnn.SpatialConvolution":
            og.append(o.bias.grad.numpy().ravel()); pg.append(p.gradBias.cpu().numpy().ravel())
    eg = rel_err(np.concatenate(pg), np.concatenate(og))
    gtol = 1e-4 if precision == "fp32" else max(tol, 1.1 * e_storage)
    print(f"[measured] P-NMG-11 isDropout {precision}: log-prob {e:.2e}, gradient {eg:.2e} (storage-only {e_storage:.2e})")
    assert eg <= gtol, ("parameter gradients", eg, "storage-only", e_storage)

    # evaluate(): the same weights in a model without dropout give the same bits
    pm.evaluate()
    ev = pm.forward(xd).clone()
    assert not pm._engine.plan.drops
    p0 = B.cifar_pnmg.createModel(B.Opt(isDropout=False, **PNMG_OPT))
    p0.precision = precision
    p0.cuda()
    for a, b_ in zip([m for m in p0.listModules() if m.own_parameters()], plist):
        for name in ("weight", "bias", "running_mean", "running_var"):
            if hasattr(b_, name):
                getattr(a, name).copy_(getattr(b_, name))
    p0.evaluate()
    ev0 = p0.forward(xd)
    torch.cuda.synchronize()
    assert torch.equal(ev, ev0)


# ------------------------------------------------------------------------------------------------ GPU, step
def _model(precision="bf16", seed=11):
    torch.manual_seed(seed)
    pm = B.cifar_pnmg.createModel(B.Opt(isDropout=True, **PNMG_OPT))
    pm.precision = precision
    pm.cuda()
    return pm


def _batch(seed=3):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(*SHAPE, generator=g).cuda(), torch.randint(1, 101, (SHAPE[0],), generator=g).cuda()


@gpu
def test_seeded_sgd_steps_are_bit_identical():
    res = []
    for _ in range(2):
        pm = _model()
        params, grads = pm.getParameters()
        crit = B.cifar_pnmg.createCriterion()
        x, t = _batch()
        st = dict(learningRate=0.05, momentum=0.9, weightDecay=5e-4, dampening=0.0)
        for _ in range(3):
            pm.zeroGradParameters()

            def feval(_p):
                B.cifar_pnmg.ftrain(x, t, pm, crit)
                return 0.0, grads
            B.cifar_pnmg.btrain(params, feval, st)
        torch.cuda.synchronize()
        assert int(pm._engine.plan.drop_step.step.item()) == 3
        res.append(params.clone())
    assert torch.equal(res[0], res[1]), float((res[0] - res[1]).abs().max())


@gpu
def test_lanes_equal_serial_plan_with_dropout(monkeypatch):
    outs = {}
    for lanes in ("1", "3"):
        monkeypatch.setenv("MGCONV_LANES", lanes)
        monkeypatch.setenv("MGCONV_AUTOTUNE", "0")
        pm = _model()
        params, grads = pm.getParameters()
        crit = B.cifar_pnmg.createCriterion()
        x, t = _batch()
        pm.zeroGradParameters()
        out, err = B.cifar_pnmg.ftrain(x, t, pm, crit)
        torch.cuda.synchronize()
        assert pm._engine.n_lanes == int(lanes)
        outs[lanes] = (out.clone(), float(err), grads.clone())
    assert outs["1"][1] == outs["3"][1]
    assert torch.equal(outs["1"][0], outs["3"][0])
    assert torch.equal(outs["1"][2], outs["3"][2])


@gpu
def test_graph_replays_draw_new_masks_like_eager_steps():
    """a captured step advances the device counter on every replay: three replays = three eager steps, bit for bit, and
    consecutive steps use different masks"""
    from mgconv.graph import GraphedStep
    x, t = _batch()
    runs = {}
    for mode in ("eager", "graph"):
        pm = _model()
        params, grads = pm.getParameters()
        crit = B.cifar_pnmg.createCriterion()
        xs, ts = x.clone(), t.clone()
        out = {}

        def step():
            pm.zeroGradParameters()
            out["o"], _ = B.cifar_pnmg.ftrain(xs, ts, pm, crit)
        step()                                   # plans, autotuning and workspaces before capture
        torch.cuda.synchronize()
        run = step
        if mode == "graph":
            run = GraphedStep(step)
        counter = pm._engine.plan.drop_step.step
        counter.zero_()
        res = []
        for _ in range(3):
            run()
            torch.cuda.synchronize()
            res.append((int(counter.item()), out["o"].clone(), grads.clone()))
        runs[mode] = res
    for (s0, o0, g0), (s1, o1, g1) in zip(runs["eager"], runs["graph"]):
        assert s0 == s1
        assert torch.equal(o0, o1) and torch.equal(g0, g1)
    assert [s for s, _, _ in runs["graph"]] == [1, 2, 3]
    assert not torch.equal(runs["eager"][0][2], runs["eager"][1][2])


@gpu
def test_data_parallel_ranks_draw_different_masks():
    """the rank a DataParallel hands to its engine is a word of the mask counter: same step, different rank, different mask"""
    pm = _model()
    x, _ = _batch()
    pm.forward(x)
    eng = pm._engine
    outs = []
    for rank in (0, 1, 0):
        eng.dropout_rank = rank
        eng.plan.drop_step.step.zero_()
        outs.append(pm.forward(x).clone())
    torch.cuda.synchronize()
    assert all(d.dp.rank == 0 for d in eng.plan.drops)
    assert torch.equal(outs[0], outs[2])
    assert not torch.equal(outs[0], outs[1])
