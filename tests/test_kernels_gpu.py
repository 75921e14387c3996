"""GPU parity tests of every libmgconv entry point against the CPU oracle (oracle/nn_ops.py),
called through the C ABI exactly as the LuaJIT/ctypes host does.

Bars (BASELINE.json north_star): pool arg-max indices and up-sample gathers bit-exact;
floating point within rel 1e-4 in fp32 mode and rel 2e-2 in bf16 (fp32 accumulate) mode.
Inputs are rounded to bf16-representable values first, so both sides read identical numbers.
"""
import ctypes as C
import os
import numpy as np
import pytest
import torch

from oracle import nn_ops as O
from mgconv import ffi
from mgconv.ffi import ptr, mg_grad_src, MG_SEG_SAME, MG_SEG_POOL, MG_SEG_UP, MG_SRC_POOL3
from util import Grid, conv_desc, dev, rel_err, max_rel, elem_rel, bf16_round, TOL, TDT, new_sums, sums_value

pytestmark = pytest.mark.gpu
DTYPES = [ffi.MG_F32, ffi.MG_BF16]
rng = np.random.default_rng(7)


@pytest.fixture(scope="module", params=DTYPES, ids=["fp32", "bf16"])
def ctx(request):
    c = ffi.Context(0, torch.cuda.current_stream().cuda_stream, request.param)
    yield c
    c.sync()
    c.close()


def rnd(*shape):
    return bf16_round(rng.standard_normal(shape))


# ---------------------------------------------------------------- layout
def test_import_export_roundtrip(ctx):
    x = rnd(2, 5, 7, 6)
    g = Grid(ctx.dtype, 2, 5, 7, 6)
    ctx.call("mg_import_nchw", ptr(dev(x)), C.byref(g.g()))
    assert np.array_equal(g.nchw(), x)
    assert not g.pad_channels().any()
    out = torch.empty(2, 5, 7, 6, device="cuda")
    g.affine(np.full(5, 2.0), np.full(5, -1.0), True)
    ctx.call("mg_export_nchw", C.byref(g.g()), ptr(out))
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), np.maximum(2 * x - 1, 0).astype(np.float32))


# ---------------------------------------------------------------- pooling / up-sampling (bit-exact)
@pytest.mark.parametrize("H,W", [(8, 8), (7, 7), (5, 9), (1, 1), (2, 3), (56, 56)])
def test_pool2x2_ceil_values_and_argmax_bit_exact(ctx, H, W):
    x = rnd(2, 11, H, W)
    x[0, 0, :min(2, H), :min(2, W)] = 1.5  # ties: the first maximum of the row-major scan must win
    x[1, 3] = 0.25                          # a whole plane of ties
    y, idx = O.maxpool_forward(x)
    gi = Grid(ctx.dtype, 2, 11, H, W, x)
    go = Grid(ctx.dtype, 2, 11, y.shape[2], y.shape[3])
    am = torch.full((2, y.shape[2], y.shape[3], 11), -1, dtype=torch.int32, device="cuda")
    ctx.call("mg_pool_forward", C.byref(gi.g()), C.byref(go.g()), 0, ptr(am))
    assert np.array_equal(go.nchw(), y)
    assert np.array_equal(am.permute(0, 3, 1, 2).cpu().numpy(), idx)


def test_pool_with_channel_offset_and_copy_channels(ctx):
    """mgPool isConcat: JoinTable(2){pool(x_{n-1}), x_n} (models/ilsvrc/rnmg.lua:201-207)"""
    a, b = rnd(2, 6, 6, 6), rnd(2, 5, 3, 3)
    ga, gb = Grid(ctx.dtype, 2, 6, 6, 6, a), Grid(ctx.dtype, 2, 5, 3, 3, b)
    out = Grid(ctx.dtype, 2, 11, 3, 3)
    ctx.call("mg_pool_forward", C.byref(ga.g()), C.byref(out.g()), 0, None)
    ctx.call("mg_copy_channels", C.byref(gb.g()), C.byref(out.g()), 6)
    ref = np.concatenate([O.maxpool_forward(a)[0], b], axis=1)
    assert np.array_equal(out.nchw(), ref)


def test_stem_pool3x3s2p1(ctx):
    x = rnd(2, 9, 12, 12)
    y, _ = O.maxpool_forward(x, 3, 2, 1, ceil_mode=False)
    gi, go = Grid(ctx.dtype, 2, 9, 12, 12, x), Grid(ctx.dtype, 2, 9, 6, 6)
    code = torch.zeros((2, 6, 6, go.Cp), dtype=torch.uint8, device="cuda") if ctx.dtype == ffi.MG_BF16 else None
    ctx.call("mg_pool3s2_forward", C.byref(gi.g()), C.byref(go.g()), ptr(code))
    assert np.array_equal(go.nchw(), y)
    if code is not None:  # arg-max codes ky*3+kx of the 3x3 window <-> the oracle's flat input index
        _, idx = O.maxpool_forward(x, 3, 2, 1, ceil_mode=False)
        cd = code[..., :9].permute(0, 3, 1, 2).cpu().numpy().astype(np.int64)
        oy, ox = np.meshgrid(np.arange(6), np.arange(6), indexing="ij")
        assert np.array_equal((2 * oy - 1 + cd // 3) * 12 + (2 * ox - 1 + cd % 3), idx)


def test_avgpool_and_global_avgpool(ctx):
    x = rnd(2, 3, 8, 8)
    gi, go = Grid(ctx.dtype, 2, 3, 8, 8, x), Grid(ctx.dtype, 2, 3, 2, 2)
    ctx.call("mg_avgpool_forward", C.byref(gi.g()), 4, C.byref(go.g()))
    assert max_rel(go.nchw(), O.avgpool_forward(x, 4)) <= TOL[ctx.dtype]
    x = rnd(3, 10, 7, 7)
    gi, go = Grid(ctx.dtype, 3, 10, 7, 7, x), Grid(ctx.dtype, 3, 10, 1, 1)
    ctx.call("mg_global_avgpool_forward", C.byref(gi.g()), C.byref(go.g()))
    assert max_rel(go.nchw(), O.avgpool_forward(x, 7, 1)) <= TOL[ctx.dtype]
    d = rnd(3, 10, 1, 1)
    gd, gin = Grid(ctx.dtype, 3, 10, 1, 1, d), Grid(ctx.dtype, 3, 10, 7, 7)
    ctx.call("mg_global_avgpool_backward", C.byref(gd.g()), C.byref(gin.g()))
    assert max_rel(gin.nchw(), O.avgpool_backward(d, x.shape, 7, 1)) <= TOL[ctx.dtype]


# ---------------------------------------------------------------- the multigrid convolution
def _mg_inputs(N, cs, H):
    """finer (2H), same (H), coarser (H/2) grids"""
    return rnd(N, cs[0], 2 * H, 2 * H), rnd(N, cs[1], H, H), rnd(N, cs[2], H // 2, H // 2)


def _oracle_cat(f, s, c):
    pooled, idx = O.maxpool_forward(f)
    return np.concatenate([pooled, s, O.upsample_forward(c)], axis=1), idx


CONV_CASES = [  # N, (C_finer, C_same, C_coarser), H, Cout, k
    (2, (5, 7, 3), 8, 6, 3),
    (2, (16, 8, 8), 14, 24, 3),     # odd finer size is impossible here; 14 -> finer 28, coarser 7
    (1, (64, 32, 16), 28, 32, 3),   # R-MG-34 block-1 grid 2 (models/ilsvrc/rnmg.lua:250)
    (2, (8, 12, 4), 4, 10, 1),      # 1x1 kernel of the coarsest CIFAR grids (models/cifar/nmg.lua:152-153)
    (3, (40, 20, 10), 2, 20, 3),    # 2x2 grid: every tap hits the border
]


@pytest.mark.parametrize("case", CONV_CASES)
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_mgconv_forward_dgrad_wgrad(ctx, case, impl):
    if impl == "auto" and ctx.dtype != ffi.MG_BF16:
        pytest.skip("tcgen05 path is bf16 only")
    N, cs, H, Cout, k = case
    pad = 0 if k == 1 else 1
    f, s, c = _mg_inputs(N, cs, H)
    cat, idx = _oracle_cat(f, s, c)
    w = bf16_round(rng.standard_normal((Cout, sum(cs), k, k)) * 0.2)
    b = bf16_round(rng.standard_normal(Cout) * 0.1)
    y_ref = O.conv_forward(cat, w, b, 1, pad)
    ctx.set_impl(ffi.MG_IMPL_SIMT if impl == "simt" else ffi.MG_IMPL_AUTO)
    gf, gs, gc = Grid(ctx.dtype, N, cs[0], 2 * H, 2 * H, f), Grid(ctx.dtype, N, cs[1], H, H, s), Grid(ctx.dtype, N, cs[2], H // 2, H // 2, c)
    # the tcgen05 path gathers by pure copies: its POOL operand is the pooled companion tensor
    if impl == "auto":
        gp = Grid(ctx.dtype, N, cs[0], H, H)
        ctx.call("mg_pool_forward", C.byref(gf.g()), C.byref(gp.g()), 0, None)
        d = conv_desc([gp, gs, gc], [MG_SEG_SAME, MG_SEG_SAME, MG_SEG_UP], k, 1, pad, Cout, H, H)
    else:
        d = conv_desc([gf, gs, gc], [MG_SEG_POOL, MG_SEG_SAME, MG_SEG_UP], k, 1, pad, Cout, H, H)
    wd, bd = dev(w), dev(b)
    wpack = wpack_t = None
    nb = ffi.lib.mg_conv_packed_bytes(C.byref(d), 0) if impl == "auto" else 0
    if nb:
        wpack = torch.zeros(nb, dtype=torch.uint8, device="cuda")
        wpack_t = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 1), dtype=torch.uint8, device="cuda")
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wpack), 0)
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wpack_t), 1)
    gy = Grid(ctx.dtype, N, Cout, H, H)
    sums = new_sums(2 * Cout)
    tc0 = ctx.tc_launches()
    ctx.call("mg_conv_forward", C.byref(d), ptr(wd), ptr(wpack), ptr(bd), C.byref(gy.g()), ptr(sums))
    assert ctx.tc_launches() - tc0 == (1 if impl == "auto" else 0), "forward must run on the tcgen05 kernel in auto/bf16 mode"
    tol = TOL[ctx.dtype]
    y = gy.nchw()
    assert max_rel(y, y_ref) <= tol, max_rel(y, y_ref)
    assert elem_rel(y, y_ref) <= tol, ("per-element", elem_rel(y, y_ref))
    assert not gy.pad_channels().any()
    # BatchNorm statistics accumulated by the conv
    cnt = N * H * H
    sm = sums_value(sums).cpu().numpy()
    assert np.allclose(sm[:Cout] / cnt, y_ref.mean(axis=(0, 2, 3)), atol=tol * np.abs(y_ref).max())
    assert np.allclose(sm[Cout:] / cnt, (y_ref ** 2).mean(axis=(0, 2, 3)), rtol=4 * tol, atol=tol)

    # backward: dcat (gradient w.r.t. the concatenated input), dW, dbias
    g = rnd(N, Cout, H, H)
    gcat_ref, gw_ref, gb_ref = O.conv_backward(cat, w, g, 1, pad)
    gg = Grid(ctx.dtype, N, Cout, H, H, g)
    cps = [gf.Cp, gs.Cp, gc.Cp]
    dcat = Grid(ctx.dtype, N, sum(cps), H, H, Cp=sum(cps))
    tc0 = ctx.tc_launches()
    ctx.call("mg_conv_backward_data", C.byref(d), ptr(wd), ptr(wpack_t), C.byref(gg.g()), C.byref(dcat.g()))
    assert ctx.tc_launches() - tc0 == (1 if impl == "auto" else 0), "dgrad must run on the tcgen05 kernel in auto/bf16 mode"
    dc = dcat.nchw()
    got = np.concatenate([dc[:, 0:cs[0]], dc[:, cps[0]:cps[0] + cs[1]], dc[:, cps[0] + cps[1]:cps[0] + cps[1] + cs[2]]], axis=1)
    assert max_rel(got, gcat_ref) <= tol, max_rel(got, gcat_ref)
    assert elem_rel(got, gcat_ref) <= tol, ("per-element", elem_rel(got, gcat_ref))
    dw = torch.zeros_like(wd)
    db = torch.zeros_like(bd)
    tc0 = ctx.tc_launches()
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 1.0)
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 0.5)  # accGradParameters accumulates
    assert ctx.tc_launches() - tc0 == (2 if impl == "auto" else 0), "wgrad must run on the tcgen05 kernel in auto/bf16 mode"
    torch.cuda.synchronize()
    assert max_rel(dw.cpu().numpy(), 1.5 * gw_ref) <= tol, max_rel(dw.cpu().numpy(), 1.5 * gw_ref)
    assert elem_rel(dw.cpu().numpy(), 1.5 * gw_ref) <= tol, ("per-element", elem_rel(dw.cpu().numpy(), 1.5 * gw_ref))
    assert max_rel(db.cpu().numpy(), 1.5 * gb_ref) <= tol
    ctx.set_impl(ffi.MG_IMPL_AUTO)


EDGE_CASES = [  # N, [(C, mode 's'|'u')], H, W, Cout, k -- shapes that take the less-travelled paths
    (1, [(8, "s")], 1, 1, 16, 3),                 # 1x1 grid: only the centre tap is ever in bounds (CIFAR coarsest grid)
    (2, [(24, "s"), (8, "u")], 6, 10, 520, 3),    # non-square, Cout > 256 -> several N tiles, rows spanning images
    (1, [(16, "s")], 5, 70, 8, 3),                # W > 64: per-tap tcgen05 kernels instead of the halo kernels
    (3, [(3, "s")], 9, 7, 40, 3),                 # Cin = 3 (Cp = 8, five zero channels), odd sizes
    (2, [(72, "s"), (40, "s"), (16, "u")], 4, 4, 24, 1),   # 1x1 kernel over three segments (CIFAR last blocks)
    (5, [(200, "s")], 3, 3, 96, 3),               # K spanning several 64-channel chunks with a ragged last chunk
]


EDGE_CASES += [
    (9, [(40, "s"), (24, "u")], 8, 12, 48, 3),    # two chunks, ragged last 256-slot tile (9 * 9 * 13 = 1053 slots)
    (4, [(136, "s")], 14, 14, 136, 3),            # three chunks with a ragged tail, N tile 144
    (2, [(16, "s"), (8, "u")], 64, 64, 24, 3),    # W = 64: the widest grid the halo kernels take (MNIST-cluttered 64x64 scale)
    (3, [(160, "s"), (80, "u")], 8, 8, 160, 3),   # dgrad column tile of 240 > threads of the CTA (bias tile filled by a loop), tap-packed last chunk
]
# kernel-selection overrides: automatic, two sub-tiles per CTA, persistent weight-resident kernel
# (context sub-tile override, context persistent override, per-layer algo of the descriptor)
TUNINGS = [(0, 0, 0), (2, 2, 0), (1, 1, 0), (0, 0, ffi.MG_ALGO_TILE128_DEEP), (0, 0, ffi.MG_ALGO_TILE256_DEEP), (0, 2, ffi.MG_ALGO_RESIDENT),
           (0, 0, ffi.MG_ALGO_TILE128_MID), (0, 0, ffi.MG_ALGO_PAIR128), (0, 0, ffi.MG_ALGO_PAIR256), (0, 2, ffi.MG_ALGO_RESIDENT_PAIR)]


@pytest.mark.parametrize("tuning", TUNINGS, ids=["auto", "subtiles2", "persistent", "algo_tile128deep", "algo_tile256deep", "algo_resident", "algo_tile128mid", "algo_pair128", "algo_pair256", "algo_resident_pair"])
@pytest.mark.parametrize("case", EDGE_CASES, ids=[f"case{i}" for i in range(len(EDGE_CASES))])
def test_conv_edge_shapes_tcgen05(case, tuning):
    """forward / dgrad / wgrad of the bf16 tensor-core path on ragged, tiny, wide and multi-tile shapes,
    under each variant of the 3x3 kernel (mg_ctx_set_tuning)"""
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    ctx.set_tuning(ffi.MG_TUNE_HALO_SUBTILES, tuning[0])
    ctx.set_tuning(ffi.MG_TUNE_PERSISTENT, tuning[1])
    N, segs, H, W, Cout, k = case
    pad = 0 if k == 1 else 1
    xs, grids, modes = [], [], []
    for c, m in segs:
        h, w = (H // 2, W // 2) if m == "u" else (H, W)
        x = rnd(N, c, h, w)
        xs.append(O.upsample_forward(x) if m == "u" else x)
        grids.append(Grid(ffi.MG_BF16, N, c, h, w, x)); modes.append(MG_SEG_UP if m == "u" else MG_SEG_SAME)
    cat = np.concatenate(xs, axis=1)
    wgt = bf16_round(rng.standard_normal((Cout, cat.shape[1], k, k)) * 0.1)
    b = bf16_round(rng.standard_normal(Cout) * 0.1)
    d = conv_desc(grids, modes, k, 1, pad, Cout, H, W)
    d.algo_fwd = d.algo_bwd_data = tuning[2]
    wd, bd = dev(wgt), dev(b)
    wp = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 0), dtype=torch.uint8, device="cuda")
    wpt = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 1), dtype=torch.uint8, device="cuda")
    ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wp), 0)
    ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wpt), 1)
    gy = Grid(ffi.MG_BF16, N, Cout, H, W)
    sums = new_sums(2 * Cout)
    tc0 = ctx.tc_launches()
    ctx.call("mg_conv_forward", C.byref(d), ptr(wd), ptr(wp), ptr(bd), C.byref(gy.g()), ptr(sums))
    y_ref = O.conv_forward(cat, wgt, b, 1, pad)
    tol = TOL[ffi.MG_BF16]
    assert max_rel(gy.nchw(), y_ref) <= tol
    assert not gy.pad_channels().any()
    assert np.allclose(sums_value(sums).cpu().numpy()[:Cout] / (N * H * W), y_ref.mean(axis=(0, 2, 3)), atol=tol * np.abs(y_ref).max())
    assert np.allclose(sums_value(sums).cpu().numpy()[Cout:] / (N * H * W), (y_ref ** 2).mean(axis=(0, 2, 3)), rtol=4 * tol, atol=tol)
    g = rnd(N, Cout, H, W)
    gcat_ref, gw_ref, gb_ref = O.conv_backward(cat, wgt, g, 1, pad)
    gg = Grid(ffi.MG_BF16, N, Cout, H, W, g)
    cps = [x.Cp for x in grids]
    dcat = Grid(ffi.MG_BF16, N, sum(cps), H, W, Cp=sum(cps))
    ctx.call("mg_conv_backward_data", C.byref(d), ptr(wd), ptr(wpt), C.byref(gg.g()), C.byref(dcat.g()))
    dc, off, lo = dcat.nchw(), 0, 0
    for (c, m), cp in zip(segs, cps):   # dcat is laid out at padded channel offsets, at the conv's own resolution
        assert max_rel(dc[:, off:off + c], gcat_ref[:, lo:lo + c]) <= tol, ("dgrad segment", c, m)
        assert not np.abs(dc[:, off + c:off + cp]).any()
        off += cp; lo += c
    dw, db = torch.zeros_like(wd), torch.zeros_like(bd)
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 1.0)
    assert ctx.tc_launches() - tc0 == 3, "all three passes must run on tcgen05 kernels"
    torch.cuda.synchronize()
    assert max_rel(dw.cpu().numpy(), gw_ref) <= tol and max_rel(db.cpu().numpy(), gb_ref) <= tol
    ctx.close()


def test_null_and_mismatched_arguments_return_status(ctx):
    """error convention: status + message, never a crash (SURVEY section 8b)"""
    g = Grid(ctx.dtype, 1, 4, 4, 4)
    o = Grid(ctx.dtype, 1, 4, 3, 3)   # wrong pooled size
    with pytest.raises(ffi.MGError, match="pool"):
        ctx.call("mg_pool_forward", C.byref(g.g()), C.byref(o.g()), 0, None)
    assert ffi.lib.mg_pool_forward(ctx.h, None, None, 0, None) == 1      # MG_ERR_INVALID_ARG
    assert ffi.lib.mg_conv_forward(None, None, None, None, None, None, None) == 1
    with pytest.raises(ffi.MGError, match="communicator not initialised"):
        ctx.call("mg_allreduce_launch", ptr(g.t), 16, 0)


@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_stem_conv7x7_stride2(ctx, impl):
    """cudnn.SpatialConvolution(3, nOP, 7,7, 2,2, 3,3) of the ImageNet stem (ilsvrc/rnmg.lua:180)"""
    if impl == "auto" and ctx.dtype != ffi.MG_BF16:
        pytest.skip("tcgen05 path is bf16 only")
    x = rnd(2, 3, 20, 20)
    w = bf16_round(rng.standard_normal((16, 3, 7, 7)) * 0.1)
    b = bf16_round(rng.standard_normal(16) * 0.1)
    y_ref = O.conv_forward(x, w, b, 2, 3)
    ctx.set_impl(ffi.MG_IMPL_SIMT if impl == "simt" else ffi.MG_IMPL_AUTO)
    gx = Grid(ctx.dtype, 2, 3, 20, 20, x)
    d = conv_desc([gx], [MG_SEG_SAME], 7, 2, 3, 16, 20, 20)
    wd, bd = dev(w), dev(b)
    wpack = None
    nb = ffi.lib.mg_conv_packed_bytes(C.byref(d), 0) if impl == "auto" else 0
    if nb:
        wpack = torch.zeros(nb, dtype=torch.uint8, device="cuda")
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wpack), 0)
    gy = Grid(ctx.dtype, 2, 16, 10, 10)
    ctx.call("mg_conv_forward", C.byref(d), ptr(wd), ptr(wpack), ptr(bd), C.byref(gy.g()), None)
    assert max_rel(gy.nchw(), y_ref) <= TOL[ctx.dtype]
    g = rnd(2, 16, 10, 10)
    _, gw_ref, gb_ref = O.conv_backward(x, w, g, 2, 3)
    gg = Grid(ctx.dtype, 2, 16, 10, 10, g)
    dw, db = torch.zeros_like(wd), torch.zeros_like(bd)
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 1.0)
    torch.cuda.synchronize()
    assert max_rel(dw.cpu().numpy(), gw_ref) <= TOL[ctx.dtype]
    assert max_rel(db.cpu().numpy(), gb_ref) <= TOL[ctx.dtype]
    ctx.set_impl(ffi.MG_IMPL_AUTO)


@pytest.mark.parametrize("case", [(3, 3, 36, 44, 64), (2, 3, 70, 30, 32), (5, 1, 17, 9, 24), (2, 3, 224, 224, 64)],
                         ids=["cout64-tma-store", "cout32", "odd-cin1", "imagenet-size"])
@pytest.mark.parametrize("fused", [0, 1], ids=["stats-pass", "stats-fused"])
def test_stem_kernel_shapes(case, fused):
    """the dedicated 7x7 / stride-2 kernel (zero-copy im2col through UMMA descriptors over parity planes of the input patch):
    ragged tiles in both directions, the TMA-store epilogue (Cout = 64) and the direct-store one, fused BatchNorm sums"""
    N, Cin, H, W, Cout = case
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    ctx.set_tuning(ffi.MG_TUNE_STEM_FUSED_STATS, fused)
    x = rnd(N, Cin, H, W)
    w = bf16_round(rng.standard_normal((Cout, Cin, 7, 7)) * 0.1)
    b = bf16_round(rng.standard_normal(Cout) * 0.1)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    gx = Grid(ffi.MG_BF16, N, Cin, H, W, x)
    d = conv_desc([gx], [MG_SEG_SAME], 7, 2, 3, Cout, H, W)
    wd, bd = dev(w), dev(b)
    wp = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 0), dtype=torch.uint8, device="cuda")
    ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wp), 0)
    gy = Grid(ffi.MG_BF16, N, Cout, Ho, Wo)
    sums = new_sums(2 * Cout)
    tc0 = ctx.tc_launches()
    ctx.call("mg_conv_forward", C.byref(d), ptr(wd), ptr(wp), ptr(bd), C.byref(gy.g()), ptr(sums))
    assert ctx.tc_launches() - tc0 == 1, "the stem must run on its tensor-core kernel"
    torch.cuda.synchronize()
    xin = torch.from_numpy(bf16_round(x)).cuda().float()
    y_ref = torch.nn.functional.conv2d(xin.double(), torch.from_numpy(w).cuda().double(), torch.from_numpy(b).cuda().double(), 2, 3)
    yn = gy.t[..., :Cout].double().permute(0, 3, 1, 2)
    assert float((yn - y_ref).abs().max() / y_ref.abs().max()) <= TOL[ffi.MG_BF16]
    assert not gy.pad_channels().any()
    sv = sums_value(sums)
    assert torch.allclose(sv[:Cout], yn.sum((0, 2, 3)), rtol=1e-5, atol=1e-2)
    assert torch.allclose(sv[Cout:], (yn * yn).sum((0, 2, 3)), rtol=1e-5, atol=1e-2)
    if N * H * W < 20000:   # small cases also against the numpy oracle
        assert max_rel(gy.nchw(), O.conv_forward(bf16_round(x), w, b, 2, 3)) <= TOL[ffi.MG_BF16]
    # weight gradient on the dedicated kernel (the patch read in place as a Toeplitz operand): against an independent fp64
    # computation on the same bf16 inputs, accumulating twice (accGradParameters adds into gradWeight)
    g = rnd(N, Cout, Ho, Wo)
    gg = Grid(ffi.MG_BF16, N, Cout, Ho, Wo, g)
    dw, db = torch.zeros_like(wd), torch.zeros_like(bd)
    tc0 = ctx.tc_launches()
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 1.0)
    if Cout <= 64:
        assert ctx.tc_launches() - tc0 == 1, "the stem weight gradient must run on its tensor-core kernel"
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 0.5)
    torch.cuda.synchronize()
    gd = torch.from_numpy(bf16_round(g)).cuda().double()
    dw_ref = torch.nn.grad.conv2d_weight(xin.double(), w.shape, gd, stride=2, padding=3) * 1.5
    assert float((dw.double() - dw_ref).abs().max() / dw_ref.abs().max()) <= 1e-4, "fp32 accumulation of exact bf16 products"
    assert torch.allclose(db.double(), gd.sum((0, 2, 3)) * 1.5, rtol=1e-4, atol=1e-3)
    ctx.close()


@pytest.mark.parametrize("shape", [(2, 3, 20, 20, 16, 7, 2, 3), (3, 3, 15, 23, 40, 7, 2, 3), (2, 1, 9, 9, 8, 3, 2, 1)])
def test_stem_im2col_then_1x1_conv_equals_strided_conv(shape):
    """mg_im2col + a 1x1 mg_conv over the column tensor, with the [Cout][Cin][k][k] weight storage reinterpreted as
    [Cout][Cin*k*k][1][1], is the strided stem convolution (ilsvrc/rnmg.lua:180): columns bit-exact against a numpy
    gather, forward / gradWeight / gradBias against the oracle"""
    N, Cin, H, W, Cout, k, stride, pad = shape
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    x = bf16_round(rnd(N, Cin, H, W))
    w = bf16_round(rng.standard_normal((Cout, Cin, k, k)) * 0.1)
    b = bf16_round(rng.standard_normal(Cout) * 0.1)
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    gx = Grid(ffi.MG_BF16, N, Cin, H, W, x)
    K = Cin * k * k
    col = Grid(ffi.MG_BF16, N, K, Ho, Wo)
    col.t.fill_(7.0)                                   # every element, pad channels included, must be overwritten
    ctx.call("mg_im2col", C.byref(gx.g()), k, stride, pad, C.byref(col.g()))
    xp = np.pad(x, ((0, 0), (0, 0), (pad, pad), (pad, pad)))
    ref = np.zeros((N, K, Ho, Wo))
    for ci in range(Cin):
        for ky in range(k):
            for kx in range(k):
                ref[:, ci * k * k + ky * k + kx] = xp[:, ci, ky:ky + stride * Ho:stride, kx:kx + stride * Wo:stride]
    assert np.array_equal(col.nchw(), ref) and not col.pad_channels().any()
    d = conv_desc([col], [MG_SEG_SAME], 1, 1, 0, Cout, Ho, Wo)
    wd, bd = dev(w), dev(b)                            # same storage, read as [Cout][K][1][1]
    wp = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 0), dtype=torch.uint8, device="cuda")
    ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wp), 0)
    gy = Grid(ffi.MG_BF16, N, Cout, Ho, Wo)
    tc0 = ctx.tc_launches()
    ctx.call("mg_conv_forward", C.byref(d), ptr(wd), ptr(wp), ptr(bd), C.byref(gy.g()), None)
    tol = TOL[ffi.MG_BF16]
    assert max_rel(gy.nchw(), O.conv_forward(x, w, b, stride, pad)) <= tol
    g = rnd(N, Cout, Ho, Wo)
    _, gw_ref, gb_ref = O.conv_backward(x, w, g, stride, pad)
    gg = Grid(ffi.MG_BF16, N, Cout, Ho, Wo, g)
    dw, db = torch.zeros_like(wd), torch.zeros_like(bd)
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 1.0)
    assert ctx.tc_launches() - tc0 == 2
    torch.cuda.synchronize()
    assert max_rel(dw.cpu().numpy(), gw_ref) <= tol and max_rel(db.cpu().numpy(), gb_ref) <= tol
    ctx.close()


@pytest.mark.parametrize("shape", [(2, 12, 10, 5), (3, 64, 32, 8), (1, 40, 136, 3)])
def test_upconv2x2_forward_backward(ctx, shape):
    """cudnn.SpatialFullConvolution(nIP, nOP, 2,2,2,2) of U-MG (models/mnist-cluttered/unmg.lua:35-41); in bf16 mode it must run
    as one 1x1 tensor-core convolution to 4 * Cout channels + depth-to-space (upconv_tc.cu), not on the CUDA cores"""
    N, Cin, Cout, H = shape
    tc0 = ctx.tc_launches()
    x = rnd(N, Cin, H, H)
    w = bf16_round(rng.standard_normal((Cin, Cout, 2, 2)) * 0.3)
    b = bf16_round(rng.standard_normal(Cout) * 0.1)
    y_ref = O.upconv2x2_forward(x, w, b)
    gx, gy = Grid(ctx.dtype, N, Cin, H, H, x), Grid(ctx.dtype, N, Cout, 2 * H, 2 * H)
    wd, bd = dev(w), dev(b)
    sums = new_sums(2 * Cout)
    ctx.call("mg_upconv2x2_forward", C.byref(gx.g()), ptr(wd), ptr(bd), C.byref(gy.g()), ptr(sums))
    tol = TOL[ctx.dtype]
    assert max_rel(gy.nchw(), y_ref) <= tol
    assert np.allclose(sums_value(sums).cpu().numpy()[:Cout] / (N * 4 * H * H), y_ref.mean(axis=(0, 2, 3)), atol=tol * np.abs(y_ref).max())
    g = rnd(N, Cout, 2 * H, 2 * H)
    gx_ref, gw_ref, gb_ref = O.upconv2x2_backward(x, w, g)
    gg, dx = Grid(ctx.dtype, N, Cout, 2 * H, 2 * H, g), Grid(ctx.dtype, N, Cin, H, H)
    dw, db = torch.zeros_like(wd), torch.zeros_like(bd)
    ctx.call("mg_upconv2x2_backward", C.byref(gx.g()), ptr(wd), C.byref(gg.g()), C.byref(dx.g()), ptr(dw), ptr(db), 1.0)
    torch.cuda.synchronize()
    assert max_rel(dx.nchw(), gx_ref) <= tol
    assert max_rel(dw.cpu().numpy(), gw_ref) <= tol and max_rel(db.cpu().numpy(), gb_ref) <= tol
    assert not gy.pad_channels().any() and not dx.pad_channels().any()
    assert ctx.tc_launches() - tc0 == (3 if ctx.dtype == ffi.MG_BF16 else 0)     # forward, dgrad, wgrad
    # accGradParameters accumulates
    ctx.call("mg_upconv2x2_backward", C.byref(gx.g()), ptr(wd), C.byref(gg.g()), None, ptr(dw), ptr(db), 0.5)
    torch.cuda.synchronize()
    assert max_rel(dw.cpu().numpy(), 1.5 * gw_ref) <= tol and max_rel(db.cpu().numpy(), 1.5 * gb_ref) <= tol


def test_conv_shape_errors_are_reported_not_fatal(ctx):
    """JoinTable would raise on inconsistent sizes in the reference; here: status + message"""
    a, b = Grid(ctx.dtype, 1, 4, 8, 8), Grid(ctx.dtype, 1, 4, 5, 5)
    d = conv_desc([a, b], [MG_SEG_SAME, MG_SEG_UP], 3, 1, 1, 4, 8, 8)
    y = Grid(ctx.dtype, 1, 4, 8, 8)
    w = torch.zeros(4, 8, 3, 3, device="cuda")
    with pytest.raises(ffi.MGError, match="UP seg"):
        ctx.call("mg_conv_forward", C.byref(d), ptr(w), None, None, C.byref(y.g()), None)


def test_persistent_weight_resident_kernel_block1_shape():
    """R-MG-34 block-1 shapes (96 -> 64 at 56x56, enough slot tiles to take the persistent weight-resident kernel):
    forward, its fused BatchNorm sums and dgrad against the CUDA-core implementation of the same entry points"""
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    for (N, H, cs, Cout) in [(32, 56, (64, 32), 64), (112, 28, (64, 32, 16), 32)]:
        grids = [Grid(ffi.MG_BF16, N, cs[0], H, H)] + [Grid(ffi.MG_BF16, N, c, H, H) for c in cs[1:-1]] + [Grid(ffi.MG_BF16, N, cs[-1], H // 2, H // 2)]
        modes = [MG_SEG_SAME] * (len(cs) - 1) + [MG_SEG_UP]
        for g_ in grids:
            g_.t[..., :g_.C].normal_()
        d = conv_desc(grids, modes, 3, 1, 1, Cout, H, H)
        w = (torch.randn(Cout, sum(cs), 3, 3, device="cuda") * 0.05).to(torch.bfloat16).float()
        b = (torch.randn(Cout, device="cuda") * 0.1).to(torch.bfloat16).float()
        wp = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 0), dtype=torch.uint8, device="cuda")
        wpt = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 1), dtype=torch.uint8, device="cuda")
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(w), ptr(wp), 0)
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(w), ptr(wpt), 1)
        ys, dcs = [], []
        gg = Grid(ffi.MG_BF16, N, Cout, H, H)
        gg.t[..., :Cout].normal_()
        cp = sum(x.Cp for x in grids)
        for impl in (ffi.MG_IMPL_AUTO, ffi.MG_IMPL_SIMT):
            ctx.set_impl(impl)
            gy = Grid(ffi.MG_BF16, N, Cout, H, H)
            sums = new_sums(2 * Cout)
            tc0 = ctx.tc_launches()
            ctx.call("mg_conv_forward", C.byref(d), ptr(w), ptr(wp), ptr(b), C.byref(gy.g()), ptr(sums))
            dcat = Grid(ffi.MG_BF16, N, cp, H, H, Cp=cp)
            ctx.call("mg_conv_backward_data", C.byref(d), ptr(w), ptr(wpt), C.byref(gg.g()), C.byref(dcat.g()))
            assert ctx.tc_launches() - tc0 == (2 if impl == ffi.MG_IMPL_AUTO else 0)
            torch.cuda.synchronize()
            ys.append(gy.t.float()); dcs.append(dcat.t.float())
            if impl == ffi.MG_IMPL_AUTO:   # the sums are those of the stored bf16 values
                yf = gy.t.double().reshape(-1, gy.Cp)[:, :Cout]
                assert torch.allclose(sums_value(sums)[:Cout], yf.sum(0), rtol=1e-5, atol=1e-2)
                assert torch.allclose(sums_value(sums)[Cout:], (yf * yf).sum(0), rtol=1e-5, atol=1e-2)
        tol = TOL[ffi.MG_BF16]
        assert float((ys[0] - ys[1]).abs().max() / ys[1].abs().max()) <= tol
        assert float((dcs[0] - dcs[1]).abs().max() / dcs[1].abs().max()) <= tol
    ctx.close()


def test_every_kernel_variant_computes_the_same_bits():
    """The variant of a 3x3 layer is chosen by timing (Engine autotune), so the choice must not change a bit: forward output, its
    fused BatchNorm sums and dgrad of every MG_ALGO_* equal the heuristic's.  At 56x56 and 28x28 the persistent CTA-pair kernel
    would use row-aligned tiles (R * (W + 1) slots), which group the slots of the fp32 partial sums differently"""
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    for (N, H, cs, Cout) in [(32, 56, (64, 32), 64), (112, 28, (64, 32, 16), 32)]:
        grids = [Grid(ffi.MG_BF16, N, cs[0], H, H)] + [Grid(ffi.MG_BF16, N, c, H, H) for c in cs[1:-1]] + [Grid(ffi.MG_BF16, N, cs[-1], H // 2, H // 2)]
        modes = [MG_SEG_SAME] * (len(cs) - 1) + [MG_SEG_UP]
        for g_ in grids:
            g_.t[..., :g_.C].normal_()
        d = conv_desc(grids, modes, 3, 1, 1, Cout, H, H)
        w = (torch.randn(Cout, sum(cs), 3, 3, device="cuda") * 0.05).to(torch.bfloat16).float()
        b = (torch.randn(Cout, device="cuda") * 0.1).to(torch.bfloat16).float()
        wp = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 0), dtype=torch.uint8, device="cuda")
        wpt = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 1), dtype=torch.uint8, device="cuda")
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(w), ptr(wp), 0)
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(w), ptr(wpt), 1)
        gg = Grid(ffi.MG_BF16, N, Cout, H, H)
        gg.t[..., :Cout].normal_()
        cp = sum(x.Cp for x in grids)
        ref = None
        for algo in range(ffi.MG_ALGO_RESIDENT_PAIR + 1):
            d.algo_fwd = d.algo_bwd_data = algo
            gy, sums, dcat = Grid(ffi.MG_BF16, N, Cout, H, H), new_sums(2 * Cout), Grid(ffi.MG_BF16, N, cp, H, H, Cp=cp)
            ctx.call("mg_conv_forward", C.byref(d), ptr(w), ptr(wp), ptr(b), C.byref(gy.g()), ptr(sums))
            ctx.call("mg_conv_backward_data", C.byref(d), ptr(w), ptr(wpt), C.byref(gg.g()), C.byref(dcat.g()))
            torch.cuda.synchronize()
            got = (gy.t, sums, dcat.t)
            ref = ref or got
            for name, a, r in zip(("output", "BatchNorm sums", "dgrad"), got, ref):
                assert torch.equal(a, r), (H, algo, name)
    ctx.close()


FULL_SHAPES = [  # R-MG-34 layers at the BASELINE batch (256 per GPU): (H, [(C, mode)], Cout)
    (56, [(64, "s"), (32, "u")], 64),                # block 1, finest grid (rnmg.lua:250)
    (28, [(128, "s"), (64, "s"), (32, "u")], 64),    # block 2, middle grid: pooled finer | same | up-sampled coarser
    (14, [(256, "s"), (128, "u")], 256),             # block 3, finest grid
    (7, [(512, "s")], 512),                          # block 4
]


@pytest.mark.parametrize("shape", FULL_SHAPES, ids=["b1g1", "b2g2", "b3g1", "b4"])
def test_full_size_conv_is_linear_and_its_gradients_are_its_adjoints(shape):
    """BASELINE-size layers (B = 256), where the oracle is too slow: size-independent properties of the three tensor-core
    passes.  <g, conv(x; w)> = <dgrad(g), cat(x)> = <wgrad(g), w> (the backward passes are the adjoints of the forward one in
    x and in w), conv(2x) = 2 conv(x) exactly (powers of two commute with bf16 rounding), the fused BatchNorm sums equal the
    sums of the stored output, and pad channels stay zero."""
    H, segs, Cout = shape
    N = 256
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    torch.manual_seed(11)
    grids, modes, parts = [], [], []
    for c, m in segs:
        h = H // 2 if m == "u" else H
        g_ = Grid(ffi.MG_BF16, N, c, h, h)
        g_.t[..., :c].normal_()
        grids.append(g_); modes.append(MG_SEG_UP if m == "u" else MG_SEG_SAME)
        x = g_.t[..., :c].float()
        parts.append(x.repeat_interleave(2, dim=1).repeat_interleave(2, dim=2) if m == "u" else x)
    cin = sum(c for c, _ in segs)
    d = conv_desc(grids, modes, 3, 1, 1, Cout, H, H)
    w = (torch.randn(Cout, cin, 3, 3, device="cuda") * 0.05).to(torch.bfloat16).float()
    zero_b = torch.zeros(Cout, device="cuda")
    wp = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 0), dtype=torch.uint8, device="cuda")
    wpt = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 1), dtype=torch.uint8, device="cuda")
    ctx.call("mg_conv_pack_weights", C.byref(d), ptr(w), ptr(wp), 0)
    ctx.call("mg_conv_pack_weights", C.byref(d), ptr(w), ptr(wpt), 1)
    y = Grid(ffi.MG_BF16, N, Cout, H, H)
    sums = new_sums(2 * Cout)
    ctx.call("mg_conv_forward", C.byref(d), ptr(w), ptr(wp), ptr(zero_b), C.byref(y.g()), ptr(sums))
    yf = y.t[..., :Cout].double()
    assert torch.allclose(sums_value(sums)[:Cout], yf.sum((0, 1, 2)), rtol=1e-5, atol=1e-1)
    assert torch.allclose(sums_value(sums)[Cout:], (yf * yf).sum((0, 1, 2)), rtol=1e-5, atol=1e-1)
    assert not y.t[..., Cout:].any()
    # linearity: doubling the input doubles every stored output bit for bit
    for g_ in grids:
        g_.t.mul_(2)
    y2 = Grid(ffi.MG_BF16, N, Cout, H, H)
    ctx.call("mg_conv_forward", C.byref(d), ptr(w), ptr(wp), ptr(zero_b), C.byref(y2.g()), None)
    assert torch.equal(y2.t, y.t * 2)
    for g_ in grids:
        g_.t.mul_(0.5)
    # adjoints
    gg = Grid(ffi.MG_BF16, N, Cout, H, H)
    gg.t[..., :Cout].normal_()
    cp = sum(x.Cp for x in grids)
    dcat = Grid(ffi.MG_BF16, N, cp, H, H, Cp=cp)
    ctx.call("mg_conv_backward_data", C.byref(d), ptr(w), ptr(wpt), C.byref(gg.g()), C.byref(dcat.g()))
    dw = torch.zeros_like(w)
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), None, 1.0)
    torch.cuda.synchronize()
    lhs = float((gg.t[..., :Cout].double() * yf).sum())
    off, mid = 0, 0.0
    for g_, part in zip(grids, parts):
        mid += float((dcat.t[..., off:off + g_.C].double() * part.double()).sum())
        assert not dcat.t[..., off + g_.C:off + g_.Cp].any()
        off += g_.Cp
    rhs = float((dw.double() * w.double()).sum())
    scale = float(gg.t[..., :Cout].double().norm() * yf.norm())     # Cauchy-Schwarz bound of the inner products
    assert abs(lhs - mid) <= 2e-3 * scale and abs(lhs - rhs) <= 2e-3 * scale, (lhs, mid, rhs, scale)
    # VALUES at the full batch against an independent fp32 computation of the same layer (PyTorch / cuDNN, TF32 off) on the
    # same bf16-representable operands: forward, dgrad and wgrad of all 256 images ...
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        xin = torch.cat(parts, dim=3).permute(0, 3, 1, 2).contiguous()          # gathered input, NCHW fp32
        gn = gg.t[..., :Cout].float().permute(0, 3, 1, 2).contiguous()
        y_ref = torch.nn.functional.conv2d(xin, w, None, 1, 1)
        dx_ref = torch.nn.grad.conv2d_input(xin.shape, w, gn, stride=1, padding=1)
        dw_ref = torch.nn.grad.conv2d_weight(xin, w.shape, gn, stride=1, padding=1)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    tol = TOL[ffi.MG_BF16]
    yn = y.t[..., :Cout].float().permute(0, 3, 1, 2)
    assert float((yn - y_ref).abs().max() / y_ref.abs().max()) <= tol
    assert float((yn - y_ref).norm() / y_ref.norm()) <= 4e-3          # bf16 rounding of the stored output: 2^-9 per element
    off = lo = 0
    for g_ in grids:
        dseg = dcat.t[..., off:off + g_.C].float().permute(0, 3, 1, 2)
        ref = dx_ref[:, lo:lo + g_.C]
        assert float((dseg - ref).abs().max() / dx_ref.abs().max()) <= tol
        assert float((dseg - ref).norm() / ref.norm()) <= 4e-3
        off += g_.Cp; lo += g_.C
    assert float((dw - dw_ref).abs().max() / dw_ref.abs().max()) <= tol
    assert float((dw - dw_ref).norm() / dw_ref.norm()) <= 1e-3        # fp32 accumulation over 256 images, fp32 result
    # ... and the first and last image of the batch against the numpy fp64 oracle (the check that anchors the comparison above)
    sel = [0, N - 1]
    xs_np = xin[sel].double().cpu().numpy()
    yo = O.conv_forward(xs_np, w.double().cpu().numpy(), np.zeros(Cout), 1, 1)
    assert max_rel(yn[sel].double().cpu().numpy(), yo) <= tol
    assert max_rel(y_ref[sel].double().cpu().numpy(), yo) <= 1e-4          # fp32 accumulation over K up to 4 608
    ctx.close()


# ---------------------------------------------------------------- BatchNorm + epilogue
@pytest.mark.parametrize("eps", [1e-5, 1e-3])
def test_bn_finalize_apply_residual_and_backward(ctx, eps):
    N, Cc, H = 3, 12, 6
    x = bf16_round(rnd(N, Cc, H, H) * 2 + 1)
    gamma, beta = rng.random(Cc) + 0.5, rng.standard_normal(Cc) * 0.1
    rm, rv = np.zeros(Cc), np.ones(Cc)
    drm, drv = dev(rm), dev(rv)   # device copies of the initial running stats (the oracle updates rm/rv in place)
    y_ref, mean, invstd = O.bn_forward_train(x, gamma, beta, eps, rm, rv)
    sc = rnd(N, 8, H, H)  # zero-padded shortcut with fewer channels (nn.Padding, ilsvrc/rnmg.lua:16)
    out_ref = O.relu_forward(y_ref + O.pad_channels(sc, Cc))
    gx = Grid(ctx.dtype, N, Cc, H, H, x)
    sums = new_sums(2 * Cc)
    ctx.call("mg_bn_stats", C.byref(gx.g()), ptr(sums))
    scale, shift = torch.zeros(gx.Cp, device="cuda"), torch.zeros(gx.Cp, device="cuda")
    smean, sinv = torch.zeros(gx.Cp, device="cuda"), torch.zeros(gx.Cp, device="cuda")
    dgam, dbet = dev(gamma), dev(beta)
    ctx.call("mg_bn_finalize", ptr(sums), N * H * H, Cc, gx.Cp, ptr(dgam), ptr(dbet), ptr(drm), ptr(drv), eps, 0.1, 1,
             ptr(scale), ptr(shift), ptr(smean), ptr(sinv))
    torch.cuda.synchronize()
    assert np.allclose(drm.cpu().numpy(), rm, atol=1e-5) and np.allclose(drv.cpu().numpy(), rv, rtol=1e-4)  # unbiased running var
    gx.scale, gx.shift = scale, shift
    gsc, gout = Grid(ctx.dtype, N, 8, H, H, sc), Grid(ctx.dtype, N, Cc, H, H)
    gpool = Grid(ctx.dtype, N, Cc, H // 2, H // 2)
    ctx.call("mg_residual_forward", C.byref(gx.g()), C.byref(gsc.g()), 1, C.byref(gout.g()), C.byref(gpool.g()))
    tol = TOL[ctx.dtype]
    out = gout.nchw()
    assert max_rel(out, out_ref) <= tol
    # the pooled companion is exactly the 2x2 max of what was stored
    assert np.array_equal(gpool.nchw(), O.maxpool_forward(out)[0])

    # backward: mask by the stored output, reduce (sum d, sum d*x), BN backward
    go = rnd(N, Cc, H, H)
    d_ref = O.relu_backward(out, go)
    gxr, dg_ref, db_ref = O.bn_backward_train(x, d_ref, gamma, mean, invstd)
    ggo, gd, gres = Grid(ctx.dtype, N, Cc, H, H, go), Grid(ctx.dtype, N, Cc, H, H), Grid(ctx.dtype, N, Cc, H, H)
    src = (mg_grad_src * 1)()
    src[0].g, src[0].c_offset, src[0].mode = ggo.g(), 0, MG_SEG_SAME
    dsums = new_sums(2 * Cc)
    xraw = Grid(ctx.dtype, N, Cc, H, H, x)
    ctx.call("mg_grad_combine", C.byref(gout.g()), 1, C.byref(xraw.g()), 1, src, C.byref(gd.g()), ptr(dsums))
    assert np.array_equal(gd.nchw(), bf16_round(d_ref) if ctx.dtype == ffi.MG_BF16 else d_ref)
    dgamma, dbeta = torch.zeros(Cc, device="cuda"), torch.zeros(Cc, device="cuda")
    coef = torch.zeros(3 * gx.Cp, device="cuda")
    conv_db = torch.zeros(Cc, device="cuda")
    ctx.call("mg_bn_backward", C.byref(xraw.g()), C.byref(gd.g()), C.byref(gres.g()), ptr(dsums), N * H * H, ptr(dgam),
             ptr(smean), ptr(sinv), ptr(dgamma), ptr(dbeta), 1.0, ptr(coef), ptr(conv_db))
    torch.cuda.synchronize()
    assert max_rel(gres.nchw(), gxr) <= tol
    # gradBias of the producing convolution = sum over pixels of the BN-backward output = A*sum(d) + B*sum(x) + C*n, evaluated in
    # fp64 from the sums: identically zero in exact arithmetic (as the oracle's fp64 sum is), no reduction, no atomics
    assert np.abs(gxr.sum(axis=(0, 2, 3))).max() <= 1e-9 * np.abs(gxr).sum()
    assert np.abs(conv_db.cpu().numpy()).max() <= 1e-5 * np.abs(gxr).sum(axis=(0, 2, 3)).max() + 1e-5 * np.abs(gxr).max()
    assert max_rel(dgamma.cpu().numpy(), dg_ref) <= tol and max_rel(dbeta.cpu().numpy(), db_ref) <= tol
    # evaluation mode uses the running statistics
    ctx.call("mg_bn_finalize", None, N * H * H, Cc, gx.Cp, ptr(dgam), ptr(dbet), ptr(drm), ptr(drv), eps, 0.1, 0,
             ptr(scale), ptr(shift), None, None)
    ctx.call("mg_residual_forward", C.byref(gx.g()), None, 0, C.byref(gout.g()), None)
    assert max_rel(gout.nchw(), O.bn_forward_eval(x, gamma, beta, rm, rv, eps)) <= tol


@pytest.mark.parametrize("training", [1, 0])
def test_bn_residual_forward_one_pass_equals_finalize_plus_residual(ctx, training):
    """mg_bn_residual_forward (finalisation fused into the apply pass) == mg_bn_finalize + mg_residual_forward:
    affine, saved statistics and running statistics to fp32 rounding (the two kernels contract their fp64
    expressions differently), outputs to one bf16 ulp, pooled companion == 2x2 max of what was stored"""
    N, Cc, H = 4, 20, 9     # Cp = 24 (pad channels), odd size (ceil-mode companion)
    x = bf16_round(rnd(N, Cc, H, H) * 1.5 - 0.3)
    gamma, beta = dev(rng.random(Cc) + 0.5), dev(rng.standard_normal(Cc) * 0.1)
    sc = rnd(N, 8, H, H)
    res = {}
    for mode in ("split", "fused"):
        rm, rv = dev(rng.standard_normal(Cc) * 0 + 0.25), dev(np.full(Cc, 1.5))
        gx = Grid(ctx.dtype, N, Cc, H, H, x)
        sums = new_sums(2 * Cc)
        ctx.call("mg_bn_stats", C.byref(gx.g()), ptr(sums))
        gx.scale, gx.shift = torch.zeros(gx.Cp, device="cuda"), torch.zeros(gx.Cp, device="cuda")
        smean, sinv = torch.zeros(gx.Cp, device="cuda"), torch.zeros(gx.Cp, device="cuda")
        gsc, gout, gpool = Grid(ctx.dtype, N, 8, H, H, sc), Grid(ctx.dtype, N, Cc, H, H), Grid(ctx.dtype, N, Cc, (H + 1) // 2, (H + 1) // 2)
        if mode == "split":
            ctx.call("mg_bn_finalize", ptr(sums), N * H * H, Cc, gx.Cp, ptr(gamma), ptr(beta), ptr(rm), ptr(rv), 1e-5, 0.1, training,
                     ptr(gx.scale), ptr(gx.shift), ptr(smean), ptr(sinv))
            ctx.call("mg_residual_forward", C.byref(gx.g()), C.byref(gsc.g()), 1, C.byref(gout.g()), C.byref(gpool.g()))
        else:
            f = ffi.mg_bn_fused()
            f.sums, f.count, f.gamma, f.beta = sums.data_ptr(), N * H * H, gamma.data_ptr(), beta.data_ptr()
            f.running_mean, f.running_var, f.eps, f.momentum, f.training = rm.data_ptr(), rv.data_ptr(), 1e-5, 0.1, training
            f.save_mean, f.save_invstd = smean.data_ptr(), sinv.data_ptr()
            ctx.call("mg_bn_residual_forward", C.byref(gx.g()), C.byref(f), C.byref(gsc.g()), 1, C.byref(gout.g()), C.byref(gpool.g()))
        torch.cuda.synchronize()
        res[mode] = [gout.nchw(), gpool.nchw(), gout.pad_channels()] + [t.cpu().numpy() for t in (gx.scale, gx.shift, smean, sinv, rm, rv)]
    for a, b in zip(res["split"][3:], res["fused"][3:]):
        assert np.allclose(a, b, rtol=1e-6, atol=1e-7)
    for a, b in zip(res["split"][:2], res["fused"][:2]):
        assert np.allclose(a, b, rtol=2.0 ** -7, atol=1e-6)
    assert not res["fused"][2].any()
    assert np.array_equal(res["fused"][1], O.maxpool_forward(res["fused"][0])[0])


def test_pack_weights_batched_equals_per_conv_packing():
    """one launch over a table of (conv, direction) jobs writes the same operand images as mg_conv_pack_weights"""
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    shapes = [(2, [(24, "s"), (8, "u")], 8, 8, 40, 3), (1, [(16, "s")], 5, 70, 8, 3), (2, [(72, "s"), (40, "s")], 4, 4, 24, 1),
              (1, [(200, "s")], 7, 7, 300, 3)]
    jobs, keep = [], []
    for N, segs, H, W, Cout, k in shapes:
        grids = [Grid(ffi.MG_BF16, N, c, H // 2 if m == "u" else H, W // 2 if m == "u" else W) for c, m in segs]
        modes = [MG_SEG_UP if m == "u" else MG_SEG_SAME for _, m in segs]
        d = conv_desc(grids, modes, k, 1, 0 if k == 1 else 1, Cout, H, W)
        w = dev(rng.standard_normal((Cout, sum(c for c, _ in segs), k, k)))
        keep.append((grids, d, w))
        for tr in (0, 1):
            nb = ffi.lib.mg_conv_packed_bytes(C.byref(d), tr)
            one = torch.full((nb,), 0xAB, dtype=torch.uint8, device="cuda")
            many = torch.full((nb,), 0xCD, dtype=torch.uint8, device="cuda")
            ctx.call("mg_conv_pack_weights", C.byref(d), ptr(w), ptr(one), tr)
            jobs.append((d, w, one, many, tr))
    n = len(jobs)
    descs = (C.POINTER(ffi.mg_conv_desc) * n)(*[C.pointer(j[0]) for j in jobs])
    ws = (C.c_void_p * n)(*[j[1].data_ptr() for j in jobs])
    outs = (C.c_void_p * n)(*[j[3].data_ptr() for j in jobs])
    tr = (C.c_int32 * n)(*[j[4] for j in jobs])
    l0 = ctx.launches()
    for _ in range(2):   # the second call reuses the uploaded job table
        ctx.call("mg_conv_pack_weights_batched", n, descs, ws, outs, tr)
    assert ctx.launches() - l0 == 2
    torch.cuda.synchronize()
    for j in jobs:
        assert torch.equal(j[2], j[3])
    ctx.close()


# ---------------------------------------------------------------- committed golden vectors (tests/golden/)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("name", ["mgconv_3scale_k3.npz", "mgconv_3scale_k1.npz"])
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_golden_mgconv(ctx, name, impl):
    """multigrid convolution against the committed oracle vectors: forward, the gradient w.r.t. the concatenated input
    routed back to the three grids (pool arg-max, identity, 2x2 block sum through mg_grad_combine), dW, dbias"""
    if impl == "auto" and ctx.dtype != ffi.MG_BF16:
        pytest.skip("tcgen05 path is bf16 only")
    G = {k: v for k, v in np.load(os.path.join(GOLDEN, name)).items()}
    f, s, c, w, b, g = (G[k].astype(np.float64) for k in ("finer", "same", "coarser", "weight", "bias", "grad_out"))
    k = int(G["k"]); pad = 0 if k == 1 else 1
    N, H, Cout = s.shape[0], s.shape[2], w.shape[0]
    cs = (f.shape[1], s.shape[1], c.shape[1])
    # arg-max of the pooling is bit-exact (indices are the only integer data of the path)
    gf_, gs_, gc_ = Grid(ctx.dtype, N, cs[0], 2 * H, 2 * H, f), Grid(ctx.dtype, N, cs[1], H, H, s), Grid(ctx.dtype, N, cs[2], H // 2, H // 2, c)
    gp = Grid(ctx.dtype, N, cs[0], H, H)
    arg = torch.zeros((N, H, H, cs[0]), dtype=torch.int32, device="cuda")
    ctx.call("mg_pool_forward", C.byref(gf_.g()), C.byref(gp.g()), 0, ptr(arg))
    torch.cuda.synchronize()
    assert np.array_equal(arg.permute(0, 3, 1, 2).cpu().numpy(), G["pool_argmax"])
    ctx.set_impl(ffi.MG_IMPL_SIMT if impl == "simt" else ffi.MG_IMPL_AUTO)
    d = conv_desc([gp, gs_, gc_], [MG_SEG_SAME, MG_SEG_SAME, MG_SEG_UP], k, 1, pad, Cout, H, H)
    wd, bd = dev(w), dev(b)
    wp = wpt = None
    if impl == "auto":
        wp = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 0), dtype=torch.uint8, device="cuda")
        wpt = torch.zeros(ffi.lib.mg_conv_packed_bytes(C.byref(d), 1), dtype=torch.uint8, device="cuda")
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wp), 0)
        ctx.call("mg_conv_pack_weights", C.byref(d), ptr(wd), ptr(wpt), 1)
    gy = Grid(ctx.dtype, N, Cout, H, H)
    ctx.call("mg_conv_forward", C.byref(d), ptr(wd), ptr(wp), ptr(bd), C.byref(gy.g()), None)
    tol = TOL[ctx.dtype]
    assert max_rel(gy.nchw(), G["y"]) <= tol
    gg = Grid(ctx.dtype, N, Cout, H, H, g)
    cps = [gp.Cp, gs_.Cp, gc_.Cp]
    dcat = Grid(ctx.dtype, N, sum(cps), H, H, Cp=sum(cps))
    ctx.call("mg_conv_backward_data", C.byref(d), ptr(wd), ptr(wpt), C.byref(gg.g()), C.byref(dcat.g()))
    dw, db = torch.zeros_like(wd), torch.zeros_like(bd)
    ctx.call("mg_conv_backward_weight", C.byref(d), C.byref(gg.g()), ptr(dw), ptr(db), 1.0)
    torch.cuda.synchronize()
    assert max_rel(dw.cpu().numpy(), G["grad_weight"]) <= tol and max_rel(db.cpu().numpy(), G["grad_bias"]) <= tol
    # route dcat back to the three grids the way a plan does (gather form)
    offs = [0, cps[0], cps[0] + cps[1]]
    for grid, off, mode, key in ((gf_, offs[0], MG_SEG_POOL, "grad_finer"), (gs_, offs[1], MG_SEG_SAME, "grad_same"), (gc_, offs[2], MG_SEG_UP, "grad_coarser")):
        src = (mg_grad_src * 1)()
        src[0].g, src[0].c_offset, src[0].mode = dcat.g(), off, mode
        out = Grid(ctx.dtype, grid.N, grid.C, grid.H, grid.W)
        ctx.call("mg_grad_combine", C.byref(grid.g()), 0, None, 1, src, C.byref(out.g()), None)
        assert max_rel(out.nchw(), G[key]) <= tol, key
    ctx.set_impl(ffi.MG_IMPL_AUTO)


@pytest.mark.parametrize("name", ["bn_shortcut_relu.npz", "bn_shortcut_relu_odd.npz"])
def test_golden_bn_shortcut_relu(ctx, name):
    """SpatialBatchNormalization (train) + zero-padded shortcut + ReLU + pooled companion and their backward against the
    committed oracle vectors, through the one-pass entry points"""
    G = {k: v for k, v in np.load(os.path.join(GOLDEN, name)).items()}
    x, sc, go = (G[k].astype(np.float64) for k in ("x", "shortcut", "grad_out"))
    N, Cc, H = x.shape[0], x.shape[1], x.shape[2]
    Cs, eps = sc.shape[1], float(G["eps"])
    gx = Grid(ctx.dtype, N, Cc, H, H, x)
    sums = new_sums(2 * Cc)
    ctx.call("mg_bn_stats", C.byref(gx.g()), ptr(sums))
    gx.scale, gx.shift = torch.zeros(gx.Cp, device="cuda"), torch.zeros(gx.Cp, device="cuda")
    smean, sinv = torch.zeros(gx.Cp, device="cuda"), torch.zeros(gx.Cp, device="cuda")
    gam, bet, rm, rv = dev(G["gamma"]), dev(G["beta"]), dev(np.zeros(Cc)), dev(np.ones(Cc))
    f = ffi.mg_bn_fused()
    f.sums, f.count, f.gamma, f.beta = sums.data_ptr(), N * H * H, gam.data_ptr(), bet.data_ptr()
    f.running_mean, f.running_var, f.eps, f.momentum, f.training = rm.data_ptr(), rv.data_ptr(), eps, 0.1, 1
    f.save_mean, f.save_invstd = smean.data_ptr(), sinv.data_ptr()
    gsc, gout, gpool = Grid(ctx.dtype, N, Cs, H, H, sc), Grid(ctx.dtype, N, Cc, H, H), Grid(ctx.dtype, N, Cc, (H + 1) // 2, (H + 1) // 2)
    ctx.call("mg_bn_residual_forward", C.byref(gx.g()), C.byref(f), C.byref(gsc.g()), 1, C.byref(gout.g()), C.byref(gpool.g()))
    tol = TOL[ctx.dtype]
    out = gout.nchw()
    assert max_rel(out, G["out"]) <= tol and max_rel(gpool.nchw(), G["pooled"]) <= tol
    assert np.allclose(rm.cpu().numpy(), G["running_mean"], atol=1e-5) and np.allclose(rv.cpu().numpy(), G["running_var"], rtol=1e-4)
    assert np.allclose(smean.cpu().numpy()[:Cc], G["save_mean"], atol=1e-5) and np.allclose(sinv.cpu().numpy()[:Cc], G["save_invstd"], rtol=1e-4)
    ggo, gd, gres = Grid(ctx.dtype, N, Cc, H, H, go), Grid(ctx.dtype, N, Cc, H, H), Grid(ctx.dtype, N, Cc, H, H)
    src = (mg_grad_src * 1)()
    src[0].g, src[0].c_offset, src[0].mode = ggo.g(), 0, MG_SEG_SAME
    dsums = new_sums(2 * Cc)
    ctx.call("mg_grad_combine", C.byref(gout.g()), 1, C.byref(gx.g()), 1, src, C.byref(gd.g()), ptr(dsums))
    assert max_rel(gd.nchw()[:, :Cs], G["grad_shortcut"]) <= tol
    dgamma, dbeta, coef = torch.zeros(Cc, device="cuda"), torch.zeros(Cc, device="cuda"), torch.zeros(3 * gx.Cp, device="cuda")
    xraw = Grid(ctx.dtype, N, Cc, H, H, x)
    ctx.call("mg_bn_backward", C.byref(xraw.g()), C.byref(gd.g()), C.byref(gres.g()), ptr(dsums), N * H * H, ptr(gam), ptr(smean), ptr(sinv),
             ptr(dgamma), ptr(dbeta), 1.0, ptr(coef), None)
    torch.cuda.synchronize()
    assert max_rel(gres.nchw(), G["grad_x"]) <= tol
    assert max_rel(dgamma.cpu().numpy(), G["grad_gamma"]) <= tol and max_rel(dbeta.cpu().numpy(), G["grad_beta"]) <= tol


# ---------------------------------------------------------------- gradient routing (bit-exact paths)
@pytest.mark.parametrize("H", [8, 7])
def test_grad_combine_routes_through_argmax_and_upsample(ctx, H):
    """ConcatTable backward-sum of ResampleConcat (ilsvrc/rnmg.lua:53-82): tensor x receives its
    gradient as the same-scale source of grid i, through the 2x2 arg-max as the pooled source of
    grid i+1 and as a 2x2 block sum as the up-sampled source of grid i-1."""
    N, Cc = 2, 6
    Hc = (H + 1) // 2
    x = rnd(N, Cc, H, H)
    x[0, 0, :2, :2] = 0.75  # tie inside a pooling window: only the first max receives gradient
    g_same = rnd(N, Cc + 4, H, H)          # dcat of conv i: channels [4, 4+Cc)
    g_pool = rnd(N, Cc, Hc, Hc)            # dcat slice of conv i+1 (coarser)
    g_up = rnd(N, Cc + 2, 2 * H, 2 * H)    # dcat of conv i-1 (finer): channels [2, 2+Cc)
    _, idx = O.maxpool_forward(x)
    ref = g_same[:, 4:4 + Cc] + O.maxpool_backward(g_pool, idx, x.shape) + O.upsample_backward(g_up[:, 2:2 + Cc])
    gx = Grid(ctx.dtype, N, Cc, H, H, x)
    a, b, c = Grid(ctx.dtype, N, Cc + 4, H, H, g_same), Grid(ctx.dtype, N, Cc, Hc, Hc, g_pool), Grid(ctx.dtype, N, Cc + 2, 2 * H, 2 * H, g_up)
    src = (mg_grad_src * 3)()
    for i, (gr, off, mode) in enumerate([(a, 4, MG_SEG_SAME), (b, 0, MG_SEG_POOL), (c, 2, MG_SEG_UP)]):
        src[i].g, src[i].c_offset, src[i].mode = gr.g(), off, mode
    gd = Grid(ctx.dtype, N, Cc, H, H)
    ctx.call("mg_grad_combine", C.byref(gx.g()), 0, None, 3, src, C.byref(gd.g()), None)
    got = gd.nchw()
    assert max_rel(got, ref) <= TOL[ctx.dtype]
    # routing itself is exact: zero / non-zero pattern of the pooled contribution alone
    src1 = (mg_grad_src * 1)()
    src1[0].g, src1[0].c_offset, src1[0].mode = b.g(), 0, MG_SEG_POOL
    ctx.call("mg_grad_combine", C.byref(gx.g()), 0, None, 1, src1, C.byref(gd.g()), None)
    assert np.array_equal(gd.nchw(), O.maxpool_backward(g_pool, idx, x.shape))


def test_grad_combine_stem_pool3(ctx):
    x = rnd(2, 5, 12, 12)
    y, idx = O.maxpool_forward(x, 3, 2, 1, ceil_mode=False)
    g = rnd(*y.shape)
    gx, gg, gd = Grid(ctx.dtype, 2, 5, 12, 12, x), Grid(ctx.dtype, 2, 5, 6, 6, g), Grid(ctx.dtype, 2, 5, 12, 12)
    src = (mg_grad_src * 1)()
    src[0].g, src[0].c_offset, src[0].mode = gg.g(), 0, MG_SRC_POOL3
    ctx.call("mg_grad_combine", C.byref(gx.g()), 0, None, 1, src, C.byref(gd.g()), None)   # arg-max recomputed from x
    assert max_rel(gd.nchw(), O.maxpool_backward(g, idx, x.shape)) <= TOL[ctx.dtype]
    if ctx.dtype == ffi.MG_BF16:  # routed through the arg-max codes written by the forward pass
        gp = Grid(ctx.dtype, 2, 5, 6, 6)
        code = torch.zeros((2, 6, 6, gp.Cp), dtype=torch.uint8, device="cuda")
        ctx.call("mg_pool3s2_forward", C.byref(gx.g()), C.byref(gp.g()), ptr(code))
        src[0].aux = code.data_ptr()
        gd2 = Grid(ctx.dtype, 2, 5, 12, 12)
        ctx.call("mg_grad_combine", C.byref(gx.g()), 0, None, 1, src, C.byref(gd2.g()), None)
        assert max_rel(gd2.nchw(), O.maxpool_backward(g, idx, x.shape)) <= TOL[ctx.dtype]  # overlapping windows: sums round


def test_stem_bn_relu_pool3_fused_equals_two_passes():
    """mg_bn_relu_pool3_forward (BN + ReLU + SpatialMaxPooling(3,3,2,2,1,1) in one pass, ilsvrc/rnmg.lua:181-183; the activation is
    never stored) == mg_bn_residual_forward + mg_pool3s2_forward bit for bit (pooled values, arg-max codes, BatchNorm state), and
    mg_grad_combine with relu_mask = 2 (mask = sign of the pooled value at the arg-max) == the masked routing through the stored
    activation, bit for bit, including the BatchNorm backward sums"""
    ctx = ffi.Context(0, torch.cuda.current_stream().cuda_stream, ffi.MG_BF16)
    for (N, Cc, H, W) in [(2, 20, 13, 12), (3, 64, 16, 16), (1, 5, 7, 9)]:
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        y = bf16_round(rnd(N, Cc, H, W) * 1.5 - 0.2)
        gamma, beta = dev(rng.random(Cc) + 0.5), dev(rng.standard_normal(Cc) * 0.3)
        g = rnd(N, Cc, Ho, Wo)
        res = {}
        for mode in ("two", "fused"):
            rm, rv = dev(np.full(Cc, 0.25)), dev(np.full(Cc, 1.5))
            gy = Grid(ffi.MG_BF16, N, Cc, H, W, y)
            sums = new_sums(2 * Cc)
            ctx.call("mg_bn_stats", C.byref(gy.g()), ptr(sums))
            gy.scale, gy.shift = torch.zeros(gy.Cp, device="cuda"), torch.zeros(gy.Cp, device="cuda")
            smean, sinv = torch.zeros(gy.Cp, device="cuda"), torch.zeros(gy.Cp, device="cuda")
            f = ffi.mg_bn_fused()
            f.sums, f.count, f.gamma, f.beta = sums.data_ptr(), N * H * W, gamma.data_ptr(), beta.data_ptr()
            f.running_mean, f.running_var, f.eps, f.momentum, f.training = rm.data_ptr(), rv.data_ptr(), 1e-5, 0.1, 1
            f.save_mean, f.save_invstd = smean.data_ptr(), sinv.data_ptr()
            ga, gp = Grid(ffi.MG_BF16, N, Cc, H, W), Grid(ffi.MG_BF16, N, Cc, Ho, Wo)
            code = torch.zeros((N, Ho, Wo, gp.Cp), dtype=torch.uint8, device="cuda")
            if mode == "two":
                ctx.call("mg_bn_residual_forward", C.byref(gy.g()), C.byref(f), None, 1, C.byref(ga.g()), None)
                ctx.call("mg_pool3s2_forward", C.byref(ga.g()), C.byref(gp.g()), ptr(code))
            else:
                ctx.call("mg_bn_relu_pool3_forward", C.byref(gy.g()), C.byref(f), C.byref(gp.g()), ptr(code))
            # backward: gradient of the pooled tensor routed back through the codes, ReLU mask, BatchNorm sums
            gg, gd = Grid(ffi.MG_BF16, N, Cc, Ho, Wo, g), Grid(ffi.MG_BF16, N, Cc, H, W)
            src = (mg_grad_src * 1)()
            src[0].g, src[0].c_offset, src[0].mode, src[0].aux = gg.g(), 0, MG_SRC_POOL3, code.data_ptr()
            dsums = new_sums(2 * Cc)
            if mode == "two":
                ctx.call("mg_grad_combine", C.byref(ga.g()), 1, C.byref(gy.g()), 1, src, C.byref(gd.g()), ptr(dsums))
            else:
                ctx.call("mg_grad_combine", C.byref(gp.g()), 2, C.byref(gy.g()), 1, src, C.byref(gd.g()), ptr(dsums))
            torch.cuda.synchronize()
            res[mode] = [gp.t.clone(), code[..., :Cc].clone(), gd.t.clone(), dsums.clone(), rm.clone(), rv.clone(), smean.clone(), sinv.clone(),
                         gy.scale.clone(), gy.shift.clone()]
        names = ["pooled", "codes", "D", "bn backward sums", "running_mean", "running_var", "save_mean", "save_invstd", "scale", "shift"]
        for nm, a, b in zip(names, res["two"], res["fused"]):
            assert torch.equal(a, b), (nm, (N, Cc, H, W), int((a != b).sum()), a.numel())
        assert res["fused"][0].abs().sum() > 0 and res["fused"][2].abs().sum() > 0
    ctx.close()


# ---------------------------------------------------------------- head, criteria, optimiser
def test_logsoftmax_nll_and_fused(ctx):
    N, Cc = 6, 37
    x = rnd(N, Cc, 1, 1)
    t = rng.integers(0, Cc, N)
    lp_ref = O.logsoftmax_forward(x.reshape(N, Cc))
    gl = Grid(ctx.dtype, N, Cc, 1, 1, x)
    lp = torch.zeros(N, Cc, device="cuda")
    ctx.call("mg_logsoftmax_forward", C.byref(gl.g()), ptr(lp))
    torch.cuda.synchronize()
    assert np.allclose(lp.cpu().numpy(), lp_ref, atol=1e-5)
    loss = torch.zeros(1, device="cuda")
    go = torch.zeros(N, Cc, device="cuda")
    td = dev(t, torch.int32)
    ctx.call("mg_nll_criterion", ptr(lp), ptr(td), N, Cc, ptr(loss), ptr(go), 1.0)
    torch.cuda.synchronize()
    assert np.allclose(loss.item(), O.nll_forward(lp_ref, t), rtol=1e-5)
    assert np.allclose(go.cpu().numpy(), O.nll_backward(lp_ref, t))
    dl = Grid(ctx.dtype, N, Cc, 1, 1)
    ctx.call("mg_logsoftmax_backward", ptr(lp), ptr(go), C.byref(dl.g()))
    ref = O.logsoftmax_backward(lp_ref, O.nll_backward(lp_ref, t)).reshape(N, Cc, 1, 1)
    assert max_rel(dl.nchw(), ref) <= TOL[ctx.dtype]
    # fused LogSoftMax + ClassNLLCriterion
    loss.zero_()
    dl2 = Grid(ctx.dtype, N, Cc, 1, 1)
    ctx.call("mg_nll_forward_backward", C.byref(gl.g()), ptr(td), None, ptr(loss), C.byref(dl2.g()), 1.0)
    torch.cuda.synchronize()
    assert np.allclose(loss.item(), O.nll_forward(lp_ref, t), rtol=1e-5)
    assert max_rel(dl2.nchw(), ref) <= TOL[ctx.dtype]


def test_sigmoid_bce(ctx):
    x = rnd(2, 3, 5, 5)
    t = (rng.random((2, 3, 5, 5)) > 0.5).astype(np.float64)
    p_ref = O.sigmoid_forward(x)
    gx = Grid(ctx.dtype, 2, 3, 5, 5, x)
    p = torch.zeros(2, 3, 5, 5, device="cuda")
    ctx.call("mg_sigmoid_forward", C.byref(gx.g()), ptr(p))
    loss, gp = torch.zeros(1, device="cuda"), torch.zeros_like(p)
    ctx.call("mg_bce_criterion", ptr(p), ptr(dev(t)), p.numel(), ptr(loss), ptr(gp), 1.0)
    torch.cuda.synchronize()
    assert np.allclose(p.cpu().numpy(), p_ref, atol=1e-6)
    assert np.allclose(loss.item(), O.bce_forward(p_ref, t), rtol=1e-4)
    assert np.allclose(gp.cpu().numpy(), O.bce_backward(p_ref, t), rtol=1e-3, atol=1e-7)
    dx = Grid(ctx.dtype, 2, 3, 5, 5)
    ctx.call("mg_sigmoid_backward", ptr(p), ptr(gp), C.byref(dx.g()))
    ref = O.bce_backward(p_ref, t) * p_ref * (1 - p_ref)
    assert max_rel(dx.nchw(), ref) <= max(TOL[ctx.dtype], 1e-3)


def test_sgd_step_matches_optim_sgd(ctx):
    w, st = rng.standard_normal(1000), {}
    dw, dv = dev(w), torch.zeros(1000, device="cuda")
    for it in range(3):
        g = rng.standard_normal(1000)
        w = O.sgd_step(w, g, st, 0.1, 0.9, 1e-4)
        ctx.call("mg_sgd_step", ptr(dw), ptr(dev(g)), ptr(dv), 1000, 0.1, 0.9, 1e-4, int(it == 0))
    torch.cuda.synchronize()
    assert np.allclose(dw.cpu().numpy(), w, atol=1e-5)


def test_launch_counter_counts_our_kernels(ctx):
    n0 = ctx.launches()
    g = Grid(ctx.dtype, 1, 3, 4, 4, rnd(1, 3, 4, 4))
    o = Grid(ctx.dtype, 1, 3, 2, 2)
    ctx.call("mg_pool_forward", C.byref(g.g()), C.byref(o.g()), 0, None)
    assert ctx.launches() == n0 + 1
