"""CPU ORACLE (test infrastructure, NOT product code) -- Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy
as 1, 2, 3", SC 2011; the generator of Random123 and cuRAND) in numpy, the dropout mask the product's nn.Dropout draws
with it (include/mgconv.h, mg_dropout), a Torch7 nn.Dropout that replays such masks and the P-NMG builder with -isDropout:

  element i -- its NHWC index over the logical channels -- is kept iff word (i & 3) of
  Philox4x32-10(counter = (i >> 2, op, step mod 2^32, rank), key = (seed mod 2^32, seed >> 32)) >= t,
  t = min(2^32 - 1, floor(p * 2^32)) with p rounded to fp32; kept elements are scaled by s = fp32(1 / (1 - p)).

Written from the algorithm's definition, not from the product's kernels; tests/test_dropout.py checks it against the
published known-answer vectors first.
"""
import math

import numpy as np
import torch

_M0, _M1 = 0xD2511F53, 0xCD9E8D57      # round multipliers
_W0, _W1 = 0x9E3779B9, 0xBB67AE85      # key schedule (Weyl) increments
_U32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: uint32 array [..., 4]; key: (k0, k1) -> uint32 array [..., 4]"""
    ctr = np.asarray(ctr, dtype=np.uint64)
    c = [ctr[..., j] for j in range(4)]
    k0, k1 = np.uint64(int(key[0]) & 0xFFFFFFFF), np.uint64(int(key[1]) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _U32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _U32]
        k0 = (k0 + np.uint64(_W0)) & _U32
        k1 = (k1 + np.uint64(_W1)) & _U32
    return np.stack(c, -1).astype(np.uint32)


def threshold(p):
    p32 = float(np.float32(p))
    return min(2 ** 32 - 1, math.floor(p32 * 2.0 ** 32))


def scale(p):
    return np.float32(1.0 / (1.0 - float(np.float32(p))))


def keep_flat(n, p, seed, op, step, rank):
    """keep flags of elements i = 0 .. n-1"""
    g = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.stack([g, np.full_like(g, op), np.full_like(g, int(step) & 0xFFFFFFFF), np.full_like(g, rank)], -1)
    u = philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32)).reshape(-1)[:n]
    return u >= np.uint32(threshold(p))


def keep_nchw(N, C, H, W, p, seed, op, step, rank):
    """keep flags of an N x C x H x W tensor (drawn in NHWC order over its C logical channels)"""
    return keep_flat(N * H * W * C, p, seed, op, step, rank).reshape(N, H, W, C).transpose(0, 3, 1, 2)


class Dropout(torch.nn.Module):
    """nn.Dropout(p), Torch7's default v2 form: training y = x * mask / (1 - p), evaluation y = x.  The mask is not random
    here: it is keep_nchw of (seed, op, step, rank), set on the module before a forward, so that a test can replay the
    product's masks.  last_shape: the input shape of the last training forward."""

    def __init__(self, p=0.5):
        super().__init__()
        self.p = p
        self.seed, self.op, self.step, self.rank = 0, 0, 1, 0
        self.last_shape = None

    def forward(self, x):
        if not self.training or self.p == 0:
            return x
        self.last_shape = tuple(x.shape)
        keep = torch.from_numpy(np.ascontiguousarray(keep_nchw(*x.shape, self.p, self.seed, self.op, self.step, self.rank)))
        return x * keep.to(x.dtype) * float(scale(self.p))


def cifar_pnmg(nLayer=1, nClass=100, blocks=None, dropouts=(0.1, 0.2, 0.3, 0.4)):
    """oracle.builders.cifar_pnmg with -isDropout (models/cifar/pnmg.lua:25-27): nn.Dropout(dropouts[b - 2]) between
    ResampleConcat and every convolution of blocks b = 2..5.  Those blocks are the last nLayer plain mg-convs + mgPool
    each, in front of the classifier, in the builder's top-level list."""
    from . import builders as OB
    model = OB.cifar_pnmg(nLayer, nClass, blocks)
    mods = list(model)
    end = len(mods) - 2                      # mgPool of the last block
    for p in reversed(dropouts):
        for mg_conv in mods[end - nLayer:end]:
            for grid in mg_conv.mods:        # Sequential{ ResampleConcat grid, Conv, BN, ReLU }
                grid.insert(1, Dropout(p))
        end -= nLayer + 1
    return model
