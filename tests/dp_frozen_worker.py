"""2-rank worker of tests/test_frozen_bn.py (launched with torchrun): -bnSync with the first quarter of the BatchNorm layers frozen
(bn:evaluate() inside a training model).  Frozen layers all-reduce no statistics in either direction and every rank adds its full
share of their dgamma / dbeta; active layers use the global statistics.  The two-GPU step must equal the single-GPU step on the
concatenated batch: same log-probabilities per shard, same (all-reduced) parameter gradients, frozen running statistics untouched."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "multigrid-neural-architectures_b200"))
import numpy as np, torch, torch.distributed as dist
from mgconv import builders as B, multigpu

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
rng = np.random.default_rng(11)
Bg = 16
x = torch.from_numpy(rng.standard_normal((Bg, 3, 32, 32)).astype(np.float32))
t = torch.from_numpy(rng.integers(1, 101, Bg))


def run(nGPU, xs, ts):
    torch.manual_seed(5)
    model = B.cifar_rnmg.createModel(B.Opt(nLayer=1, nGPU=nGPU, bnSync=nGPU > 1))
    inner = model.model if nGPU > 1 else model
    inner.precision = "fp32"
    bns = inner.findModules("nn.SpatialBatchNormalization")
    g = torch.Generator().manual_seed(7)
    for b in bns:
        b.running_mean.copy_(torch.randn(b.running_mean.shape, generator=g) * 0.2)
        b.running_var.copy_(torch.rand(b.running_var.shape, generator=g) * 1.5 + 0.5)
    frozen = range(len(bns) // 4)
    for i in frozen:
        bns[i].evaluate()
    model.cuda()
    params, grads = model.getParameters()
    rs = [(b.running_mean.clone(), b.running_var.clone()) for b in bns]
    crit = B.cifar_rnmg.createCriterion()
    model.zeroGradParameters()
    out, err = B.cifar_rnmg.ftrain(xs.cuda(), ts.cuda(), model, crit)
    torch.cuda.synchronize()
    for i in frozen:
        assert torch.equal(bns[i].running_mean, rs[i][0]) and torch.equal(bns[i].running_var, rs[i][1]), i
    assert any(not torch.equal(b.running_var, v) for b, (_, v) in list(zip(bns, rs))[len(bns) // 4:])
    return out.clone(), float(err), grads.clone()


lo, hi = multigpu.shard_range(Bg, world, rank)
out2, err2, g2 = run(world, x[lo:hi], t[lo:hi])
out1, err1, g1 = run(1, x, t)
rel = lambda a, b: float((a - b).norm() / b.norm())
e_out, e_g = rel(out2, out1[lo:hi]), rel(g2, g1)
assert e_out <= 1e-4, ("log-probabilities", e_out)
assert e_g <= 1e-3, ("gradients", e_g)
dist.barrier()
print(f"dp-frozen ok rank {rank}: sync-BN with frozen layers vs single GPU: out {e_out:.2e} grad {e_g:.2e}", flush=True)
dist.destroy_process_group()
