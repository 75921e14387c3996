"""2-rank worker of tests/test_split_backward.py (launched with torchrun): a DataParallel step written with updateGradInput +
accGradParameters equals the step written with backward bit for bit -- with per-replica BatchNorm, with -bnSync, and with
-iterSize 2 (two micro-batches accumulated before the step)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "multigrid-neural-architectures_b200"))
import numpy as np, torch, torch.distributed as dist
from mgconv import builders as B, multigpu

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
variant = sys.argv[1]
os.environ["MGCONV_AUTOTUNE"] = "0"
rng = np.random.default_rng(11)
Bg = 16
x = torch.from_numpy(rng.standard_normal((2, Bg, 3, 32, 32)).astype(np.float32))
t = torch.from_numpy(rng.integers(1, 101, (2, Bg)))
lo, hi = multigpu.shard_range(Bg, world, rank)


def run(split):
    torch.manual_seed(5)
    model = B.cifar_rnmg.createModel(B.Opt(nLayer=1, nGPU=world, bnSync=variant == "bnSync"))
    model.model.precision = "bf16"
    model.cuda()
    params, grads = model.getParameters()
    crit = B.cifar_rnmg.createCriterion()
    model.zeroGradParameters()
    for mb in range(2 if variant == "iterSize2" else 1):
        xs, ts = x[mb, lo:hi].cuda(), t[mb, lo:hi].cuda()
        out = model.forward(xs)
        crit.forward(out, ts)
        go = crit.backward(out, ts)
        if split:
            model.updateGradInput(xs, go)
            model.accGradParameters(xs, go, 1.0)
        else:
            model.backward(xs, go, 1.0)
    torch.cuda.synchronize()
    bns = model.findModules("nn.SpatialBatchNormalization")
    return [out.clone(), grads.clone()] + [b.running_var.clone() for b in bns]


ref, got = run(False), run(True)
for i, (a, b) in enumerate(zip(ref, got)):
    assert torch.equal(a, b), (variant, i)
dist.barrier()
print(f"dp-split ok rank {rank} [{variant}]", flush=True)
dist.destroy_process_group()
