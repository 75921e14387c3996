"""Cost of frozen BatchNorm on R-MG-34 (ilsvrc/rnmg depth 34), batch 256 at 224x224, bf16, one GPU.

Prints, from one process: the GPU's name and power limit; ms per training step (fwd + NLL + bwd + SGD) with every BatchNorm
training and with the first quarter of the BatchNorm layers frozen (bn:evaluate()); and ms per evaluate() forward with the
convolutions reducing the BatchNorm statistics (what the plan did before frozen layers skipped them) and without.  Variants are
timed with CUDA events in alternating rounds after warm-up.
    python scratch/frozen_bn_bench.py [--rounds 5] [--steps 10] [--batch 256]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "multigrid-neural-architectures_b200"))
import torch
from mgconv import builders as B, ops as O
from mgconv.ffi import ptr


def build(batch, frozen):
    torch.manual_seed(2)
    net = B.load_net("ilsvrc/rnmg")
    model = net.createModel(B.Opt(nGPU=1, depth=34))
    model.precision = "bf16"
    model.cuda()
    if frozen:
        bns = model.findModules("nn.SpatialBatchNormalization")
        for b in bns[:len(bns) // 4]:
            b.evaluate()
    params, grads = model.getParameters()
    crit = net.createCriterion()
    st = dict(learningRate=0.05, momentum=0.9, weightDecay=5e-4, dampening=0.0)
    g = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn(batch, 3, 224, 224, generator=g).cuda()
    t = torch.randint(1, 1001, (batch,), generator=g).cuda()

    def step():
        model.zeroGradParameters()

        def feval(_p):
            net.ftrain(x, t, model, crit)
            return 0.0, grads
        net.btrain(params, feval, st)
    return model, x, step


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=256)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None}), flush=True)

    # training step: all BatchNorms active vs. the first quarter frozen
    runs = {k: build(args.batch, k) for k in (False, True)}
    for _, _, step in runs.values():
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    times = {False: [], True: []}
    for _ in range(args.rounds):
        for k in (False, True):
            times[k].append(timed(runs[k][2], args.steps))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    print(json.dumps({"workload": f"ilsvrc/rnmg depth 34, B {args.batch}, bf16, fwd+NLL+bwd+SGD",
                      "ms_per_step_active": [round(v, 3) for v in times[False]], "ms_per_step_quarter_frozen": [round(v, 3) for v in times[True]],
                      "median_active": round(med[False], 3), "median_quarter_frozen": round(med[True], 3)}), flush=True)

    # evaluate() forward: statistics skipped (this plan) vs reduced and unused (the plan before)
    model, x, _ = runs[False]
    model.evaluate()
    skip = lambda: model.forward(x)
    stats_fn = O._stats

    def reduce_stats():
        O._stats = lambda conv: ptr(conv.sums)
        try:
            model.forward(x)
        finally:
            O._stats = stats_fn
    for fn in (skip, reduce_stats):
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    ev = {"skip": [], "reduce": []}
    for _ in range(args.rounds):
        ev["skip"].append(timed(skip, args.steps))
        ev["reduce"].append(timed(reduce_stats, args.steps))
    med = {k: sorted(v)[len(v) // 2] for k, v in ev.items()}
    print(json.dumps({"workload": f"ilsvrc/rnmg depth 34, B {args.batch}, bf16, evaluate() forward",
                      "ms_stats_skipped": [round(v, 3) for v in ev["skip"]], "ms_stats_reduced": [round(v, 3) for v in ev["reduce"]],
                      "median_skipped": round(med["skip"], 3), "median_reduced": round(med["reduce"], 3)}), flush=True)


if __name__ == "__main__":
    main()
