"""Cost of -isDropout on P-NMG (cifar/pnmg, wide blocks, nLayer 1), batch 256, bf16, one GPU.

Prints, from one process: the GPU's name and power limit; ms per training step (fwd + NLL + bwd + SGD) with isDropout off and
on, timed with CUDA events in alternating rounds after warm-up; the bytes the dropout passes move per step, computed from the
plan's shapes; and their kernel time from a separate torch.profiler run.
    python scratch/dropout_bench.py [--rounds 5] [--steps 20]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "multigrid-neural-architectures_b200"))
import torch
from mgconv import builders as B

SHAPE = (256, 3, 32, 32)


def build(dropout):
    torch.manual_seed(2)
    net = B.load_net("cifar/pnmg")
    model = net.createModel(B.Opt(nGPU=1, nLayer=1, isDropout=dropout))
    model.precision = "bf16"
    model.cuda()
    params, grads = model.getParameters()
    crit = net.createCriterion()
    st = dict(learningRate=0.05, momentum=0.9, weightDecay=5e-4, dampening=0.0)
    g = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn(*SHAPE, generator=g).cuda()
    t = torch.randint(1, 101, (SHAPE[0],), generator=g).cuda()

    def step():
        model.zeroGradParameters()

        def feval(_p):
            net.ftrain(x, t, model, crit)
            return 0.0, grads
        net.btrain(params, feval, st)
    return model, step


def dropout_bytes(plan):
    """HBM bytes of the dropout passes per step: forward reads every source element once and writes the dropped tensor;
    backward reads and writes its gradient in place (bf16, padded channel pitch)"""
    fwd = bwd = 0
    for d in plan.drops:
        t = d.out
        fwd += sum(s.N * s.H * s.W * s.Cp * 2 for s, _ in d.segs) + t.N * t.H * t.W * t.Cp * 2
        bwd += 2 * t.N * t.H * t.W * t.Cp * 2
    return fwd, bwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None}), flush=True)

    runs = {False: build(False), True: build(True)}
    for _, step in runs.values():
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    times = {False: [], True: []}
    for _ in range(args.rounds):
        for dropout in (False, True):
            step = runs[dropout][1]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            e1.synchronize()
            times[dropout].append(e0.elapsed_time(e1) / args.steps)
    model = runs[True][0]
    fwd, bwd = dropout_bytes(model._engine.plan)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    print(json.dumps({"workload": "cifar/pnmg wide nLayer 1, B 256, bf16, fwd+NLL+bwd+SGD",
                      "ms_per_step_off": [round(v, 3) for v in times[False]], "ms_per_step_on": [round(v, 3) for v in times[True]],
                      "median_off": round(med[False], 3), "median_on": round(med[True], 3),
                      "overhead_ms": round(med[True] - med[False], 3),
                      "dropout_ops": len(model._engine.plan.drops),
                      "dropout_bytes_fwd": fwd, "dropout_bytes_bwd": bwd}), flush=True)

    # kernel time of the dropout passes, in a run of its own
    from torch.profiler import profile, ProfilerActivity
    step = runs[True][1]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            step()
        torch.cuda.synchronize()
    us, calls = {}, {}
    for e in prof.key_averages():
        if "dropout" in e.key:
            us[e.key] = e.device_time_total / 5
            calls[e.key] = e.count / 5
    total_us = sum(us.values())
    print(json.dumps({"profiler_steps": 5, "dropout_kernel_us_per_step": round(total_us, 1),
                      "per_kernel_us": {k[:60]: round(v, 1) for k, v in us.items()}, "calls_per_step": {k[:60]: v for k, v in calls.items()},
                      "dropout_GB_per_s": round((fwd + bwd) / (total_us * 1e-6) / 1e9, 1) if total_us else None}), flush=True)


if __name__ == "__main__":
    main()
