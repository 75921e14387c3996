"""Cost of the split backward on R-MG-34 (ilsvrc/rnmg depth 34), batch 256 at 224x224, bf16, one GPU.

Prints, from one process: the GPU's name and power limit; ms per evaluate() forward + backward against evaluate() forward +
updateGradInput on a model with needInputGrad (the image-gradient use: saliency maps, adversarial inputs), and ms per training
step (fwd + NLL + backward + SGD) against the same step written with updateGradInput + accGradParameters.  The two variants of
each pair are timed with CUDA events in alternating rounds after warm-up; the image gradients of the first pair are compared.
    python scratch/split_backward_bench.py [--rounds 5] [--steps 10] [--batch 256]
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


def build(batch, need_input_grad):
    torch.manual_seed(2)
    net = B.load_net("ilsvrc/rnmg")
    model = net.createModel(B.Opt(nGPU=1, depth=34))
    model.precision = "bf16"
    model.needInputGrad = need_input_grad
    model.cuda()
    params, grads = model.getParameters()
    g = torch.Generator(device="cpu").manual_seed(3)
    x = torch.randn(batch, 3, 224, 224, generator=g).cuda()
    t = torch.randint(1, 1001, (batch,), generator=g).cuda()
    return net, model, params, grads, x, t


def timed(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def alternate(fns, rounds, steps):
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            times[k].append(timed(fn, steps))
    return {k: [round(v, 3) for v in vs] for k, vs in times.items()}, {k: round(sorted(vs)[len(vs) // 2], 3) for k, vs in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=256)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None}), flush=True)

    # image gradient: evaluate() + needInputGrad, backward (every weight gradient too) vs updateGradInput alone
    net, model, _, _, x, t = build(args.batch, True)
    model.evaluate()
    crit = net.createCriterion()
    out = model.forward(x)
    crit.forward(out, t)
    go = crit.backward(out, t).clone()
    gis = {}

    def with_backward():
        model.forward(x)
        gis["backward"] = model.backward(x, go)

    def with_update():
        model.forward(x)
        gis["update"] = model.updateGradInput(x, go)
    all_ms, med = alternate({"backward": with_backward, "updateGradInput": with_update}, args.rounds, args.steps)
    with_backward(); a = gis["backward"].clone()
    with_update(); b = gis["update"].clone()
    torch.cuda.synchronize()
    print(json.dumps({"workload": f"ilsvrc/rnmg depth 34, B {args.batch}, bf16, evaluate() forward + image gradient",
                      "ms_forward_backward": all_ms["backward"], "ms_forward_updateGradInput": all_ms["updateGradInput"],
                      "median_backward": med["backward"], "median_updateGradInput": med["updateGradInput"],
                      "image_gradient_bit_equal": bool(torch.equal(a, b))}), flush=True)
    del model, out, go, gis, a, b
    torch.cuda.empty_cache()

    # training step: backward vs updateGradInput + accGradParameters
    net, model, params, grads, x, t = build(args.batch, False)
    crit = net.createCriterion()
    st = dict(learningRate=0.05, momentum=0.9, weightDecay=5e-4, dampening=0.0)

    def step(split):
        def run():
            model.zeroGradParameters()

            def feval(_p):
                out = model.forward(x)
                crit.forward(out, t)
                go = crit.backward(out, t)
                if split:
                    model.updateGradInput(x, go)
                    model.accGradParameters(x, go)
                else:
                    model.backward(x, go)
                return 0.0, grads
            net.btrain(params, feval, st)
        return run
    all_ms, med = alternate({"backward": step(False), "split": step(True)}, args.rounds, args.steps)
    print(json.dumps({"workload": f"ilsvrc/rnmg depth 34, B {args.batch}, bf16, fwd+NLL+bwd+SGD",
                      "ms_per_step_backward": all_ms["backward"], "ms_per_step_split": all_ms["split"],
                      "median_backward": med["backward"], "median_split": med["split"]}), flush=True)


if __name__ == "__main__":
    main()
