#!/usr/bin/env python
"""bench.py -- R-MG-34 ImageNet-shape training throughput (BASELINE.json metric), one JSON line.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA hot path)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed (.npy)

A "step" is what pipelines/standard/train.lua:trainBatch does between its synchronisations:
zeroGradParameters -> NETOBJ.ftrain (forward, ClassNLL, backward; models/basic_model.lua:56-62)
-> NETOBJ.btrain (optim.sgd momentum .9, wd 1e-4, lr .1; 64-66) on `-netType ilsvrc/rnmg -depth 34`,
synthetic N(0,1) images [B,3,224,224] and uniform labels 1..1000, B = 256 per GPU (weak scaling).

value  : images/s with the batch already resident in HBM (CUDA events, max over ranks).
e2e    : the same step driven from HOST buffers: pinned-memory H2D copy of images+labels (the
         reference's put2GPU, utils/utilfuncs.lua:3-30) and a D2H read of the loss, inside the timed region.
roofline: the implicit-GEMM multigrid convolution kernels (forward, dgrad, wgrad) -- algorithmic
         FLOPs = 2*MACs*3 of every conv of the plan / their summed CUDA-event time in the timed steps.
cpu_baseline: the oracle's PyTorch-CPU restatement of the same network (the reference's Torch7 nn
         path cannot run: no Lua/Torch7 here) on a bounded sample, all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "multigrid-neural-architectures_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "R-MG-34 train images/sec"
WORKLOAD = "R-MG-34 (ilsvrc/rnmg -depth 34) ImageNet 224x224 synthetic, batch 256/GPU, fwd+NLL+bwd+SGD"

# BASELINE.json configs: the headline (default) and the secondary ones, all through the same code path.
# name: (netType, createModel options, per-GPU input shape, criterion kind, classes / output maps, oracle ctor name + args, workload text)
CONFIGS = {
    "rmg34": ("ilsvrc/rnmg", dict(depth=34), (256, 3, 224, 224), "nll", 1000, ("ilsvrc_rnmg", (34,)), WORKLOAD),
    "rmg22": ("cifar/rnmg", dict(nLayer=2), (128, 3, 32, 32), "nll", 100, ("cifar_rnmg", (2,)),
              "R-MG-22 (cifar/rnmg -nLayer 2) CIFAR-100 32x32 synthetic, batch 128/GPU, fwd+NLL+bwd+SGD"),
    "prnmg30": ("cifar/prnmg", dict(nLayer=2), (256, 3, 32, 32), "nll", 100, ("cifar_prnmg", (2,)),
                "PR-NMG-30 (cifar/prnmg -nLayer 2) CIFAR-100 32x32 synthetic, batch 256/GPU, fwd+NLL+bwd+SGD"),
    "mg6": ("cifar/nmg", dict(nLayer=1), (64, 3, 32, 32), "nll", 100, ("cifar_nmg", (1,)),
            "MG-6 (cifar/nmg -nLayer 1) CIFAR-100 32x32 synthetic, batch 64/GPU, fwd+NLL+bwd+SGD"),
    "prnmg_mnist": ("mnist-cluttered/prnmg.mnist", dict(nLayer=1, dataset="mnist-spt"), (128, 1, 64, 64), "bce", 1, ("mnist_prnmg", (1, 1)),
                    "PR-NMG (mnist-cluttered/prnmg.mnist) 64x64 synthetic, batch 128/GPU, fwd+BCE+bwd+SGD"),
    "unmg": ("mnist-cluttered/unmg", dict(dataset="mnist-seg"), (128, 1, 64, 64), "bce", 10, ("mnist_unmg", (10,)),
             "U-MG (mnist-cluttered/unmg, nn.ConcatUnet) 64x64 synthetic, batch 128/GPU, fwd+BCE+bwd+SGD"),
}
CONFIG_METRIC = {"rmg34": METRIC, "rmg22": "R-MG-22 train images/sec", "prnmg30": "PR-NMG-30 train images/sec", "mg6": "MG-6 train images/sec",
                 "prnmg_mnist": "PR-NMG MNIST-cluttered train images/sec", "unmg": "U-MG MNIST-cluttered train images/sec"}


# --dump-outputs: an array with more elements than this (16 MB in float32) is written as a sample, so that a dump of the
# four arrays of a step stays under 64 MB
DUMP_MAX_ELEMENTS = 1 << 22


def dump_outputs(dirname, arrays):
    """Write each tensor of `arrays` (name -> tensor) as DIR/<name>.npy in float32.  A larger array is replaced by the
    elements of its flattened form at DUMP_MAX_ELEMENTS sorted indices drawn with a fixed seed: the same positions in
    every run, so that the dumps of two builds compare element for element."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        a = torch.as_tensor(t).detach().float()
        if a.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(a.numel(), DUMP_MAX_ELEMENTS, replace=False))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(dirname, name + ".npy"), a.cpu().numpy())


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("bf16_tflops_sustained", 1405.9), d.get("hbm_gbs", 6542.1), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        self.proc = p
        for line in p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])
            if self.stop_flag:
                break
        p.kill()

    def summary(self):
        self.stop_flag = True
        time.sleep(0.25)
        try:
            self.proc.kill()
        except Exception:
            pass
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(cfg, batch, steps, warmup):
    """oracle port of the same network on the host cores (bounded sample): `warmup` untimed + `steps` timed train steps"""
    import torch
    from oracle import builders as OB
    nt, opt, shape, kind, ncls, (octor, oargs), workload = CONFIGS[cfg]
    torch.manual_seed(2)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    om = getattr(OB, octor)(*oargs)
    opt_ = torch.optim.SGD(om.parameters(), lr=0.1 if cfg == "rmg34" else 0.05, momentum=0.9, weight_decay=1e-4)
    x = torch.randn(batch, *shape[1:])
    if kind == "nll":
        t = torch.randint(0, ncls, (batch,))
    else:
        t = (torch.rand(batch, ncls, shape[2], shape[3]) < 0.1).float()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt_.zero_grad(set_to_none=False)
        out = om(x)
        loss = torch.nn.functional.nll_loss(out, t) if kind == "nll" else torch.nn.functional.binary_cross_entropy(out, t)
        loss.backward()
        opt_.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return {"value": batch / dt, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"{workload.split(',')[0]} fp32 PyTorch-CPU oracle, batch {batch}, {steps} timed steps after {warmup} warm-up"}, dt


def run_reference(args):
    """the reference's CPU path on this box's host cores.  Torch7 cannot run here (no Lua), so this is the oracle's PyTorch-CPU
    restatement of the same network, on a bounded sample (batch --cpu-batch) of the same workload; `steps` / `warmup` in the
    line are the counts really run (the requested ones, capped so that the arm ends within a few minutes)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.config
    batch = args.cpu_batch or (32 if cfg == "rmg34" else min(CONFIGS[cfg][2][0], 128))
    _, dt1 = cpu_baseline(cfg, batch, 1, 0)                                   # one probing step (also the first warm-up)
    budget_s = 150.0
    steps = max(1, min(args.steps, int(budget_s / max(dt1, 1e-3)) - args.warmup))
    warmup = max(0, min(args.warmup, 3))
    cb, dt = cpu_baseline(cfg, batch, steps, warmup)
    line = {"metric": CONFIG_METRIC[cfg], "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": CONFIGS[cfg][6], "note": "reference = Torch7 nn CPU path; Torch7 cannot run here, timed as the oracle's "
                       "PyTorch-CPU restatement on a bounded sample", "sample_batch": batch, "steps_requested": args.steps, "warmup_requested": args.warmup},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mgconv")
    ap.add_argument("--config", default="rmg34", choices=sorted(CONFIGS), help="BASELINE.json config (default: the headline R-MG-34)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the config's)")
    ap.add_argument("--depth", type=int, default=34)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--cpu-batch", type=int, default=0, help="batch of the CPU sample (default 32 for R-MG-34)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--bn-sync", action="store_true", help="cross-replica BatchNorm statistics (default: per replica, as the reference)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output, loss, parameters and parameter gradients of the last "
                    "timed step as DIR/<name>.npy (float32; arrays above %d elements as a fixed seeded sample). Inputs and "
                    "initial weights are seeded: two runs with the same arguments write the same values" % DUMP_MAX_ELEMENTS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computes; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from mgconv import builders as B, ffi
    from mgconv.engine import criterion_ctx

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"

    torch.manual_seed(2)  # -manualSeed default (opts.lua:23); identical initial weights on every rank
    nt, copt, shape, kind, ncls, _, workload = CONFIGS[args.config]
    copt = dict(copt)
    if args.config == "rmg34":
        copt["depth"] = args.depth
    net = B.load_net(nt)
    model = net.createModel(B.Opt(nGPU=world, bnSync=args.bn_sync, **copt))
    (model.model if hasattr(model, "model") else model).precision = args.precision
    model.cuda()
    criterion = net.createCriterion()
    params, grads = model.getParameters()
    rule = net.trainRule(1, B.Opt(nEpochs=20))   # opts.lua:32: -nEpochs defaults to 20
    optimState = dict(learningRate=rule["LR"], momentum=0.9, weightDecay=rule["WD"], dampening=0.0, learningRateDecay=0.0)

    Bsz = args.batch or shape[0]
    headline = args.config == "rmg34" and args.depth == 34 and Bsz == 256
    g = torch.Generator(device="cpu").manual_seed(100 + rank)
    host_x = torch.randn(Bsz, *shape[1:], generator=g).pin_memory()
    if kind == "nll":
        host_t = torch.randint(1, ncls + 1, (Bsz,), generator=g).pin_memory()
    else:
        host_t = (torch.rand(Bsz, ncls, shape[2], shape[3], generator=g) < 0.1).float().pin_memory()
    dev_x, dev_t = host_x.to(dev), host_t.to(dev)
    state = {}

    def step(x, t):
        model.zeroGradParameters()

        def feval(_p):
            outputs, err = net.ftrain(x, t, model, criterion)
            state["outputs"], state["loss"] = outputs, err
            return err, grads
        net.btrain(params, feval, optimState)

    def engine():
        return (model.model if hasattr(model, "model") else model)._engine

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step(dev_x, dev_t)
    sync_all()
    eng = engine()
    cctx = criterion_ctx(params)
    l0 = eng.ctx.launches() + cctx.launches()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.profiler.start()   # ncu --profile-from-start off captures exactly the timed steps
    e0.record()
    for _ in range(args.steps):
        step(dev_x, dev_t)
    e1.record()
    sync_all()
    torch.cuda.profiler.stop()
    clocks = sampler.summary()
    ms = e0.elapsed_time(e1)
    launches = eng.ctx.launches() + cctx.launches() - l0
    if args.dump_outputs and rank == 0:
        # now, before the steps below overwrite the output buffers and move the parameters
        dump_outputs(args.dump_outputs, {"output": state["outputs"], "loss": state["loss"], "parameters": params, "grad_parameters": grads})
    # Roofline of the convolution kernels: the timed region above runs WITHOUT the per-call event instrumentation (it costs
    # ~3 % of the step) and, with lanes, overlaps kernels of different scales, so a kernel's own duration cannot be read
    # there.  It is taken from extra steps of the SERIAL plan (one stream, kernels back to back -- what the ncu launch
    # list in profiles/ sees) right after the timed region, every conv entry point bracketed by CUDA events on its stream.
    lanes = eng.n_lanes if eng._use_lanes() else 1
    eng.n_lanes = 1
    step(dev_x, dev_t)
    sync_all()
    eng.ctx.call("mg_ctx_profile", 1)
    ps = max(1, min(args.steps, 5))
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(ps):
        step(dev_x, dev_t)
    s1.record()
    sync_all()
    sp = eng.ctx.profile_read()
    eng.ctx.call("mg_ctx_profile", 0)
    serial = {"steps": ps, "ms_per_step": s0.elapsed_time(s1) / ps, "conv_ms_per_step": sp["conv_ms"] / ps, "lanes": lanes,
              "conv_launches_per_step": sp["conv_launches"] / ps}
    eng.n_lanes = lanes
    if world > 1:
        tms = torch.tensor([ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = tms.item()
    ms_per_step = ms / args.steps
    value = Bsz * world / (ms_per_step * 1e-3)

    # end to end through the public API from host buffers: every step's batch crosses PCIe inside the
    # timed region (put2GPU, utils/utilfuncs.lua:3-30, into persistent device tensors) and the loss is
    # read back.  Like the reference's loader threads (data.lua:15-31) the NEXT batch is staged while the
    # current one trains: the copy runs on a side stream into the other of two device buffers.
    e2e = None
    if not args.no_e2e:
        from mgconv.utilfuncs import Put2GPU
        stg = Put2GPU(local)                         # the package's double-buffered put2GPU (mgconv/utilfuncs.py)
        sync_all()
        e0.record()
        stg.stage(0, host_x, host_t)
        for i in range(args.steps):
            if i + 1 < args.steps:
                stg.stage(i + 1, host_x, host_t)
            bx, bt = stg.get(i)
            step(bx, bt)
            stg.done(i)
            _ = float(state["loss"])                # D2H read of the step's loss
        e1.record()
        sync_all()
        ems = e0.elapsed_time(e1)
        if world > 1:
            tms = torch.tensor([ems], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ems = tms.item()
        e2e = {"value": Bsz * world / (ems / args.steps * 1e-3), "unit": "images/s",
               "h2d_bytes_per_step": host_x.numel() * host_x.element_size() + host_t.numel() * host_t.element_size(), "d2h_bytes_per_step": 4,
               "note": "H2D of batch i+1 overlaps step i on a copy stream (double-buffered put2GPU)"}

    in_sync = None
    if world > 1:   # every rank applied the same all-reduced gradient: parameters must be bit-identical
        lo, hi = params.clone(), params.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        in_sync = bool(torch.equal(lo, hi))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    from mgconv import lower as L
    summ = L.plan_summary(eng.plan)
    # per image: 2 FLOP/MAC x (fwd + dgrad + wgrad); the three stem convs read the image and have no dgrad
    no_dgrad = sum(sum(t.C for t, _ in o.segs) * o.Cout * o.k * o.k * o.Ho * o.Wo for o in eng.conv_ops if not o.needs_dgrad)
    conv_flops_step = Bsz * (2.0 * summ["macs"] * 3 - 2.0 * no_dgrad)
    tf_peak, hbm_peak, which = peaks()
    conv_ms_step = serial["conv_ms_per_step"]
    ref_step_ms = serial["ms_per_step"]
    achieved = conv_flops_step / (conv_ms_step * 1e-3) / 1e12 if conv_ms_step else None
    # DRAM bytes of the same launches from the committed ncu pass (profiles/): per step, like `achieved`
    traffic, traffic_src = None, None
    tname = "r2_conv_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r2_conv_traffic.json")) else "r1i_conv_traffic.json"
    tpath = os.path.join(ROOT, "profiles", tname)
    if os.path.exists(tpath) and headline:
        tj = json.load(open(tpath))
        traffic, traffic_src = tj["dram_bytes_per_step"], f"profiles/{tname} (ncu dram__bytes_read.sum + dram__bytes_write.sum over the conv launches of one step)"
    roofline = {"bound": "tensor", "kernel": "implicit-GEMM multigrid conv (fwd+dgrad+wgrad launches)",
                "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": (achieved / tf_peak) if achieved else None,
                "traffic": traffic, "traffic_unit": "bytes per step over the same launches", "traffic_source": traffic_src, "peak_source": which, "conv_ms_per_step": conv_ms_step, "conv_launches_per_step": serial["conv_launches_per_step"],
                "share_of_step": (conv_ms_step / ref_step_ms) if conv_ms_step else None,
                "algorithmic_flops_per_step": conv_flops_step,
                "timing": ("CUDA events around every conv entry point in %d extra steps of the serial plan (lanes off, %.2f ms/step) right after the "
                           "timed region; the timed steps themselves run uninstrumented on %d lane(s)" % (serial["steps"], serial["ms_per_step"], serial["lanes"]))}
    cb = None
    if not args.no_cpu_baseline and world == 1:
        cb, _ = cpu_baseline(args.config, args.cpu_batch or (8 if args.config == "rmg34" else min(Bsz, 64)), 2, 1)
    line = {"metric": CONFIG_METRIC[args.config], "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": workload if (args.config != "rmg34" or headline) else f"R-MG-{args.depth} batch {Bsz}/GPU (NOT the headline config)",
                       "name": args.config,
                       "global_batch": Bsz * world, "parallelism": f"dp{world}", "bn": "sync" if (args.bn_sync and world > 1) else "per-replica (reference DataParallelTable behaviour)", "l2_flush": "inputs larger than L2 (%.0f MB of inputs, %.1f GB of activations per step)" % (host_x.numel() * 4 / 1e6, eng.bytes / 1e9),
                       "impl": os.environ.get("MGCONV_IMPL", "auto"), "device_bytes": eng.bytes,
                       "dp_params_in_sync": in_sync, "tc_launches": eng.ctx.tc_launches(), "lanes": eng.n_lanes if eng._use_lanes() else 1},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cb,
            "loss": float(state["loss"])}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
