"""Record the libmgconv call sequence of every engine pass without running a kernel, for comparing two versions of the host.

    python scratch/call_trace.py [--pkg DIR] --out FILE

Each network is lowered normally (MGCONV_AUTOTUNE=0), then the engine's context is replaced by a recorder that logs every
ctx.call by name -- with the lane or event id of mg_ctx_lane / mg_ctx_event_record / mg_ctx_event_wait -- and forwards
nothing but set_stream.  Engine.param_done reports are logged as the module's index in model.listModules().  Passes:
forward, backward, updateGradInput, accGradParameters (twice), at MGCONV_LANES 1 and 3 and with -bnSync over 0 and 2 ranks
(one GPU: mg_allreduce_inline is only logged), then a serial step and a laned step again as bench.py's roofline toggles
n_lanes.  `--pkg` puts another copy of the mgconv package first on the path (it loads the same libmgconv.so through
MGCONV_LIB).  Needs a GPU for the device buffers; no kernel runs.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PNMG_OPT = dict(nLayer=1)
# name, network, options, input shape, mode
NETS = [
    ("R-MG-34 B8", "ilsvrc/rnmg", dict(depth=34), (8, 3, 224, 224), "train"),
    ("PR-NMG-30", "cifar/prnmg", dict(nLayer=2), (4, 3, 32, 32), "train"),
    ("prnmg.mnist", "mnist-cluttered/prnmg.mnist", dict(dataset="mnist-seg"), (2, 1, 64, 64), "train"),
    ("U-MG", "mnist-cluttered/unmg", dict(dataset="mnist-seg"), (2, 1, 64, 64), "train"),
    ("P-NMG isDropout", "cifar/pnmg", dict(isDropout=True, **PNMG_OPT), (8, 3, 32, 32), "train"),
    ("R-MG-34 quarter frozen", "ilsvrc/rnmg", dict(depth=34), (8, 3, 224, 224), "quarter-frozen"),
    ("R-MG-34 evaluate needInputGrad", "ilsvrc/rnmg", dict(depth=34), (2, 3, 224, 224), "evaluate"),
]


class Recorder:
    def __init__(self, log, real):
        self.log, self.real = log, real

    def call(self, name, *args):
        if name in ("mg_ctx_lane", "mg_ctx_event_record", "mg_ctx_event_wait"):
            self.log.append(f"{name} {int(args[0])}")
        else:
            self.log.append(name)

    def set_stream(self, stream):
        self.real.set_stream(stream)


def trace(B, torch, net, opt, shape, mode, lanes, bn_sync):
    os.environ["MGCONV_LANES"] = str(lanes)
    torch.manual_seed(7)
    m = B.load_net(net).createModel(B.Opt(nGPU=1, **opt))
    m.needInputGrad = mode == "evaluate"
    m.cuda()
    if mode == "evaluate":
        m.evaluate()
    elif mode == "quarter-frozen":
        bns = m.findModules("nn.SpatialBatchNormalization")
        for b in bns[:max(1, len(bns) // 4)]:
            b.evaluate()
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(11)).cuda()
    eng = m._get_engine(x)
    log = []
    eng.ctx = Recorder(log, eng.ctx)
    index = {id(mod): i for i, mod in enumerate(m.listModules())}
    eng.on_param_done = lambda mod: log.append(f"param_done {index[id(mod)]}")
    if bn_sync:
        eng.set_bn_sync(bn_sync)

    def section(title, fn):
        log.append(f"== {title}")
        return fn()

    out = section("forward", lambda: m.forward(x))
    go = torch.randn(*out.shape, generator=torch.Generator().manual_seed(12)).cuda()
    section("backward", lambda: m.backward(x, go))
    section("forward", lambda: m.forward(x))
    section("updateGradInput", lambda: m.updateGradInput(x, go))
    section("accGradParameters", lambda: m.accGradParameters(x, go, 0.5))
    section("accGradParameters", lambda: m.accGradParameters(x, go, 0.5))
    kept = eng.n_lanes
    eng.n_lanes = 1
    section("forward n_lanes=1", lambda: m.forward(x))
    section("backward n_lanes=1", lambda: m.backward(x, go))
    eng.n_lanes = kept
    section("forward", lambda: m.forward(x))
    section("backward", lambda: m.backward(x, go))
    return log


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pkg", default=os.path.join(ROOT, "multigrid-neural-architectures_b200"))
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    os.environ["MGCONV_AUTOTUNE"] = "0"
    os.environ.setdefault("MGCONV_LIB", os.path.join(ROOT, "multigrid-neural-architectures_b200", "mgconv", "libmgconv.so"))
    sys.path.insert(0, os.path.abspath(args.pkg))
    import torch
    from mgconv import builders as B
    with open(args.out, "w") as f:
        for name, net, opt, shape, mode in NETS:
            for lanes in (1, 3):
                for bn_sync in (0, 2):
                    log = trace(B, torch, net, opt, shape, mode, lanes, bn_sync)
                    f.write(f"### {name} lanes={lanes} bn_sync={bn_sync}: {len(log)} entries\n")
                    f.write("\n".join(log) + "\n")
                    print(f"{name} lanes={lanes} bn_sync={bn_sync}: {len(log)} entries", flush=True)


if __name__ == "__main__":
    main()
