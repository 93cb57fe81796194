"""Where the Matching Net's time goes: every ConvBR_3d of the REAL reference Network (oracle/_ref) with its (C, O, kernel,
stride) and input shape, and the CUDA kernel time of one eval forward and one training step attributed to layer kinds.

    python tools/matching_profile.py [--size 288x576] [--batch 4] [--out profiles/r3_matching_profile.md]

The network is built as tools/network_bench.py builds it, unpatched (PyTorch eager + cuDNN, TF32 on as by default).
Forward hooks list the layers.  In a run of its own, torch.profiler records one eval forward and one training step; each
ConvBR_3d call is wrapped in a record_function range named by its (C, O, kernel, stride), so forward kernels are attributed
to those layer kinds; every kernel (forward and backward) is also attributed to the aten op that launched it (convolution,
its backward, batch_norm, relu, interpolate, cat, add, ...).  Without oracle/_ref the digest says so and nothing is measured."""
import argparse
import collections
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import refimport as R  # noqa: E402

OP_KINDS = [("convolution_backward", "conv backward"), ("cudnn_convolution", "conv forward"), ("convolution", "conv forward"),
            ("batch_norm_backward", "BatchNorm backward"), ("batch_norm", "BatchNorm"), ("threshold_backward", "ReLU backward"),
            ("relu", "ReLU"), ("upsample", "interpolate"), ("cat", "cat"), ("add", "add / sum"), ("sum", "add / sum")]


def kind_of(name):
    for key, kind in OP_KINDS:
        if key in name:
            return kind
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", default="288x576")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = [f"# Matching Net profile (tools/matching_profile.py --size {a.size} --batch {a.batch})", ""]
    if not R.available():
        lines.append("oracle/_ref (the unmodified reference) is not installed on this machine: nothing was measured. The per-layer "
                     "timings of profiles/r3_matching_conv_times.jsonl are the evidence for the (C, O) set.")
        text = "\n".join(lines) + "\n"
        print(text)
        if a.out:
            open(a.out, "w").write(text)
        return
    H, W = (int(v) for v in a.size.split("x"))
    dev = torch.device("cuda:0")
    ref = R.import_reference()
    torch.manual_seed(0)
    net = ref.rag_model.Network(R.make_genotype(ref, 0), dev).to(dev)
    g = torch.Generator().manual_seed(1)
    left, right = torch.randn(a.batch, 3, H, W, generator=g).to(dev), torch.randn(a.batch, 3, H, W, generator=g).to(dev)
    gt = (torch.rand(a.batch, H, W, generator=g) * 150).to(dev)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    lines += [f"Card: {q.strip().splitlines()[0] if q.strip() else torch.cuda.get_device_name()}", ""]

    convbr = ref.operations_3d.ConvBR_3d
    seen = collections.OrderedDict()
    names = {m: n for n, m in net.named_modules()}

    def key(m, x):
        c = m.conv
        return f"ConvBR_3d C={c.in_channels} O={c.out_channels} k={c.kernel_size[0]} s={c.stride[0]}"

    def listing(m, inp, out):
        x = inp[0]
        seen.setdefault(names[m], (key(m, x), tuple(x.shape) if torch.is_tensor(x) else type(x).__name__))

    hooks = [m.register_forward_hook(listing) for m in net.modules() if isinstance(m, convbr)]
    net.eval()
    with torch.no_grad():
        net.forward(left, right, 0, net.arch_init)
    for h in hooks:
        h.remove()
    lines += ["## Every ConvBR_3d of one forward", "", "| module | layer | input shape |", "|---|---|---|"]
    lines += [f"| {n} | {k} | {list(s) if isinstance(s, tuple) else s} |" for n, (k, s) in seen.items()]
    lines.append("")

    ranges = {}

    def pre(m, inp):
        r = torch.profiler.record_function(key(m, inp[0]))
        r.__enter__()
        ranges[id(m)] = r

    def post(m, inp, out):
        ranges.pop(id(m)).__exit__(None, None, None)

    hooks = [m.register_forward_pre_hook(pre) for m in net.modules() if isinstance(m, convbr)]
    hooks += [m.register_forward_hook(post) for m in net.modules() if isinstance(m, convbr)]

    def fwd():
        with torch.no_grad():
            net.forward(left, right, 0, net.arch_init)

    def step():
        net.zero_grad(set_to_none=True)
        disp = net.forward(left, right, 0, net.arch_init)
        mask = (gt < 192) & (gt > 0)
        F.smooth_l1_loss(disp[mask], gt[mask]).backward()

    for title, mode, fn in (("eval forward", "eval", fwd), ("training step", "train", step)):
        getattr(net, mode)()
        fn(); fn()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA, torch.profiler.ProfilerActivity.CPU]) as prof:
            fn()
            torch.cuda.synchronize()
        by_layer, by_kind = collections.Counter(), collections.Counter()
        total = 0.0
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if e.key.startswith("ConvBR_3d"):
                by_layer[e.key] += t / 1e3
        # kernel time per aten op: self device time of the leaf ops (no double counting through parents)
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = e.self_cuda_time_total
            if t > 0:
                by_kind[kind_of(e.key)] += t / 1e3
                total += t / 1e3
        lines += [f"## {title}: {total:.2f} ms of CUDA kernel time", "", "| op kind | ms | share |", "|---|---|---|"]
        lines += [f"| {k} | {v:.3f} | {100 * v / total:.1f} % |" for k, v in by_kind.most_common()]
        lines += ["", "| ConvBR_3d kind (forward kernels inside its range, all instances) | ms |", "|---|---|"]
        lines += [f"| {k} | {v:.3f} |" for k, v in by_layer.most_common()]
        lines.append("")
    for h in hooks:
        h.remove()
    text = "\n".join(lines) + "\n"
    print(text)
    if a.out:
        open(a.out, "w").write(text)


if __name__ == "__main__":
    main()
