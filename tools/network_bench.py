"""Whole-network timing of the REAL reference Network (oracle/_ref) on this GPU, unpatched vs rag_b200.network.install():
how much of a full forward / training step the hot path (and the rows next to it) is worth end to end.

    python tools/network_bench.py [--size 288x576] [--batch 4]

Five configurations, same weights and inputs: (a) the unmodified reference (PyTorch eager + cuDNN, TF32 on as by default),
(b) install() -- cost volume + disparity head through the hand-written kernels, (c) install(fuse_stem=True, upsample=True) --
additionally the first Matching-Net layer fused with the volume (never materialised, forward and backward) and the tail
(upsample_12/6, last_3_3d), (d) as (c) plus matching_convs=True -- the interior 3x3x3 ConvBR_3d layers on csrc/conv3d_cc.cu,
(e) as (d) plus pointwise_convs=True -- the pointwise 1x1x1 ConvBR_3d layers on csrc/conv3d_pw.cu.
Forward = eval() under no_grad (approaches/rag.py:408-441); training step = train() forward +
masked smooth-L1 + backward (approaches/rag.py:205-216, optimizer step excluded).  Prints one JSON line per configuration;
without the reference installed in oracle/_ref it prints one line saying the network was not measured."""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import refimport as R  # noqa: E402
from rag_b200 import network as N  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", default="288x576")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    H, W = (int(v) for v in a.size.split("x"))
    dev = torch.device("cuda:0")
    if not R.available():
        print(json.dumps({"note": "not measured: the unmodified reference is not installed in oracle/_ref"}), flush=True)
        return
    ref = R.import_reference()
    torch.manual_seed(0)
    net = ref.rag_model.Network(R.make_genotype(ref, 0), dev).to(dev)
    g = torch.Generator().manual_seed(1)
    left, right = torch.randn(a.batch, 3, H, W, generator=g).to(dev), torch.randn(a.batch, 3, H, W, generator=g).to(dev)
    gt = (torch.rand(a.batch, H, W, generator=g) * 150).to(dev)

    def timed(fn):
        fn(); fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.reps, torch.cuda.max_memory_allocated() / 2**30

    def fwd():
        with torch.no_grad():
            net.forward(left, right, 0, net.arch_init)

    def step():
        net.zero_grad(set_to_none=True)
        disp = net.forward(left, right, 0, net.arch_init)
        mask = (gt < 192) & (gt > 0)
        F.smooth_l1_loss(disp[mask], gt[mask]).backward()

    rows = []
    for name, kw in (("reference (unpatched)", None), ("install()", {}),
                     ("install(fuse_stem=True, upsample=True)", dict(operations_3d=ref.operations_3d, fuse_stem=True, upsample=True)),
                     ("install(fuse_stem=True, upsample=True, matching_convs=True)",
                      dict(operations_3d=ref.operations_3d, fuse_stem=True, upsample=True, matching_convs=True)),
                     ("install(fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True)",
                      dict(operations_3d=ref.operations_3d, fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True))):
        N.uninstall()
        if kw is not None:
            N.install(ref.rag_model, ref.mdenas_basicmodel, **kw)
        net.eval()
        f_ms, f_mem = timed(fwd)
        net.train()
        s_ms, s_mem = timed(step)
        rows.append({"config": name, "size": a.size, "batch": a.batch, "forward_ms": round(f_ms, 3), "forward_peak_GiB": round(f_mem, 2),
                     "train_step_ms": round(s_ms, 3), "train_peak_GiB": round(s_mem, 2)})
        print(json.dumps(rows[-1]), flush=True)
    N.uninstall()
    base = rows[0]
    for r in rows[1:]:
        print(json.dumps({"config": r["config"], "forward_speedup": round(base["forward_ms"] / r["forward_ms"], 2),
                          "train_step_speedup": round(base["train_step_ms"] / r["train_step_ms"], 2),
                          "train_peak_memory_ratio": round(r["train_peak_GiB"] / base["train_peak_GiB"], 2)}), flush=True)


if __name__ == "__main__":
    main()
