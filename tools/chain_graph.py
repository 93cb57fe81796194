"""GPU-side limit of the two-stream training schedule without host launch overhead (tuning tool): N steps of the volume chain
(cv_fwd, cv_bwd) on one stream and N steps of the head chain (head_fwd, head_bwd) on another, captured into ONE CUDA graph as
two independent chains, replayed.  Compares with the eager two-stream loop and the serial loop.
    python tools/chain_graph.py [--cfg 288x576 --batch 4 --n 20] [--cvf 3 --cvb 2]"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rag_b200 import functional as F_  # noqa: E402

CFGS = {"288x576": (96, 192, 64, 192), "480x960": (160, 320, 64, 192)}
ap = argparse.ArgumentParser()
ap.add_argument("--cfg", default="288x576")
ap.add_argument("--batch", type=int, default=4)
ap.add_argument("--n", type=int, default=20)
a = ap.parse_args()
hf, wf, df, md = CFGS[a.cfg]
b, c, dev = a.batch, 12, "cuda"
g = torch.Generator(device=dev).manual_seed(1)
x = torch.randn(b, c, hf, wf, device=dev, generator=g)
y = torch.randn(b, c, hf, wf, device=dev, generator=g)
cl = torch.randn(b, 1, df, hf, wf, device=dev, generator=g)
gd = torch.randn(b, 3 * hf, 3 * wf, device=dev, generator=g) * (torch.rand(b, 3 * hf, 3 * wf, device=dev, generator=g) < 0.3)
gc = torch.randn(b, 2 * c, df, hf, wf, device=dev, generator=g)
disp0, stats0 = F_.disp_head_forward(cl, md, True)
sA, sB = torch.cuda.Stream(), torch.cuda.Stream()
ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731


def chains(cvf, cvb, order):
    def A():
        F_.cost_volume_forward(x, y, df, variant=cvf)
        F_.cost_volume_backward(gc, c, variant=cvb)

    def B():
        d, s = F_.disp_head_forward(cl, md, True)
        F_.disp_head_backward(cl, gd, d, s, md)

    cur = torch.cuda.current_stream()
    side = torch.cuda.Stream()
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        A(); B()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr, stream=side):
        s0 = torch.cuda.current_stream()
        sA.wait_stream(s0); sB.wait_stream(s0)
        first, second = ((sA, A), (sB, B)) if order == "A" else ((sB, B), (sA, A))
        for st, fn in (first, second):
            with torch.cuda.stream(st):
                for _ in range(a.n):
                    fn()
        s0.wait_stream(sA); s0.wait_stream(sB)
    for _ in range(2):
        gr.replay()
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record()
    for _ in range(5):
        gr.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 5 / a.n


out = {"cfg": a.cfg, "batch": b, "n": a.n}
for cvf, cvb in ((3, 2), (1, 0), (3, 0)):
    for order in ("A", "B"):
        out[f"chains cv_fwd v{cvf} cv_bwd v{cvb} captured {order}-chain first: ms/step"] = round(chains(cvf, cvb, order), 4)
print(json.dumps(out, indent=1))
