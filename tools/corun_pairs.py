"""How the volume kernels and the head kernels behave when they share the GPU on two streams (tuning tool).

    python tools/corun_pairs.py [--cfg 288x576 --batch 4]

For each pair (cost-volume fwd || head fwd, cost-volume bwd || head bwd) and each volume-kernel variant / launch order:
the duration of each kernel alone, and -- launched together on two streams -- each kernel's own start->end span and the
span of the pair (CUDA events on both streams, L2 flushed before each repetition).
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rag_b200 import functional as F_  # noqa: E402

CFGS = {"288x576": (96, 192, 64, 192), "480x960": (160, 320, 64, 192)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", default="288x576")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    hf, wf, df, md = CFGS[a.cfg]
    b, c = a.batch, 12
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(b, c, hf, wf, device=dev, generator=g)
    y = torch.randn(b, c, hf, wf, device=dev, generator=g)
    cl = torch.randn(b, 1, df, hf, wf, device=dev, generator=g)
    gd = torch.randn(b, 3 * hf, 3 * wf, device=dev, generator=g) * (torch.rand(b, 3 * hf, 3 * wf, device=dev, generator=g) < 0.3)
    gc = torch.randn(b, 2 * c, df, hf, wf, device=dev, generator=g)
    disp, stats = F_.disp_head_forward(cl, md, True)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    sA, sB = torch.cuda.Stream(), torch.cuda.Stream()
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def alone(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(a.iters):
            flush.add_(1.0)
            torch.cuda.synchronize()
            e0, e1 = ev(), ev()
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    def pair(fa, fb, a_first=True):
        res = []
        for it in range(a.iters + 3):
            flush.add_(1.0)
            torch.cuda.synchronize()
            t0, a0, a1, b0, b1 = ev(), ev(), ev(), ev(), ev()
            t0.record()
            sA.wait_stream(torch.cuda.current_stream()); sB.wait_stream(torch.cuda.current_stream())
            def la():
                with torch.cuda.stream(sA):
                    a0.record(); fa(); a1.record()
            def lb():
                with torch.cuda.stream(sB):
                    b0.record(); fb(); b1.record()
            (la(), lb()) if a_first else (lb(), la())
            torch.cuda.synchronize()
            if it >= 3:
                res.append((a0.elapsed_time(a1), b0.elapsed_time(b1), max(t0.elapsed_time(a1), t0.elapsed_time(b1)) - min(t0.elapsed_time(a0), t0.elapsed_time(b0))))
        res.sort(key=lambda r: r[2])
        return res[len(res) // 2]

    out = {"cfg": a.cfg, "batch": b}
    hfw = lambda: F_.disp_head_forward(cl, md, True)           # noqa: E731
    hbw = lambda: F_.disp_head_backward(cl, gd, disp, stats, md)  # noqa: E731
    out["head_fwd_alone"] = round(alone(hfw), 4)
    out["head_bwd_alone"] = round(alone(hbw), 4)
    for v in (1, 3):
        f = lambda v=v: F_.cost_volume_forward(x, y, df, variant=v)  # noqa: E731
        out[f"cv_fwd_v{v}_alone"] = round(alone(f), 4)
        for first in (True, False):
            ra, rb, span = pair(f, hfw, first)
            out[f"cv_fwd_v{v}||head_fwd ({'cv' if first else 'head'} first)"] = {"cv": round(ra, 4), "head": round(rb, 4), "span": round(span, 4)}
    for v in (0, 2):
        f = lambda v=v: F_.cost_volume_backward(gc, c, variant=v)  # noqa: E731
        out[f"cv_bwd_v{v}_alone"] = round(alone(f), 4)
        for first in (True, False):
            ra, rb, span = pair(f, hbw, first)
            out[f"cv_bwd_v{v}||head_bwd ({'cv' if first else 'head'} first)"] = {"cv": round(ra, 4), "head": round(rb, 4), "span": round(span, 4)}
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
