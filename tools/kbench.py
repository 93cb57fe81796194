"""Per-kernel A/B timing of librag_b200 variants (CUDA events, L2 flushed between iterations).

    python tools/kbench.py [--cfg 288x576|480x960|384x1248|384x1248m288] [--batch B] [--iters N]

Prints one JSON line per (kernel, variant): time, algorithmic GB/s and fraction of the measured HBM
peak (MEASURED_PEAKS.json).  Tuning tool only; bench.py is the contract benchmark.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rag_b200 import functional as F_  # noqa: E402

CFGS = {
    "288x576": (96, 192, 64, 192),
    "480x960": (160, 320, 64, 192),
    "384x1248": (128, 416, 64, 192),
    "384x1248m288": (128, 416, 96, 288),
}


def peak():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        return 6650.0


def timeit(fn, iters, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.add_(1.0)  # > L2: evicts the previous iteration's lines
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", default="480x960")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--only", default="")
    ap.add_argument("--sigma", type=float, default=1.0, help="scale of the synthetic matching cost (peaked distributions: 20+)")
    a = ap.parse_args()
    hf, wf, df, md = CFGS[a.cfg]
    b, c = a.batch, 12
    pk = peak()
    dev = "cuda"
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    g = torch.Generator(device=dev).manual_seed(1234)
    x = torch.randn(b, c, hf, wf, device=dev, generator=g)
    y = torch.randn(b, c, hf, wf, device=dev, generator=g)
    cost_lr = torch.randn(b, 1, df, hf, wf, device=dev, generator=g) * a.sigma
    gd = torch.randn(b, 3 * hf, 3 * wf, device=dev, generator=g) * (torch.rand(b, 3 * hf, 3 * wf, device=dev, generator=g) < 0.3)
    vol_bytes = 4 * (2 * c * hf * wf + 2 * c * df * hf * wf) * b
    hf_bytes = 4 * (df * hf * wf + 9 * hf * wf) * b
    hb_bytes = 4 * (2 * df * hf * wf + 9 * hf * wf) * b

    def report(name, variant, med, best, nbytes):
        print(json.dumps({"kernel": name, "variant": variant, "cfg": a.cfg, "batch": b, "ms_median": round(med, 4),
                          "ms_best": round(best, 4), "alg_GBps": round(nbytes / med / 1e6, 1),
                          "frac_of_measured_hbm": round(nbytes / med / 1e6 / pk, 4),
                          "us_per_pair": round(med * 1e3 / b, 2)}), flush=True)

    def want(k):
        return not a.only or k in a.only.split(",")

    if want("cv_fwd"):
        for v in (0, 1, 3):
            med, best = timeit(lambda: F_.cost_volume_forward(x, y, df, variant=v), a.iters, flush)
            report("cv_fwd", v, med, best, vol_bytes)
        # torch baseline for scale: a plain device copy of the same number of bytes
        src = torch.empty(vol_bytes // 8, device=dev)
        dst = torch.empty_like(src)
        med, best = timeit(lambda: dst.copy_(src), a.iters, flush)
        report("torch_copy_same_bytes(r+w)", -1, med, best, vol_bytes)
        del src, dst
        dst = torch.empty(vol_bytes // 4, device=dev)
        med, best = timeit(lambda: dst.fill_(1.0), a.iters, flush)
        report("torch_fill_same_bytes(w)", -1, med, best, vol_bytes)
        del dst
    if want("cv_bwd"):
        gc = torch.randn(b, 2 * c, df, hf, wf, device=dev, generator=g)
        for v in (0, 1, 2):
            med, best = timeit(lambda: F_.cost_volume_backward(gc, c, variant=v), a.iters, flush)
            report("cv_bwd", v, med, best, vol_bytes)
        med, best = timeit(lambda: gc.sum(), a.iters, flush)
        report("torch_sum_same_bytes(r)", -1, med, best, vol_bytes)
        del gc
    if want("cv_stem"):
        from rag_b200.fused_stem import cv_stem_forward
        wgt = torch.randn(12, 24, 3, 3, 3, device=dev, generator=g) * 0.05
        sc = torch.rand(12, device=dev, generator=g) + 0.5
        sh = torch.randn(12, device=dev, generator=g)
        out_bytes = 4 * (12 * df * hf * wf + 2 * c * hf * wf) * b
        for v in (2, 1):
            med, best = timeit(lambda: cv_stem_forward(x, y, wgt, sc, sh, True, md, variant=v), a.iters, flush)
            report("cv_stem_fused(conv+bn+relu)", v, med, best, out_bytes)
        conv = torch.nn.Conv3d(24, 12, 3, padding=1, bias=False).to(dev)
        bn = torch.nn.BatchNorm3d(12).to(dev).eval()
        with torch.no_grad():
            for tf32 in (True, False):
                torch.backends.cudnn.allow_tf32 = tf32
                med, best = timeit(lambda: torch.relu_(bn(conv(F_.cost_volume_forward(x, y, df)))), 3, flush)
                report("cost_volume+cudnn_conv3d_bn_relu(tf32=%s)" % tf32, -1, med, best, out_bytes)
            torch.backends.cudnn.allow_tf32 = True
    if want("last_conv"):
        from rag_b200.last_conv import conv3d_c1_forward
        feat = torch.randn(b, 12, df, hf, wf, device=dev, generator=g)
        wl = torch.randn(1, 12, 3, 3, 3, device=dev, generator=g) * 0.1
        lc_bytes = 4 * (12 + 1) * df * hf * wf * b
        med, best = timeit(lambda: conv3d_c1_forward(feat, wl), a.iters, flush)
        report("last_3_3d conv (12->1, fp32)", 0, med, best, lc_bytes)
        conv = torch.nn.Conv3d(12, 1, 3, padding=1, bias=False).to(dev)
        with torch.no_grad():
            for tf32 in (True, False):
                torch.backends.cudnn.allow_tf32 = tf32
                med, best = timeit(lambda: conv(feat), 3, flush)
                report("cudnn_conv3d_12to1(tf32=%s)" % tf32, -1, med, best, lc_bytes)
            torch.backends.cudnn.allow_tf32 = True
        del feat
    if want("head_fwd"):
        for v in (2, 1):
            try:
                med, best = timeit(lambda: F_.disp_head_forward(cost_lr, md, True, variant=v), a.iters, flush)
                report("head_fwd", v, med, best, hf_bytes)
            except RuntimeError as e:
                print("head_fwd variant", v, "skipped:", e)
    if want("head_bwd"):
        disp, stats = F_.disp_head_forward(cost_lr, md, True)
        for v in (1, 2, 0):
            try:
                it = a.iters if v >= 1 else 2
                med, best = timeit(lambda: F_.disp_head_backward(cost_lr, gd, disp, stats, md, variant=v), it, flush)
                report("head_bwd", v, med, best, hb_bytes)
            except RuntimeError as e:
                print("head_bwd variant", v, "skipped:", e)


if __name__ == "__main__":
    main()
