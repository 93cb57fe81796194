"""Schedules of the two-stream step (tuning tool): launch-order sharing vs co-resident persistent grids.

    python tools/coresident.py [--cfg 288x576 --batch 4] [--steps 100]

1. The new kernel variants give the same bits as the defaults (torch.equal).
2. Each kernel alone, default vs variant (CUDA events, median of steady-state launches, L2 kept cold by the volume).
3. The overlapped training step (cv_fwd, cv_bwd on one stream; head_fwd, head_bwd on the other; free-running, K steps in
   flight) and the overlapped inference step for every schedule in rag_b200.pipeline.SCHEDULES plus mixes.
"""
import argparse
import itertools
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rag_b200 import functional as F_  # noqa: E402
from rag_b200 import pipeline as P_  # noqa: E402

CFGS = {"288x576": (96, 192, 64, 192), "480x960": (160, 320, 64, 192), "384x1248": (128, 416, 64, 192)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cfg", default="288x576")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--full", action="store_true", help="also sweep mixed variant sets")
    ap.add_argument("--infer-only", action="store_true", help="sweep the inference step only (volume forward x head forward variants)")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--cvb", default="3", help="cost-volume backward variants to A/B (beside the default and RAG_CV_BWD_SHARED)")
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
    out = {"cfg": a.cfg, "batch": b}
    cvbs = tuple(int(v) for v in a.cvb.split(",") if v)

    # ---- 1. parity of the variants ----
    disp, stats = F_.disp_head_forward(cl, md, True)
    d4, s4 = F_.disp_head_forward(cl, md, True, variant=P_.HEAD_FWD_SHARED)
    g1 = F_.disp_head_backward(cl, gd, disp, stats, md)
    g3 = F_.disp_head_backward(cl, gd, disp, stats, md, variant=P_.HEAD_BWD_SHARED)
    cv = F_.cost_volume_forward(x, y, df)
    cv5 = F_.cost_volume_forward(x, y, df, variant=P_.CV_FWD_SLIM)
    gx, gy = F_.cost_volume_backward(gc, c)
    cvb = {}
    for v in cvbs:
        gx3, gy3 = F_.cost_volume_backward(gc, c, variant=v)
        cvb[v] = bool(torch.equal(gx, gx3) and torch.equal(gy, gy3))
    out["parity"] = {"head_fwd": bool(torch.equal(disp, d4) and torch.equal(stats, s4)), "head_bwd": bool(torch.equal(g1, g3)),
                     "cv_fwd": bool(torch.equal(cv, cv5)), "cv_bwd": cvb}
    del cv, cv5, d4, s4, g3, gx3, gy3
    print(json.dumps(out), flush=True)

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def alone(fn, n=30):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return round(e0.elapsed_time(e1) / n, 4)

    # ---- 2. each kernel alone (back-to-back launches; the volume kernels' own traffic keeps everything cold) ----
    k = {}
    for v in (None, P_.CV_FWD_SHARED, P_.CV_FWD_SLIM):
        k[f"cv_fwd v{v}"] = alone(lambda v=v: F_.cost_volume_forward(x, y, df, variant=v))
    for v in (None, P_.CV_BWD_SHARED) + cvbs:
        k[f"cv_bwd v{v}"] = alone(lambda v=v: F_.cost_volume_backward(gc, c, variant=v))
    for v in (None, P_.HEAD_FWD_SHARED):
        k[f"head_fwd v{v}"] = alone(lambda v=v: F_.disp_head_forward(cl, md, True, variant=v))
    for v in (None, P_.HEAD_BWD_SHARED):
        k[f"head_bwd v{v}"] = alone(lambda v=v: F_.disp_head_backward(cl, gd, disp, stats, md, variant=v))
    out["alone_ms"] = k
    print(json.dumps({"alone_ms": k}), flush=True)

    # ---- 3. overlapped steps ----
    def timed(path, step, K):
        for _ in range(10):
            o = step()
        path.join()
        torch.cuda.synchronize()
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(K):
            o = step()
        path.join()
        e1.record()
        torch.cuda.synchronize()
        del o
        return round(e0.elapsed_time(e1) / K, 4)

    sets = dict(P_.SCHEDULES)
    if a.infer_only:
        sets = {f"cf{vcf} hf{vhf}": (vcf, vhf, None, None) for vcf in (P_.CV_FWD_SHARED, P_.CV_FWD_SLIM) for vhf in (None, P_.HEAD_FWD_SHARED)}
    elif a.full:
        for vcf, vhf, vcb, vhb in itertools.product((P_.CV_FWD_SLIM,), (None, P_.HEAD_FWD_SHARED),
                                                    (None,) + cvbs, (None, P_.HEAD_BWD_SHARED)):
            sets[f"cf{vcf} hf{vhf} cb{vcb} hb{vhb}"] = (vcf, vhf, vcb, vhb)
    res_t, res_i = {}, {}
    for name, vs in sets.items():
        tp = P_.OverlappedTrainPath(md, dev, schedule=vs)
        res_t[name] = [] if a.infer_only else [timed(tp, lambda: tp.step(x, y, cl, gc, gd), a.steps) for _ in range(a.reps)]
        ip = P_.OverlappedPath(md, dev, schedule=vs)
        res_i[name] = [timed(ip, lambda: ip.step(x, y, cl), a.steps) for _ in range(a.reps)]
        print(json.dumps({"schedule": name, "train_ms": res_t[name], "infer_ms": res_i[name]}), flush=True)
    out["train_step_ms"] = res_t
    out["infer_step_ms"] = res_i
    print(json.dumps(out))


if __name__ == "__main__":
    main()
