"""Timing of the cells' resampling on the drop-in F.interpolate (rag_b200/resample.py, csrc/trilinear.cu) against ATen, on the GPU.

    python tools/resample_time.py [--reps 20] [--out profiles/r5_resample_times.jsonl]

Shapes are the cells' resamples at B=4 288x576 and B=8 480x960, with levels 3 / 6 / 12 at 1/3, 1/6, 1/12 of the image and
D = 64 / 32 / 16 (maxdisp 192).  The channel counts 12 / 24 / 48 at levels 3 / 6 / 12 are inferred (DESIGN.md 5.10), not
read from the reference: trilinear, align_corners=True, 3 -> 6, 3 -> 12, 6 -> 12 and 12 -> 6.  The 2-D rows are indicative
Feature-Net resamples (bilinear, align_corners=True, 32 channels) between its levels 3, 6 and 12.
  ours:  forward through resample.interpolate, and backward through autograd (the fixed-order gather);
  ATen:  F.interpolate forward and backward, deterministic mode off (its backward scatters with atomicAdd);
  ATen deterministic: forward + backward under torch.use_deterministic_algorithms(True), where F.interpolate takes
         torch's decomposition (gathers, lerps, an index_put_ backward) -- what the mode costs without the kernels.
Method: CUDA events around each pass, a 256 MB buffer overwritten between passes (L2 flush, outside the events), median of
--reps passes after 3 warm-up passes.  HBM floors from bytes at 6460.5 GB/s (the copy bandwidth measured on a B200,
DESIGN.md 5): each direction reads one side and writes the other once, 4 * (in + out elements) bytes.  A down-sampling
forward reads only the input rows it references, so there that floor is not a bound (fractions above 1).  One JSON line per
case, with the card name, power limit and SM clock read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rag_b200.resample import interpolate, plan  # noqa: E402

HBM_BPS = 6460.5e9


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def cases():
    out = []
    for size, (b, h3, w3) in {"B=4 288x576": (4, 96, 192), "B=8 480x960": (8, 160, 320)}.items():
        lv = {3: (64, h3, w3), 6: (32, h3 // 2, w3 // 2), 12: (16, h3 // 4, w3 // 4)}
        ch = {3: 12, 6: 24, 12: 48}
        for a, z in ((3, 6), (3, 12), (6, 12), (12, 6)):
            out.append((f"{a}->{z}", size, "trilinear", (b, ch[a]) + lv[a], lv[z]))
        for a, z in ((3, 6), (6, 12), (12, 6), (6, 3)):
            out.append((f"2-D {a}->{z} (indicative)", size, "bilinear", (b, 32) + lv[a][1:], lv[z][1:]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("resample_time.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    flush = torch.empty(64 * 2**20, dtype=torch.float32, device=dev)

    def timed(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(a.reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return statistics.median(ts)

    out = open(a.out, "w") if a.out else None
    who = card()
    for name, size, mode, shape, osize in cases():
        g = torch.Generator().manual_seed(0)
        x = torch.randn(shape, generator=g).to(dev)
        go = torch.randn(shape[:2] + tuple(osize), generator=g).to(dev)
        xg = x.clone().requires_grad_(True)
        kw = dict(mode=mode, align_corners=True)
        routed = plan(x, osize, **kw) is not None
        res = {}
        with torch.no_grad():
            res["ours_fwd"] = timed(lambda: interpolate(x, osize, **kw))
            res["aten_fwd"] = timed(lambda: F.interpolate(x, osize, **kw))
        ours = interpolate(xg, osize, **kw)
        aten = F.interpolate(xg, osize, **kw)
        res["ours_bwd"] = timed(lambda: torch.autograd.grad(ours, xg, go, retain_graph=True))
        res["aten_bwd"] = timed(lambda: torch.autograd.grad(aten, xg, go, retain_graph=True))
        # agreement with ATen at the timed size
        gi_o = torch.autograd.grad(ours, xg, go, retain_graph=True)[0]
        gi_a = torch.autograd.grad(aten, xg, go, retain_graph=True)[0]
        err_bwd = ((gi_o - gi_a).abs().max() / gi_a.abs().max()).item()
        err_fwd = ((ours.detach() - aten.detach()).abs().max() / aten.detach().abs().max()).item()
        del ours, aten, gi_o, gi_a
        torch.use_deterministic_algorithms(True)
        try:
            res["aten_deterministic_fwd_bwd"] = timed(lambda: torch.autograd.grad(F.interpolate(xg, osize, **kw), xg, go))
        finally:
            torch.use_deterministic_algorithms(False)
        floor = 4.0 * (x.numel() + go.numel()) / HBM_BPS * 1e3
        row = {"case": name, "size": size, "mode": mode, "shape": list(shape), "out": list(osize), "hbm_floor_ms": round(floor, 4)}
        row.update({k: round(v, 4) for k, v in res.items()})
        row["fwd_frac_of_floor"] = round(floor / res["ours_fwd"], 3)
        row["bwd_frac_of_floor"] = round(floor / res["ours_bwd"], 3)
        row["fwd_speedup_vs_aten"] = round(res["aten_fwd"] / res["ours_fwd"], 2)
        row["bwd_speedup_vs_aten"] = round(res["aten_bwd"] / res["ours_bwd"], 2)
        row["fwd_bwd_speedup_vs_aten_deterministic"] = round(res["aten_deterministic_fwd_bwd"] / (res["ours_fwd"] + res["ours_bwd"]), 2)
        row["at_least_as_fast_as_aten"] = bool(res["ours_fwd"] <= res["aten_fwd"] and res["ours_bwd"] <= res["aten_bwd"])
        row["max_rel_err_vs_aten"] = {"fwd": float(f"{err_fwd:.2e}"), "bwd": float(f"{err_bwd:.2e}")}
        row["routed_to_kernels"] = bool(routed)
        row["card"] = who
        row["method"] = "CUDA events per pass, 256 MB L2 flush between passes, median of %d" % a.reps
        print(json.dumps(row), flush=True)
        if out:
            out.write(json.dumps(row) + "\n")
        del x, go, xg
        torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
