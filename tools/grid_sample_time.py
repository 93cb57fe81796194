"""Timing of the drop-in F.grid_sample (rag_b200/grid_sample.py, csrc/grid_sample.cu) against ATen, on the GPU.

    python tools/grid_sample_time.py [--reps 20] [--out profiles/r6_grid_sample_times.jsonl]

Shapes: image warps [4,3,288,576] and [8,3,480,960], feature warps [4,12,96,192] and [4,32,96,192], each with a stereo grid
(x shifted left by a random disparity of up to a quarter of the width, y = the row; align_corners=True, zeros padding) and a
random grid in [-1.1, 1.1]^2.  The output has the input's size.
  ours:  forward through grid_sample.grid_sample, backward through autograd (input and grid gradients, fixed order);
  F.grid_sample: forward and backward, deterministic mode off.  For this call (zeros padding, align_corners=True) torch sends
         CUDA tensors to cuDNN's sampler;
  ATen:  ATen's own grid_sampler_2d kernel (torch.grid_sampler_2d), the kernels' contract, whose input gradient scatters with
         atomicAdd;
  ours under the mode: forward + backward under torch.use_deterministic_algorithms(True), where ATen's backward raises.
Method: CUDA events around each pass, a 256 MB buffer overwritten between passes (L2 flush, outside the events), median of
--reps passes after 3 warm-up passes.  HBM floor from bytes at 6460.5 GB/s (the copy bandwidth measured on a B200, DESIGN.md
5): the forward reads the input and the grid and writes the output once; the backward reads gout, the input and the grid and
writes gin and ggrid once.  One JSON line per case, with the card name, power limit and SM clock read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rag_b200.grid_sample import grid_sample, routes  # noqa: E402

HBM_BPS = 6460.5e9


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def make_grid(kind, n, h, w, g):
    if kind == "random":
        return torch.rand(n, h, w, 2, generator=g) * 2.2 - 1.1
    xs = torch.arange(w).view(1, 1, w).float() - torch.rand(n, h, w, generator=g) * w / 4
    ys = torch.arange(h).view(1, h, 1).float().expand(n, h, w)
    return torch.stack([2 * xs / (w - 1) - 1, 2 * ys / (h - 1) - 1], -1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("grid_sample_time.py measures on a GPU; none is visible")
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
    shapes = {"image B=4 288x576": (4, 3, 288, 576), "image B=8 480x960": (8, 3, 480, 960),
              "feature C=12": (4, 12, 96, 192), "feature C=32": (4, 32, 96, 192)}
    for name, shape in shapes.items():
        for kind in ("stereo", "random"):
            g = torch.Generator().manual_seed(0)
            n, c, h, w = shape
            x = torch.randn(shape, generator=g).to(dev)
            grid = make_grid(kind, n, h, w, g).to(dev)
            go = torch.randn(shape, generator=g).to(dev)
            kw = dict(mode="bilinear", padding_mode="zeros", align_corners=True)
            assert routes(x, grid, **kw)
            xg, gg = x.clone().requires_grad_(True), grid.clone().requires_grad_(True)
            res = {}
            with torch.no_grad():
                res["ours_fwd"] = timed(lambda: grid_sample(x, grid, **kw))
                res["aten_fwd"] = timed(lambda: torch.grid_sampler_2d(x, grid, 0, 0, True))
                res["f_grid_sample_fwd"] = timed(lambda: F.grid_sample(x, grid, **kw))
            ours = grid_sample(xg, gg, **kw)
            aten = torch.grid_sampler_2d(xg, gg, 0, 0, True)
            fgs = F.grid_sample(xg, gg, **kw)
            res["ours_bwd"] = timed(lambda: torch.autograd.grad(ours, (xg, gg), go, retain_graph=True))
            res["aten_bwd"] = timed(lambda: torch.autograd.grad(aten, (xg, gg), go, retain_graph=True))
            res["f_grid_sample_bwd"] = timed(lambda: torch.autograd.grad(fgs, (xg, gg), go, retain_graph=True))
            del fgs
            go_o = torch.autograd.grad(ours, (xg, gg), go, retain_graph=True)
            go_a = torch.autograd.grad(aten, (xg, gg), go, retain_graph=True)
            err = {"fwd": ((ours - aten).abs().max() / aten.abs().max()).item(),
                   "gin": ((go_o[0] - go_a[0]).abs().max() / go_a[0].abs().max()).item(),
                   "ggrid": ((go_o[1] - go_a[1]).abs().max() / go_a[1].abs().max()).item()}
            fwd_bits = bool(torch.equal(ours, aten))
            del ours, aten, go_o, go_a
            torch.use_deterministic_algorithms(True)
            try:
                res["ours_deterministic_fwd_bwd"] = timed(lambda: torch.autograd.grad(grid_sample(xg, gg, **kw), (xg, gg), go))
            finally:
                torch.use_deterministic_algorithms(False)
            floor_fwd = 4.0 * (x.numel() + grid.numel() + go.numel()) / HBM_BPS * 1e3
            floor_bwd = 4.0 * (go.numel() + 2 * x.numel() + 2 * grid.numel()) / HBM_BPS * 1e3
            row = {"case": name, "grid": kind, "shape": list(shape), "hbm_floor_fwd_ms": round(floor_fwd, 4),
                   "hbm_floor_bwd_ms": round(floor_bwd, 4)}
            row.update({k: round(v, 4) for k, v in res.items()})
            row["fwd_speedup_vs_aten"] = round(res["aten_fwd"] / res["ours_fwd"], 2)
            row["bwd_speedup_vs_aten"] = round(res["aten_bwd"] / res["ours_bwd"], 2)
            row["fwd_frac_of_floor"] = round(floor_fwd / res["ours_fwd"], 3)
            row["bwd_frac_of_floor"] = round(floor_bwd / res["ours_bwd"], 3)
            row["fwd_bit_identical_to_aten"] = fwd_bits
            row["max_rel_err_vs_aten"] = {k: float(f"{v:.2e}") for k, v in err.items()}
            row["card"] = who
            row["method"] = "CUDA events per pass, 256 MB L2 flush between passes, median of %d" % a.reps
            print(json.dumps(row), flush=True)
            if out:
                out.write(json.dumps(row) + "\n")
            del x, grid, go, xg, gg
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
