"""The weight gradient of the interior ConvBR_3d layers in fp32 (csrc/conv3d_cc.cu), in TF32 on the tensor cores
(csrc/conv3d_cc_tf32.cu) and on cuDNN TF32, and a ConvBR3dFn training pass with ``matching_tf32`` alone and with
``matching_tf32_wgrad`` as well, on the GPU.

    python tools/matching_conv_tf32_wgrad_time.py [--reps 20] [--out profiles/r8_matching_conv_tf32_wgrad_times.jsonl]

The six shapes of DESIGN.md 5.10.1 (B=4 288x576 and B=8 480x960; Df = 64, level 6 halves D, H, W).  4 -> 4 has no TF32
weight gradient (its row times fp32 and cuDNN only).  Floors of the weight gradient: HBM, reading x and gz once, 4 (C + O)
bytes per voxel at 6460.5 GB/s (the B200's measured HBM copy peak, DESIGN.md 5); TF32, 2 * 27 * C * O FLOP per voxel at the
data sheet's dense 1125 TFLOP/s.  Method: CUDA events around each pass, a 256 MB buffer overwritten between passes (L2
flush, outside the events), median of --reps passes after 3 warm-up passes.  One JSON line per shape, with the card name,
power limit and SM clock read in the same run."""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rag_b200 import _cabi, matching_conv  # noqa: E402
from rag_b200.matching_conv import matching_forward  # noqa: E402
from tools.matching_conv_tf32_time import HBM_GBPS, ConvBR_3d, card  # noqa: E402

TF32_TFLOPS = 1125.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(64 * 2**20, dtype=torch.float32, device=dev)
    torch.backends.cudnn.allow_tf32 = True

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

    sizes = {"B=4 288x576": (4, 96, 192), "B=8 480x960": (8, 160, 320)}
    layers = [("stem3d1", 12, 12, 1), ("level-3 op", 4, 4, 1), ("level-6 op", 8, 8, 2)]
    out = open(a.out, "w") if a.out else None
    L = _cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    who = card()
    for size, (b, hf, wf) in sizes.items():
        for name, c, o, lv in layers:
            d, h, w = 64 // lv, hf // lv, wf // lv
            g = torch.Generator().manual_seed(0)
            x = torch.randn(b, c, d, h, w, generator=g).to(dev)
            gz = torch.randn(b, o, d, h, w, generator=g).to(dev)
            lay = ConvBR_3d(c, o).to(dev).train()
            xg = x.clone().requires_grad_(True)
            wshape = (o, c, 3, 3, 3)
            res = {}
            gw32, gwtf = torch.empty(wshape, device=dev), torch.empty(wshape, device=dev)
            ws32 = torch.empty(int(L.rag_conv3d_cc_bwd_workspace_bytes(b, c, o, d, h, w)) // 4, device=dev)
            res["ours_fp32_wgrad"] = timed(lambda: _cabi.check(L.rag_conv3d_cc_bwd(
                gz.data_ptr(), x.data_ptr(), None, None, gw32.data_ptr(), ws32.data_ptr(), b, c, o, d, h, w, st), "bwd"))
            nws = int(L.rag_conv3d_cc_tf32_bwd_weight_workspace_bytes(b, c, o, d, h, w)) // 4
            if nws:
                wstf = torch.empty(nws, device=dev)
                res["ours_tf32_wgrad"] = timed(lambda: _cabi.check(L.rag_conv3d_cc_tf32_bwd_weight(
                    gz.data_ptr(), x.data_ptr(), gwtf.data_ptr(), wstf.data_ptr(), b, c, o, d, h, w, st), "bwd_weight"))
            res["cudnn_tf32_wgrad"] = timed(lambda: torch.nn.grad.conv3d_weight(x, wshape, gz, padding=1))
            matching_conv.set_tf32(True)
            for tag, on in (("tf32", False), ("tf32_wgrad", True)):
                matching_conv.set_tf32_wgrad(on)
                res[f"ours_{tag}_train_fwd_bwd"] = timed(lambda: matching_forward(lay, xg).backward(gz))
            matching_conv.set_tf32(False)
            matching_conv.set_tf32_wgrad(False)
            vox = b * d * h * w
            hbm_ms = 4.0 * (c + o) * vox / (HBM_GBPS * 1e9) * 1e3
            flop_ms = 2.0 * 27 * c * o * vox / (TF32_TFLOPS * 1e12) * 1e3
            row = {"layer": name, "C": c, "O": o, "size": size, "shape": [b, c, d, h, w],
                   "wgrad_hbm_floor_ms": round(hbm_ms, 4), "wgrad_tf32_floor_ms": round(flop_ms, 4)}
            row.update({k: round(v, 4) for k, v in res.items()})
            if nws:
                row["tf32_wgrad_frac_of_floor"] = round(max(hbm_ms, flop_ms) / res["ours_tf32_wgrad"], 3)
                row["tf32_wgrad_speedup_vs_fp32"] = round(res["ours_fp32_wgrad"] / res["ours_tf32_wgrad"], 2)
                ref = torch.nn.grad.conv3d_weight(x.double(), wshape, gz.double(), padding=1)
                row["tf32_wgrad_maxnorm_rel_vs_fp64"] = float(f"{((gwtf.double() - ref).abs().max() / ref.abs().max()).item():.3e}")
                row["fp32_wgrad_maxnorm_rel_vs_fp64"] = float(f"{((gw32.double() - ref).abs().max() / ref.abs().max()).item():.3e}")
            row["card"] = who
            row["method"] = "CUDA events per pass, 256 MB L2 flush between passes, median of %d" % a.reps
            print(json.dumps(row), flush=True)
            if out:
                out.write(json.dumps(row) + "\n")
            del x, gz, xg, lay
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
