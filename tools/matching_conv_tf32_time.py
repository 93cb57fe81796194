"""The interior ConvBR_3d layers in fp32 (csrc/conv3d_cc.cu), in TF32 on the tensor cores (csrc/conv3d_cc_tf32.cu) and on
cuDNN TF32, on the GPU.

    python tools/matching_conv_tf32_time.py [--reps 20] [--out profiles/r7_matching_conv_tf32_times.jsonl]

The shapes of DESIGN.md 5.10 for the three routed pairs (B=4 288x576 and B=8 480x960; Df = 64, level 6 halves D, H, W).
Per shape: the eval forward (conv + folded BatchNorm + ReLU) and the training forward + backward through ``matching_forward``
with ``matching_tf32`` off and on, the mirror ConvBR_3d on cuDNN with TF32 on, and the two TF32 kernels alone.  The TF32
forward kernel's HBM floor is reading x and writing out once, 4 (C + O) bytes per voxel, at 6460.5 GB/s (the B200's
measured HBM copy peak, DESIGN.md 5).  Method: CUDA events around each pass, a 256 MB buffer overwritten between passes
(L2 flush, outside the events), median of --reps passes after 3 warm-up passes.  One JSON line per shape, with the card name,
power limit and SM clock read in the same run."""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rag_b200 import _cabi, matching_conv  # noqa: E402
from rag_b200.matching_conv import conv3d_cc_forward, matching_forward  # noqa: E402

HBM_GBPS = 6460.5


class ConvBR_3d(nn.Module):
    def __init__(self, c, o):
        super().__init__()
        self.relu, self.use_bn = True, True
        self.conv = nn.Conv3d(c, o, 3, stride=1, padding=1, bias=False)
        self.bn = nn.BatchNorm3d(o)

    def forward(self, x):
        return F.relu(self.bn(self.conv(x)), inplace=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


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
    for size, (b, hf, wf) in sizes.items():
        for name, c, o, lv in layers:
            d, h, w = 64 // lv, hf // lv, wf // lv
            g = torch.Generator().manual_seed(0)
            x = torch.randn(b, c, d, h, w, generator=g).to(dev)
            gout = torch.randn(b, o, d, h, w, generator=g).to(dev)
            lay = ConvBR_3d(c, o).to(dev)
            xg = x.clone().requires_grad_(True)
            res = {}
            for tag, on in (("fp32", False), ("tf32", True)):
                matching_conv.set_tf32(on)
                lay.eval()
                with torch.no_grad():
                    res[f"ours_{tag}_eval_fwd"] = timed(lambda: matching_forward(lay, x))
                lay.train()
                res[f"ours_{tag}_train_fwd_bwd"] = timed(lambda: matching_forward(lay, xg).backward(gout))
            matching_conv.set_tf32(False)
            wt = lay.conv.weight.detach()
            res["ours_fp32_conv_fwd_kernel"] = timed(lambda: conv3d_cc_forward(x, wt))
            res["ours_tf32_conv_fwd_kernel"] = timed(lambda: conv3d_cc_forward(x, wt, tf32=True))
            gin = torch.empty_like(x)
            res["ours_tf32_data_grad_kernel"] = timed(lambda: _cabi.check(L.rag_conv3d_cc_tf32_bwd_data(gout.data_ptr(), wt.data_ptr(), gin.data_ptr(), b, c, o, d, h, w, st), "bwd_data"))
            ref = copy.deepcopy(lay)
            ref.eval()
            with torch.no_grad():
                res["cudnn_tf32_eval_fwd"] = timed(lambda: ref(x))
            ref.train()
            res["cudnn_tf32_train_fwd_bwd"] = timed(lambda: ref(xg).backward(gout))
            # outputs of the two kernels on the same inputs: TF32 against fp32
            with torch.no_grad():
                z32, ztf = conv3d_cc_forward(x, wt), conv3d_cc_forward(x, wt, tf32=True)
                tf32_vs_fp32 = ((ztf - z32).abs().max() / z32.abs().max()).item()
            vox = b * d * h * w
            hbm_ms = 4.0 * (c + o) * vox / (HBM_GBPS * 1e9) * 1e3
            row = {"layer": name, "C": c, "O": o, "size": size, "shape": [b, c, d, h, w], "hbm_floor_ms": round(hbm_ms, 4)}
            row.update({k: round(v, 4) for k, v in res.items()})
            row["tf32_fwd_kernel_frac_of_hbm_floor"] = round(hbm_ms / res["ours_tf32_conv_fwd_kernel"], 3)
            row["tf32_fwd_kernel_speedup_vs_fp32"] = round(res["ours_fp32_conv_fwd_kernel"] / res["ours_tf32_conv_fwd_kernel"], 2)
            row["tf32_vs_fp32_maxnorm_rel"] = float(f"{tf32_vs_fp32:.3e}")
            row["card"] = card()
            row["method"] = "CUDA events per pass, 256 MB L2 flush between passes, median of %d" % a.reps
            print(json.dumps(row), flush=True)
            if out:
                out.write(json.dumps(row) + "\n")
            del x, gout, xg, gin, lay, ref
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
