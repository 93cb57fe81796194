"""Per-layer timing of the interior ConvBR_3d layers (csrc/conv3d_cc.cu) against cuDNN, on the GPU.

    python tools/matching_conv_time.py [--reps 20] [--level12] [--out profiles/r3_matching_conv_times.jsonl]

For every routed (C, O) at its level shape of B=4 288x576 and B=8 480x960 (Hf, Wf = H/3, W/3, Df = 64; level 6 / 12 halve /
quarter all three):
  ours:  eval forward (folded BatchNorm + ReLU, one kernel); training forward (conv + moments + finalize + normalise, with
         autograd); backward (gz, data gradient, weight gradient); and the three convolution kernels alone;
  cuDNN: the mirror ConvBR_3d through PyTorch eager, eval forward and train forward + backward, TF32 on (the reference's
         default) and off.
Method: CUDA events around each pass, a 256 MB buffer overwritten between passes (L2 flush, outside the events), median of
--reps passes after 3 warm-up passes.  FLOP = 2*B*O*D*H*W*C*27 per convolution pass; floor = FLOP / 72 TFLOP/s (FP32 issue).
One JSON line per case, with the card name, power limit and SM clock read in the same run.  --level12 adds the level-12
16 -> 16 op, which is not compiled (it lost to cuDNN TF32 at these shapes, DESIGN.md 5.10): its rows hold cuDNN's times only."""
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
from rag_b200 import _cabi  # noqa: E402
from rag_b200.matching_conv import PAIRS, conv3d_cc_forward, matching_forward  # noqa: E402

FP32_PEAK = 72e12


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
    ap.add_argument("--level12", action="store_true", help="also time cuDNN on the level-12 16 -> 16 op (not compiled here)")
    a = ap.parse_args()
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

    sizes = {"B=4 288x576": (4, 96, 192), "B=8 480x960": (8, 160, 320)}
    layers = [("stem3d1", 12, 12, 1), ("level-3 op", 4, 4, 1), ("level-6 op", 8, 8, 2)] + ([("level-12 op", 16, 16, 4)] if a.level12 else [])
    out = open(a.out, "w") if a.out else None
    L = _cabi.lib()
    for size, (b, hf, wf) in sizes.items():
        for name, c, o, lv in layers:
            d, h, w = 64 // lv, hf // lv, wf // lv
            g = torch.Generator().manual_seed(0)
            x = torch.randn(b, c, d, h, w, generator=g).to(dev)
            gout = torch.randn(b, o, d, h, w, generator=g).to(dev)
            lay = ConvBR_3d(c, o).to(dev)
            flop = 2.0 * b * o * d * h * w * c * 27
            floor_ms = flop / FP32_PEAK * 1e3
            res = {}
            # ---- ours ----
            ours = (c, o) in PAIRS
            xg = x.clone().requires_grad_(True)
            gz = gin = ws = None
            if ours:
                lay.eval()
                with torch.no_grad():
                    res["ours_eval_fwd"] = timed(lambda: matching_forward(lay, x))
                    res["ours_conv_fwd_kernel"] = timed(lambda: conv3d_cc_forward(x, lay.conv.weight))
                lay.train()
                res["ours_train_fwd"] = timed(lambda: matching_forward(lay, xg))
                res["ours_train_fwd_bwd"] = timed(lambda: matching_forward(lay, xg).backward(gout))
                res["ours_bwd"] = res["ours_train_fwd_bwd"] - res["ours_train_fwd"]
                gz, gin, gw = torch.empty_like(gout), torch.empty_like(x), torch.empty_like(lay.conv.weight)
                ws = torch.empty(int(L.rag_conv3d_cc_bwd_workspace_bytes(b, c, o, d, h, w)) // 4, device=dev)
                st = torch.cuda.current_stream().cuda_stream
                wt = lay.conv.weight.detach()
                res["ours_data_grad_kernel"] = timed(lambda: _cabi.check(L.rag_conv3d_cc_bwd(gout.data_ptr(), x.data_ptr(), wt.data_ptr(), gin.data_ptr(), None, None, b, c, o, d, h, w, st), "bwd"))
                res["ours_weight_grad_kernels"] = timed(lambda: _cabi.check(L.rag_conv3d_cc_bwd(gout.data_ptr(), x.data_ptr(), wt.data_ptr(), None, gw.data_ptr(), ws.data_ptr(), b, c, o, d, h, w, st), "bwd"))
                consts = torch.rand(o, 7, device=dev)
                res["ours_gz_kernel"] = timed(lambda: _cabi.check(L.rag_bn3d_bwd_gz(gout.data_ptr(), gout.data_ptr(), consts.data_ptr(), gz.data_ptr(), b, o, d, h, w, st), "gz"))
            # ---- cuDNN through the mirror layer ----
            ref = copy.deepcopy(lay)
            for tf32 in (True, False):
                torch.backends.cudnn.allow_tf32 = tf32
                tag = "tf32" if tf32 else "fp32"
                ref.eval()
                with torch.no_grad():
                    res[f"cudnn_{tag}_eval_fwd"] = timed(lambda: ref(x))
                ref.train()
                res[f"cudnn_{tag}_train_fwd_bwd"] = timed(lambda: ref(xg).backward(gout))
            torch.backends.cudnn.allow_tf32 = True
            row = {"layer": name, "C": c, "O": o, "size": size, "shape": [b, c, d, h, w], "gflop_per_conv": round(flop / 1e9, 2),
                   "fp32_floor_ms": round(floor_ms, 4)}
            row.update({k: round(v, 4) for k, v in res.items()})
            if ours:
                row["conv_fwd_frac_of_floor"] = round(floor_ms / res["ours_conv_fwd_kernel"], 3)
                row["conv_fwd_tflops"] = round(flop / res["ours_conv_fwd_kernel"] / 1e9, 1)
                row["train_fwd_bwd_frac_of_floor"] = round(3 * floor_ms / res["ours_train_fwd_bwd"], 3)
                row["faster_than_cudnn_tf32"] = bool(res["ours_eval_fwd"] < res["cudnn_tf32_eval_fwd"] and res["ours_train_fwd_bwd"] < res["cudnn_tf32_train_fwd_bwd"])
            else:
                row["note"] = "not compiled: cuDNN only"
            row["card"] = card()
            row["method"] = "CUDA events per pass, 256 MB L2 flush between passes, median of %d" % a.reps
            print(json.dumps(row), flush=True)
            if out:
                out.write(json.dumps(row) + "\n")
            del x, gout, xg, gz, gin, ws, lay, ref
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
