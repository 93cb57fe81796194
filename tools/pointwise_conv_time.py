"""Per-layer timing of the pointwise ConvBR_3d layers (csrc/conv3d_pw.cu) against cuDNN, on the GPU.

    python tools/pointwise_conv_time.py [--reps 20] [--out profiles/r4_pointwise_conv_times.jsonl]

Shapes at B=4 288x576 and B=8 480x960 (Hf, Wf = H/3, W/3, Df = 64; level 6 / 12 halve / quarter all three):
`last_12_3d` 48 -> 24 at level 12, `last_6_3d` 24 -> 12 at level 6, and the likely cell 1x1x1 layers 12 -> 4 (level 3),
24 -> 8 (level 6), 48 -> 16 (level 12); and 48 -> 28, 64 -> 32 at level 6, the forward's two register-capped tiles
(OT = 28, 32).  --layers picks pairs.
  ours:  eval forward (folded BatchNorm + ReLU, one kernel) through the layer (with batchnorm.eval_fold's small torch ops)
         and the kernel alone; training forward + backward with autograd; the fused backward kernel alone (gin +
         weight-gradient partials + final pass, from g, z and the BatchNorm constants);
  cuDNN: the mirror ConvBR_3d through PyTorch eager, eval forward and train forward + backward, TF32 on (the reference's
         default) and off.
Method: CUDA events around each pass, a 256 MB buffer overwritten between passes (L2 flush, outside the events), median of
--reps passes after 3 warm-up passes.  HBM floors from bytes at 6460.5 GB/s (the copy bandwidth measured on a B200, DESIGN.md
5): eval forward reads x and writes out once, 4*B*S*(C+O) bytes; the fused backward reads g, z and x and writes gin,
4*B*S*(2*O + 2*C) bytes.  `routed_to_kernels` says whether install(..., pointwise_convs=True) sends the shape to the kernels
(pointwise_conv.MIN_VOXELS); the kernels are timed either way.  One JSON line per case, with the card name, power limit
and SM clock read in the same run."""
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
from rag_b200 import _cabi, batchnorm, pointwise_conv  # noqa: E402
from rag_b200.pointwise_conv import conv3d_pw_forward, convbr_forward, qualifies  # noqa: E402

HBM_BPS = 6460.5e9


class ConvBR_3d(nn.Module):
    def __init__(self, c, o):
        super().__init__()
        self.relu, self.use_bn = True, True
        self.conv = nn.Conv3d(c, o, 1, stride=1, padding=0, bias=False)
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
    ap.add_argument("--layers", default=None, help="only these C:O pairs, comma-separated (e.g. 48:28,64:32)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pointwise_conv_time.py measures on a GPU; none is visible")
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
    layers = [("last_12_3d", 48, 24, 4), ("last_6_3d", 24, 12, 2),
              ("cell 1x1x1 (inferred)", 12, 4, 1), ("cell 1x1x1 (inferred)", 24, 8, 2), ("cell 1x1x1 (inferred)", 48, 16, 4),
              ("OT=28 probe", 48, 28, 2), ("OT=32 probe", 64, 32, 2)]
    if a.layers:
        keep = {tuple(int(v) for v in p.split(":")) for p in a.layers.split(",")}
        layers = [r for r in layers if (r[1], r[2]) in keep]
    out = open(a.out, "w") if a.out else None
    L = _cabi.lib()
    who = card()
    for size, (b, hf, wf) in sizes.items():
        for name, c, o, lv in layers:
            d, h, w = 64 // lv, hf // lv, wf // lv
            S = d * h * w
            g = torch.Generator().manual_seed(0)
            x = torch.randn(b, c, d, h, w, generator=g).to(dev)
            gout = torch.randn(b, o, d, h, w, generator=g).to(dev)
            lay = ConvBR_3d(c, o).to(dev)
            xg = x.clone().requires_grad_(True)
            res = {}
            # ---- ours ----
            lay.eval()
            with torch.no_grad():
                routed = qualifies(lay, x)                         # what install(..., pointwise_convs=True) does here
                floor_voxels, pointwise_conv.MIN_VOXELS = pointwise_conv.MIN_VOXELS, 0
                assert qualifies(lay, x)                           # the kernels are timed on every shape
                res["ours_eval_fwd"] = timed(lambda: convbr_forward(lay, x))
                scale, shift = batchnorm.eval_fold(lay.bn)
                res["ours_eval_fwd_kernel"] = timed(lambda: conv3d_pw_forward(x, lay.conv.weight, scale, shift, relu=True))
            lay.train()
            res["ours_train_fwd"] = timed(lambda: convbr_forward(lay, xg))
            res["ours_train_fwd_bwd"] = timed(lambda: convbr_forward(lay, xg).backward(gout))
            z = torch.randn(b, o, d, h, w, generator=g).to(dev)
            consts = torch.rand(o, 7, device=dev)
            gin, gw = torch.empty_like(x), torch.empty(o, c, device=dev)
            ws = torch.empty(int(L.rag_conv3d_pw_bwd_workspace_bytes(b, c, o, d, h, w)) // 4, device=dev)
            wt = lay.conv.weight.detach()
            st = torch.cuda.current_stream().cuda_stream
            res["ours_fused_bwd_kernels"] = timed(lambda: _cabi.check(L.rag_conv3d_pw_bwd(
                gout.data_ptr(), z.data_ptr(), consts.data_ptr(), x.data_ptr(), wt.data_ptr(), gin.data_ptr(), gw.data_ptr(),
                ws.data_ptr(), b, c, o, d, h, w, st), "rag_conv3d_pw_bwd"))
            gz = torch.empty_like(gout)
            res["ours_gz_kernel"] = timed(lambda: _cabi.check(L.rag_bn3d_bwd_gz(
                gout.data_ptr(), z.data_ptr(), consts.data_ptr(), gz.data_ptr(), b, o, d, h, w, st), "rag_bn3d_bwd_gz"))
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
            eval_floor = 4.0 * b * S * (c + o) / HBM_BPS * 1e3
            bwd_floor = 4.0 * b * S * (2 * o + 2 * c) / HBM_BPS * 1e3
            row = {"layer": name, "C": c, "O": o, "size": size, "shape": [b, c, d, h, w],
                   "eval_hbm_floor_ms": round(eval_floor, 4), "fused_bwd_hbm_floor_ms": round(bwd_floor, 4)}
            row.update({k: round(v, 4) for k, v in res.items()})
            row["eval_fwd_frac_of_floor"] = round(eval_floor / res["ours_eval_fwd"], 3)
            row["eval_fwd_kernel_frac_of_floor"] = round(eval_floor / res["ours_eval_fwd_kernel"], 3)
            row["fused_bwd_frac_of_floor"] = round(bwd_floor / res["ours_fused_bwd_kernels"], 3)
            row["eval_speedup_vs_cudnn_tf32"] = round(res["cudnn_tf32_eval_fwd"] / res["ours_eval_fwd"], 2)
            row["train_speedup_vs_cudnn_tf32"] = round(res["cudnn_tf32_train_fwd_bwd"] / res["ours_train_fwd_bwd"], 2)
            row["faster_than_cudnn_tf32"] = bool(res["ours_eval_fwd"] < res["cudnn_tf32_eval_fwd"]
                                                 and res["ours_train_fwd_bwd"] < res["cudnn_tf32_train_fwd_bwd"])
            row["routed_to_kernels"] = bool(routed)
            row["card"] = who
            row["method"] = "CUDA events per pass, 256 MB L2 flush between passes, median of %d" % a.reps
            print(json.dumps(row), flush=True)
            if out:
                out.write(json.dumps(row) + "\n")
            pointwise_conv.MIN_VOXELS = floor_voxels
            del x, gout, xg, z, gz, gin, ws, lay, ref
            torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
