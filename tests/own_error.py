"""Own error of the head-forward variants vs the fp64 evaluation of the reference formula (test infrastructure, lives under tests/ because it
imports the oracle).  usage: own_error.py [v ...]"""
import os, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))  # tests/ -> repo root
sys.path.insert(0, ROOT)
from rag_b200 import functional as F_
from oracle import rag_oracle as O
vs = [int(a) for a in sys.argv[1:]] or [0, 1, 2, 4]
for (dl, hl, wl, md, sigma) in ((64, 48, 96, 192, 1.0), (64, 48, 96, 192, 5.0), (96, 24, 64, 288, 1.0), (64, 48, 96, 192, 20.0)):
    g = torch.Generator().manual_seed(7)
    cost = torch.randn(2, 1, dl, hl, wl, generator=g) * sigma
    d64, _ = O.disp_head_f64(cost[:, 0].numpy(), md)
    ref = O.disp_head_ref(cost.cuda(), md).cpu().numpy()
    print(f"Dl={dl} {3*hl}x{3*wl} maxdisp={md} sigma={sigma}: reference(torch CUDA fp32) vs fp64: max {np.abs(ref-d64).max():.2e} mean {np.abs(ref-d64).mean():.2e}")
    for v in vs:
        out = F_.disp_head_forward(cost.cuda(), md, False, variant=v)[0].cpu().numpy()
        e = np.abs(out - d64)
        print(f"   variant {v:2d}: own max {e.max():.2e} mean {e.mean():.2e} p99.9 {np.quantile(e, 0.999):.2e} | vs reference max {np.abs(out-ref).max():.2e}")
