"""Small shapes through every kernel/variant (written for compute-sanitizer memcheck/racecheck runs; the tool is
closed on this GPU pool, where the script serves as a plain smoke run and tests/test_guard_bands_gpu.py -- canary
windows around every output -- is the out-of-bounds check)."""
import os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rag_b200 import functional as F_, metrics as M, staging as S

dev = "cuda"
refused = 0


def run(fn, *a, **k):
    """A variant may refuse a shape with an argument error (RuntimeError from the ABI): that is fine here."""
    global refused
    try:
        return fn(*a, **k)
    except RuntimeError as e:
        if "failed with code" not in str(e):
            raise
        refused += 1
        return None


g = torch.Generator(device=dev).manual_seed(0)
for (b, c, hf, wf, md) in [(1, 12, 9, 36, 96), (2, 3, 5, 37, 30), (1, 4, 7, 70, 192), (1, 2, 3, 10, 48)]:
    x = torch.randn(b, c, hf, wf, device=dev, generator=g); y = torch.randn(b, c, hf, wf, device=dev, generator=g)
    df = int(md / 3)
    for v in (None, 0, 1, 3, 5):
        cost = run(F_.cost_volume_forward, x, y, df, variant=v)
    cost = F_.cost_volume_forward(x, y, df)
    gc = torch.randn_like(cost)
    for v in (None, 0, 1, 2, 3):
        run(F_.cost_volume_backward, gc, c, variant=v)
for (b, dl, hl, wl, md) in [(1, 16, 5, 36, 48), (2, 8, 3, 7, 24), (1, 20, 9, 4, 60), (1, 12, 3, 4, 48), (1, 64, 6, 40, 192)]:
    cl = torch.randn(b, 1, dl, hl, wl, device=dev, generator=g)
    gd = torch.randn(b, 3 * hl, 3 * wl, device=dev, generator=g)
    x3 = md == 3 * dl
    for vf in [None, 0] + ([1, 2, 4] if x3 else []):
        run(F_.disp_head_forward, cl, md, True, variant=vf)
    disp, st = F_.disp_head_forward(cl, md, True)
    for vb in [None, 0] + ([1, 2, 3] if x3 else []):
        run(F_.disp_head_backward, cl, gd, disp, st, md, variant=vb)
    F_.upsample_trilinear(cl, md, True)
p = torch.softmax(torch.randn(1, 24, 6, 10, device=dev, generator=g), 1).contiguous().requires_grad_(True)
F_.DisparityRegressionFn.apply(p, 24).sum().backward()
gt = torch.rand(2, 20, 30, device=dev, generator=g) * 250 - 20
est = (gt + torch.randn(2, 20, 30, device=dev, generator=g)).requires_grad_(True)
loss, sums = M.masked_smooth_l1(est, gt, 192); loss.backward()
S.normalize_pad(torch.randint(0, 256, (2, 10, 14, 3), device=dev, dtype=torch.uint8), 12, 18)
# next rows: fused stem (all variants) and the last_3_3d convolution
from rag_b200.fused_stem import cv_stem_forward
from rag_b200.last_conv import conv3d_c1_forward
for (b, hf, wf, md) in [(1, 5, 12, 24), (2, 4, 40, 48), (1, 3, 36, 96)]:
    x = torch.randn(b, 12, hf, wf, device=dev, generator=g); y = torch.randn(b, 12, hf, wf, device=dev, generator=g)
    w = torch.randn(12, 24, 3, 3, 3, device=dev, generator=g) * 0.1
    sc = torch.rand(12, device=dev, generator=g) + 0.5; sh = torch.randn(12, device=dev, generator=g)
    for relu in (True, False):
        for v in (None, 0, 1, 2):
            run(cv_stem_forward, x, y, w, sc, sh, relu, md, variant=v)
for (b, c, d, h, w_) in [(1, 12, 18, 9, 12), (2, 12, 5, 17, 72), (1, 12, 64, 8, 64)]:
    conv3d_c1_forward(torch.randn(b, c, d, h, w_, device=dev, generator=g), torch.randn(1, c, 3, 3, 3, device=dev, generator=g))
torch.cuda.synchronize()
print("sanitize_smoke ok; calls refused with an argument error:", refused)
