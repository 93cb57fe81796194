"""The weight gradients whose fixed grid makes each CTA (or warp) walk several work items, against fp64 at shapes where the
walk wraps: some CTA (warp) takes two items or more and the last round is uneven (tests/_grids.py restates the grids).  What
only a second item exercises -- the prefetch of the next item's first plane while the current one is computed, fp32 partial
sums carried across items, shared memory reused from one tile to the next -- is checked here:

* conv3d_cc's weight gradient (the Matching Net's 3x3x3 ConvBR_3d, csrc/conv3d_cc.cu) through ``matching_forward`` in
  train(), as tests/test_matching_conv_gpu.py::test_training_vs_fp64 does, on a ragged synthetic shape and at the training
  crop (B=4 288x576: [4, C, 64, 96, 192]);
* last_3_3d's weight gradient (csrc/last_conv_bwd.cu) through ``Conv3dC1Fn``, with the bounds of
  tests/test_tail_gpu.py::test_last_conv_backward_vs_fp64.

The disparity head's persistent variants loop at the BASELINE sizes of tests/test_disp_head_gpu.py and at the training shape of
tests/test_next_rows_gpu.py, where they are compared bit for bit with the default grids.

Each case prints the items per CTA (warp), the max-norm error against fp64 of ours and of plain fp32 (cuDNN, TF32 off), its
wall time and its peak device memory."""
import time
import zlib

import pytest
import torch
import torch.nn.functional as F

from tests import _grids
from tests._util import gen, randn
from tests.test_matching_conv_gpu import _fp32_convs, _layer, _masked, _mx, _run  # noqa: F401  (_fp32_convs: autouse, TF32 off)

pytestmark = pytest.mark.gpu
NAMES = ["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]


@pytest.fixture(autouse=True)
def _measured(request):
    """Frees the case's temporaries (the fp64 ones are GBs at the training crop) and prints its wall time and peak memory."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    print(f"  [{request.node.name}: {time.perf_counter() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB]")
    torch.cuda.empty_cache()


def _report(name, span, errs):
    return f"\n{name}: {span}; vs fp64 ours / fp32: " + ", ".join(f"{n} {e:.2e} / {e32:.2e}" for n, (e, e32) in errs.items())


# (pair, (B, D, H, W)).  [3, C, 17, 37, 136]: 513 tiles on 296 CTAs; D = 17 ends in a one-plane tile (the prefetch crosses
# into the next tile at once), H odd, W leaves an 8-wide w tail.  [4, C, 64, 96, 192]: the training crop, 4608 tiles; (12,12)
# is stem3d1, (4,4) and (8,8) the level-3 conv_3x3 of cells with k = 4 and 8.
CC_CASES = [((c, c), s) for s in ((3, 17, 37, 136), (4, 64, 96, 192)) for c in (4, 8, 12)]


@pytest.mark.parametrize("pair, shape", CC_CASES, ids=[f"{p[0]}x{p[1]}-" + "x".join(map(str, s)) for p, s in CC_CASES])
def test_matching_conv_training_vs_fp64_many_tiles_per_cta(pair, shape):
    from rag_b200.matching_conv import matching_forward, qualifies

    c, o = pair
    b, d, h, w = shape
    span = _grids.loops(*_grids.cc_wgrad(b, d, h, w))
    g = gen(zlib.crc32(repr((pair, shape)).encode()) % 991)
    layer = _layer(c, o, g).train()
    x0 = randn((b, c, d, h, w), g).cuda()
    gout = randn((b, o, d, h, w), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)
    assert qualifies(layer, x0.clone().requires_grad_(True))
    ours, _ = _run(layer, x0, gout, matching_forward, torch.float32)
    mask = ours[0] > 0

    def plain(lay, x):
        return _masked(lay, x, mask)

    ref64, pre64 = _run(layer, x0, gout, plain, torch.float64)
    pre64 = pre64.detach()
    flips = (pre64 > 0) != mask
    n_flips = int(flips.sum())
    flip = pre64[flips].abs().max().item() / pre64.abs().max().item() if n_flips else 0.0
    del pre64, flips
    fp32, _ = _run(layer, x0, gout, plain, torch.float32)
    errs = {n: (_mx(a, r), _mx(f, r)) for n, a, f, r in zip(NAMES, ours, fp32, ref64)}
    print(_report(f"conv3d_cc {pair} {list(shape)}", span, errs) + f"; {n_flips} ReLU decisions differ from fp64 (largest |pre| {flip:.1e} of the max)")
    assert flip <= 1e-5, "ReLU decision differs from fp64 beyond rounding"
    for n, (e, e32) in errs.items():
        assert e <= 1e-5, f"{n}: ours {e:.3e} (fp32 {e32:.3e})"


# (B, C, D, H, W).  [24, 3, 33, 38, 132]: 2400 items on 1184 warps per channel pair, 32 warps take 3; D = 33 leaves a
# one-plane segment, H and W have tails, C = 3 leaves the last channel pair single.  [8, 12, 64, 96, 192]: the training crop at
# batch 8, 2304 items.
C1_CASES = [(24, 3, 33, 38, 132), (8, 12, 64, 96, 192)]


@pytest.mark.parametrize("case", C1_CASES, ids=lambda c: "x".join(map(str, c)))
def test_last_conv_backward_vs_fp64_many_items_per_warp(case):
    from rag_b200.last_conv import Conv3dC1Fn

    b, c, d, h, w = case
    span = _grids.loops(*_grids.c1_bwd_weight(b, d, h, w))
    g = gen(zlib.crc32(repr(case).encode()) % 983)
    x0 = randn((b, c, d, h, w), g).cuda()
    w0 = (randn((1, c, 3, 3, 3), g) * 0.2).cuda()
    go = randn((b, 1, d, h, w), g).cuda()

    def grads(fn, dtype):
        x, wt = x0.to(dtype, copy=True).requires_grad_(True), w0.to(dtype, copy=True).requires_grad_(True)
        fn(x, wt).backward(go.to(dtype))
        return x.grad, wt.grad

    def plain(x, wt):
        return F.conv3d(x, wt, padding=1)

    ours = grads(Conv3dC1Fn.apply, torch.float32)
    ref64 = grads(plain, torch.float64)
    fp32 = grads(plain, torch.float32)
    errs = {n: (_mx(a, r), _mx(f, r)) for n, a, f, r in zip(["gx", "gweight"], ours, fp32, ref64)}
    print(_report(f"last_3_3d {list(case)}", span, errs))
    assert errs["gx"][0] <= 2e-6, f"data gradient {errs['gx'][0]:.2e}"
    assert errs["gweight"][0] <= 1e-5, f"weight gradient {errs['gweight'][0]:.2e}"
