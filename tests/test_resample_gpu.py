"""The drop-in F.interpolate on the GPU (rag_b200/resample.py, csrc/trilinear.cu): bilinear and trilinear forward and
fixed-order backward against ATen and fp64, repeatability, launch counts, CUDA-graph replay, the routing, and a training
step of a network with the RAG structure under torch.use_deterministic_algorithms(True)."""
from copy import deepcopy

import pytest
import torch
import torch.nn.functional as F

from tests._stand_in import _stand_in
from tests._util import gen, randn

pytestmark = pytest.mark.gpu


def _mx(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


CASES = [
    # (mode, B, C, in size, out size, align_corners)
    ("trilinear", 2, 3, (8, 12, 16), (4, 6, 8), True),            # down by 2 (the cells' 3 -> 6)
    ("trilinear", 1, 2, (16, 12, 32), (4, 3, 8), True),           # down by 4 (3 -> 12)
    ("trilinear", 1, 4, (4, 6, 8), (8, 12, 16), False),           # up by 2
    ("trilinear", 1, 2, (5, 7, 9), (3, 4, 5), False),             # odd sizes: the per-voxel kernels
    ("trilinear", 1, 2, (4, 6, 320), (2, 3, 160), True),          # level-3 width at 480x960: per-voxel forward, row backward
    ("trilinear", 1, 2, (4, 5, 416), (2, 3, 208), False),         # level-3 width at 384x1248
    ("trilinear", 1, 1, (2, 3, 320), (3, 5, 416), True),          # up from a 320-wide row
    ("trilinear", 1, 3, (16, 24, 320), (4, 6, 80), True),         # 3 -> 12 at 480x960, one depth quarter
    ("bilinear", 2, 3, (12, 16), (6, 8), True),                   # down by 2
    ("bilinear", 1, 2, (24, 32), (6, 8), True),                   # down by 4
    ("bilinear", 2, 3, (6, 8), (12, 16), False),                  # up by 2
    ("bilinear", 1, 2, (7, 9), (11, 13), True),                   # odd sizes, up
    ("bilinear", 1, 2, (7, 9), (4, 5), False),                    # odd sizes, down
    ("bilinear", 1, 2, (6, 320), (3, 160), True),                 # the level-3 widths
    ("bilinear", 1, 2, (5, 416), (9, 208), False),
    ("bilinear", 2, 3, (10, 320), (20, 416), True),
    ("bilinear", 2, 8, (48, 96), (24, 48), True),                 # Feature-Net level 6 -> 12 at 288x576
    ("bilinear", 1, 1, (1, 4), (5, 9), True),                     # singleton axis (scale 0 with align_corners)
    ("bilinear", 1, 2, (5, 6), (5, 6), False),                    # identity
]


@pytest.mark.parametrize("case", CASES, ids=str)
def test_forward_backward_vs_aten_and_fp64(case):
    from rag_b200 import _cabi
    from rag_b200.resample import interpolate

    mode, b, c, si, so, ac = case
    g = gen(hash(case) % 977)
    x0 = randn((b, c) + si, g).cuda()
    go = randn((b, c) + so, g).cuda()
    xr = x0.clone().requires_grad_(True)
    ref = F.interpolate(xr, so, mode=mode, align_corners=ac)
    ref.backward(go)
    x64 = x0.double().requires_grad_(True)
    r64 = F.interpolate(x64, so, mode=mode, align_corners=ac)
    r64.backward(go.double())
    x = x0.clone().requires_grad_(True)
    n0 = _cabi.launch_count()
    out = interpolate(x, so, mode=mode, align_corners=ac)
    assert _cabi.launch_count() - n0 == 1
    out.backward(go)
    assert _cabi.launch_count() - n0 == 2
    assert out.shape == ref.shape and out.is_contiguous()
    assert _mx(out.detach(), ref.detach()) <= 1e-6, f"fwd vs ATen fp32: {_mx(out.detach(), ref.detach()):.2e}"
    assert _mx(x.grad, xr.grad) <= 1e-6, f"bwd vs ATen fp32: {_mx(x.grad, xr.grad):.2e}"
    # fp64 has exact lambdas; ATen's fp32 lambdas (reproduced here) are off by ~6e-8 * index: as close as ATen, or closer
    assert _mx(out.detach(), r64.detach()) <= 2 * _mx(ref.detach(), r64.detach()) + 1e-6
    assert _mx(x.grad, x64.grad) <= 2 * _mx(xr.grad, x64.grad) + 1e-6


@pytest.mark.parametrize("mode", ["trilinear", "bilinear"])
def test_backward_is_bitwise_repeatable(mode):
    from rag_b200.resample import interpolate

    g = gen(5)
    shape, size = ((2, 12, 16, 24, 48), (8, 12, 24)) if mode == "trilinear" else ((2, 24, 48, 96), (24, 48))
    x0 = randn(shape, g).cuda()
    go = randn(shape[:2] + size, g).cuda()
    grads, outs = [], []
    for _ in range(3):
        x = x0.clone().requires_grad_(True)
        out = interpolate(x, size, mode=mode, align_corners=True)
        out.backward(go)
        grads.append(x.grad)
        outs.append(out.detach())
    assert all(torch.equal(grads[0], gr) for gr in grads[1:]) and all(torch.equal(outs[0], o) for o in outs[1:])


@pytest.mark.parametrize("mode", ["trilinear", "bilinear"])
def test_cuda_graph_capture_replays_bit_exact(mode):
    from rag_b200.resample import interpolate

    g = gen(11)
    shape, size = ((2, 4, 8, 12, 320), (16, 24, 160)) if mode == "trilinear" else ((2, 4, 12, 320), (24, 160))
    x = randn(shape, g).cuda().requires_grad_(True)
    go = randn(shape[:2] + size, g).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = interpolate(x, size, mode=mode, align_corners=True)
        eager.backward(go)
        e_out, e_gx = eager.detach().clone(), x.grad.clone()
    torch.cuda.current_stream().wait_stream(s)
    x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = interpolate(x, size, mode=mode, align_corners=True)
        out.backward(go)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out.detach(), e_out) and torch.equal(x.grad, e_gx)


def test_routing_on_the_device():
    """Routed calls launch the kernels; every other call is F.interpolate itself (bit-identical, no launch)."""
    from rag_b200 import _cabi
    from rag_b200.resample import interpolate

    g = gen(13)
    x4, x5 = randn((2, 3, 6, 8), g).cuda(), randn((1, 2, 4, 6, 8), g).cuda()
    routed = [(x4, dict(size=(12, 16), mode="bilinear", align_corners=True)),
              (x4, dict(scale_factor=2, mode="bilinear", align_corners=True)),
              (x4, dict(scale_factor=0.5, mode="bilinear", recompute_scale_factor=True)),
              (x5, dict(size=(2, 3, 4), mode="trilinear")),
              (x5, dict(scale_factor=(2, 0.5, 1.5), mode="trilinear", align_corners=True))]
    for x, kw in routed:
        n0 = _cabi.launch_count()
        out = interpolate(x, **kw)
        assert _cabi.launch_count() - n0 == 1, kw
        ref = F.interpolate(x, **kw)
        assert out.shape == ref.shape and _mx(out, ref) <= 1e-6, kw
    through = [(x4, dict(scale_factor=2, mode="bilinear", align_corners=False)),
               (x4.contiguous(memory_format=torch.channels_last), dict(size=(12, 16), mode="bilinear", align_corners=True)),
               (x4.double(), dict(size=(12, 16), mode="bilinear", align_corners=True)),
               (x4, dict(size=(12, 16), mode="nearest")),
               (x4, dict(size=(12, 16), mode="bicubic", align_corners=True)),
               (x4, dict(size=(12, 16), mode="bilinear", align_corners=True, antialias=True)),
               (x5[:, :, :, :, ::2], dict(size=(8, 12, 8), mode="trilinear", align_corners=True))]      # not contiguous
    for x, kw in through:
        n0 = _cabi.launch_count()
        out = interpolate(x, **kw)
        assert _cabi.launch_count() - n0 == 0, kw
        ref = F.interpolate(x, **kw)
        assert torch.equal(out, ref) and out.stride() == ref.stride(), kw


# ---------------------------------------------------------------------------------------------------------------------
# A training step under torch.use_deterministic_algorithms(True), on a stand-in with the RAG structure
# ---------------------------------------------------------------------------------------------------------------------
class _CountDecomposition:
    """Counts the calls F.interpolate makes, under deterministic mode, into torch's linear-mode decomposition."""

    def __init__(self, monkeypatch):
        import torch._decomp.decompositions as D

        self.n, orig = 0, D._upsample_linear_vec

        def counted(*a, **k):
            self.n += 1
            return orig(*a, **k)

        monkeypatch.setattr(D, "_upsample_linear_vec", counted)


def _train_step(net, state, left, right, gt):
    """One step of the reference's training: the masked smooth-L1 loss (approaches/rag.py)."""
    net.load_state_dict(state)
    net.train()
    net.zero_grad(set_to_none=True)
    pred = net(left, right, 0)
    mask = (gt < net.maxdisp) & (gt > 0)
    loss = F.smooth_l1_loss(pred[mask], gt[mask], reduction="mean")
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in net.named_parameters()}
    bufs = {n: b.detach().clone() for n, b in net.named_buffers()}
    return loss.detach().clone(), pred.detach().clone(), grads, bufs


def test_training_step_under_deterministic_mode(monkeypatch):
    """install(fuse_stem, upsample, matching_convs, pointwise_convs, resample): a whole training step of the stand-in runs
    under torch.use_deterministic_algorithms(True) on the kernels, twice with bit-identical loss, gradients and running
    statistics, everything finite although the mode fills torch.empty with NaN.  Without resample=True the cells'
    F.interpolate calls go to torch's decomposition instead (ATen's own kernel refuses the mode)."""
    from rag_b200 import _cabi, pointwise_conv
    from rag_b200 import network as N

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)        # the stand-in is small: its 1x1x1 layers take the kernels
    rag_model, ops3d, cells = _stand_in()
    g = gen(21)
    left, right = randn((2, 3, 48, 96), g).cuda(), randn((2, 3, 48, 96), g).cuda()
    gt = (torch.rand(2, 48, 96, generator=g) * 60 - 6).cuda()        # some pixels outside (0, maxdisp): masked out
    flags = dict(fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True)
    N.uninstall()
    was = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    try:
        N.install(rag_model, None, ops3d, **flags)
        torch.manual_seed(7)
        net = rag_model.Network().cuda()                          # built after install: the head is rag_b200.Disp
        state = deepcopy(net.state_dict())
        torch.use_deterministic_algorithms(True)
        assert torch.utils.deterministic.fill_uninitialized_memory
        # positive control: ATen's bilinear / trilinear backward refuse the mode, and F.interpolate avoids them through
        # torch's decomposition -- which the stand-in's cells take while resample is off
        for shape, fn in (((1, 2, 6, 8), torch._C._nn.upsample_bilinear2d), ((1, 2, 4, 6, 8), torch._C._nn.upsample_trilinear3d)):
            x = torch.ones(shape, device="cuda", requires_grad=True)
            with pytest.raises(RuntimeError, match="deterministic"):
                fn(x, [2 * s for s in shape[2:]], True, None).sum().backward()
        count = _CountDecomposition(monkeypatch)
        n0 = _cabi.launch_count()
        loss_off, pred_off, _, _ = _train_step(net, state, left, right, gt)
        n_off = _cabi.launch_count() - n0
        assert count.n == 6, count.n          # 2 bilinear per feature pass (left and right) + 2 trilinear in the 3-D cell
        # the feature under test
        N.install(rag_model, None, ops3d, resample=True, resample_modules=(cells,), **flags)
        count.n = 0
        n0 = _cabi.launch_count()
        first = _train_step(net, state, left, right, gt)
        n_on = _cabi.launch_count() - n0
        second = _train_step(net, state, left, right, gt)
        assert count.n == 0
        assert n_on - n_off == 2 * 6          # each of the six resamples: one forward and one backward launch
        loss, pred, grads, bufs = first
        assert torch.equal(loss, second[0]) and torch.equal(pred, second[1])
        assert all(torch.equal(grads[n], second[2][n]) for n in grads), [n for n in grads if not torch.equal(grads[n], second[2][n])]
        assert all(torch.equal(bufs[n], second[3][n]) for n in bufs)
        assert torch.isfinite(loss) and torch.isfinite(pred).all()
        assert all(torch.isfinite(v).all() for v in grads.values()) and all(torch.isfinite(v.float()).all() for v in bufs.values())
        assert any(v.abs().sum() > 0 for n, v in grads.items() if n.startswith("cell2d")), "no gradient reached the 2-D cell"
        # torch's decomposition and the kernels compute the same step, up to fp32 rounding
        assert abs(loss.item() - loss_off.item()) <= 1e-4 * abs(loss_off.item())
        assert _mx(pred, pred_off) <= 1e-4
    finally:
        torch.use_deterministic_algorithms(was[0], warn_only=was[1])
        N.uninstall()


def test_resample_on_the_real_network(monkeypatch):
    """The same on the reference's own Network, skipped when oracle/_ref is absent."""
    import os
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle import refimport as R

    if not R.available():
        pytest.skip("the unmodified reference is not installed in oracle/_ref")
    from rag_b200 import _cabi, pointwise_conv
    from rag_b200 import network as N

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)
    ref = R.import_reference()
    N.uninstall()
    g = gen(23)
    H, W = 96, 192
    left, right = randn((2, 3, H, W), g).cuda(), randn((2, 3, H, W), g).cuda()
    gt = (torch.rand(2, H, W, generator=g) * 200 - 8).cuda()
    was = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    try:
        N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, fuse_stem=True, upsample=True, matching_convs=True,
                  pointwise_convs=True, resample=True)
        torch.manual_seed(3)
        net = ref.rag_model.Network(R.make_genotype(ref, 3), "cuda").cuda().train()
        state = deepcopy(net.state_dict())
        torch.use_deterministic_algorithms(True)

        def step():
            net.load_state_dict(state)
            net.zero_grad(set_to_none=True)
            pred = net.forward(left, right, 0, net.arch_init)
            mask = (gt < net.maxdisp) & (gt > 0)
            loss = F.smooth_l1_loss(pred[mask], gt[mask], reduction="mean")
            loss.backward()
            return loss.detach().clone(), {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}

        n0 = _cabi.launch_count()
        l1, g1 = step()
        assert _cabi.launch_count() > n0
        l2, g2 = step()
        assert torch.equal(l1, l2) and torch.isfinite(l1)
        assert set(g1) == set(g2) and all(torch.equal(g1[n], g2[n]) for n in g1)
        assert all(torch.isfinite(v).all() for v in g1.values())
    finally:
        torch.use_deterministic_algorithms(was[0], warn_only=was[1])
        N.uninstall()
