"""Fused cost volume + first Matching-Net convolution (SURVEY.md section 8f rank 1) against the reference
composition: cost volume (rag_model.py:375-383) -> Conv3d(2C->O,3,pad 1,bias=False) -> BatchNorm3d(eval)
-> ReLU (operations_3d.py:31-47), evaluated in full fp32 (TF32 off) on the materialised oracle volume.

Tolerance: the fused kernel sums the same 648 products per output in a different order (all fp32):
max-norm relative 1e-5 of the conv output."""
import copy

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import rag_oracle as O
from tests._util import gen, randn

pytestmark = pytest.mark.gpu


class ConvBR_3d(nn.Module):
    """Same fields / forward as the reference's ConvBR_3d (operations_3d.py:31-47)."""

    def __init__(self, c_in, c_out, bn=True, relu=True):
        super().__init__()
        self.relu = relu
        self.use_bn = bn
        self.conv = nn.Conv3d(c_in, c_out, 3, stride=1, padding=1, bias=False)
        self.bn = nn.BatchNorm3d(c_out)

    def forward(self, x):
        x = self.conv(x)
        if self.use_bn:
            x = self.bn(x)
        if self.relu:
            x = F.relu(x, inplace=True)
        return x


@pytest.fixture(autouse=True)
def _fp32_convs():
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = old


def ref_stem(x, y, layer, maxdisp):
    return ConvBR_3d.forward(layer, O.cost_volume_ref(x, y, maxdisp))


SHAPES = [
    # (B, C, Hf, Wf, maxdisp, O)
    (2, 12, 6, 40, 48, 12),     # Df = 16
    (1, 12, 5, 96, 192, 12),    # Df = 64 > band, Wf % 4 == 0
    (1, 12, 4, 38, 30, 12),     # Wf % 4 == 2 -> scalar store path
    (1, 12, 3, 12, 48, 12),     # Wf < Df: mostly masked
    (1, 12, 7, 416, 288, 5),    # config-5 width, O != C
    (1, 12, 4, 16, 9, 12),      # Df = 3: classes only, no interior d
    (1, 12, 3, 16, 6, 12),      # Df = 2 -> direct kernel
    (1, 5, 3, 20, 24, 4),       # C != 12 -> direct kernel
]


@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_fused_stem_matches_reference(shape):
    from rag_b200.fused_stem import cv_stem_forward

    b, c, hf, wf, md, o = shape
    g = gen(hash(shape) % 991)
    x, y = randn((b, c, hf, wf), g).cuda(), randn((b, c, hf, wf), g).cuda()
    torch.manual_seed(1)
    layer = ConvBR_3d(2 * c, o).cuda().eval()
    with torch.no_grad():
        layer.bn.running_mean.normal_(0, 0.5)
        layer.bn.running_var.uniform_(0.5, 2.0)
        layer.bn.weight.normal_(1, 0.2)
        layer.bn.bias.normal_(0, 0.3)
        conv_ref = layer.conv(O.cost_volume_ref(x, y, md))
        full_ref = ref_stem(x, y, layer, md)
        scale = layer.bn.weight * torch.rsqrt(layer.bn.running_var + layer.bn.eps)
        shift = layer.bn.bias - layer.bn.running_mean * scale
        for v in (None, 0) + ((1,) if (c == 12 and int(md / 3) >= 3 and wf >= 8) else ()) + ((2,) if (c == 12 and int(md / 3) >= 3 and wf >= 8 and wf % 4 == 0) else ()):
            conv = cv_stem_forward(x, y, layer.conv.weight, maxdisp=md, variant=v)
            assert conv.shape == conv_ref.shape
            err = (conv - conv_ref).abs().max().item() / conv_ref.abs().max().item()
            assert err <= 1e-5, f"variant {v}: conv rel err {err}"
            full = cv_stem_forward(x, y, layer.conv.weight, scale, shift, True, md, variant=v)
            err = (full - full_ref).abs().max().item() / max(full_ref.abs().max().item(), 1e-6)
            assert err <= 1e-5, f"variant {v}: conv+bn+relu rel err {err}"


def test_dropin_stem_forward_paths():
    """stem_forward bound onto a ConvBR_3d-shaped module: fused in eval/no-grad, conv-only fused with
    batch-statistics BN, materialised fallback under autograd -- all equal to the reference composition."""
    from rag_b200.fused_stem import VirtualCostVolume, stem_forward

    g = gen(3)
    md = 48
    x, y = randn((2, 12, 5, 40), g).cuda(), randn((2, 12, 5, 40), g).cuda()
    torch.manual_seed(2)
    layer = ConvBR_3d(24, 12).cuda()
    with torch.no_grad():
        layer.bn.running_mean.normal_(0, 0.5)
        layer.bn.running_var.uniform_(0.5, 2.0)
    # eval, no grad: fully fused
    layer.eval()
    with torch.no_grad():
        out = stem_forward(layer, VirtualCostVolume(x, y, md))
        ref = ref_stem(x, y, layer, md)
    assert (out - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
    # a plain tensor goes through the reference code path unchanged
    with torch.no_grad():
        vol = O.cost_volume_ref(x, y, md)
        assert torch.equal(stem_forward(layer, vol.clone()), ref_stem(x, y, layer, md))
    # training-mode BN, no grad: fused conv + torch BN with batch statistics (running stats updated identically)
    l1, l2 = copy.deepcopy(layer).train(), copy.deepcopy(layer).train()
    with torch.no_grad():
        a = stem_forward(l1, VirtualCostVolume(x, y, md))
        b_ = ref_stem(x, y, l2, md)
    assert (a - b_).abs().max().item() <= 2e-5 * b_.abs().max().item()
    assert torch.allclose(l1.bn.running_mean, l2.bn.running_mean, rtol=1e-5, atol=1e-6)
    # autograd: falls back to the materialised volume, gradients flow to the features and the weights
    xr, yr = x.clone().requires_grad_(True), y.clone().requires_grad_(True)
    l3 = copy.deepcopy(layer).train()
    stem_forward(l3, VirtualCostVolume(xr, yr, md)).sum().backward()
    assert xr.grad is not None and yr.grad is not None and l3.conv.weight.grad is not None


def test_network_forward_with_fused_stem():
    """End to end through the drop-in forward with install(fuse_stem=True)-like wiring on a stand-in network."""
    from rag_b200 import network as N
    from rag_b200.fused_stem import stem_forward
    from rag_b200.modules import Disp

    class Net(nn.Module):
        def __init__(self, md):
            super().__init__()
            self.maxdisp = md
            self.disp = Disp(md)
            self.f = nn.Conv2d(3, 12, 3, stride=3, bias=False)
            self.stem3d0 = nn.ModuleList([ConvBR_3d(24, 12)])
            self.last = nn.Conv3d(12, 1, 3, padding=1, bias=False)

        def feature(self, img, task_arch=None, path=None):
            return self.f(img)

        def matching(self, cost, task_arch=None, path=None):
            return self.last(self.stem3d0[0](cost))

    md = 48
    torch.manual_seed(4)
    net = Net(md).cuda().eval()
    g = gen(8)
    left, right = randn((2, 3, 24, 96), g).cuda(), randn((2, 3, 24, 96), g).cuda()
    with torch.no_grad():
        ref = O.disp_head_ref(net.matching(O.cost_volume_ref(net.feature(left), net.feature(right), md)), md)
        import types

        ops3d = types.SimpleNamespace(ConvBR_3d=ConvBR_3d)
        try:
            N.install(operations_3d=ops3d, fuse_stem=True)
            assert ConvBR_3d.forward is stem_forward
            out = N.network_forward(net, left, right, 0)
            net.rag_b200_fuse_stem = False                      # per-instance opt-out: the materialised path
            out_plain = N.network_forward(net, left, right, 0)
            del net.rag_b200_fuse_stem
            N.install(fuse_stem=False)                          # a later plain install() switches the default off
            assert N._FUSE_STEM is False
        finally:
            N.uninstall()
        assert ConvBR_3d.forward is not stem_forward
    assert (out_plain - ref).abs().max().item() <= 1e-4
    assert (out - ref).abs().max().item() <= 2e-4


def test_golden_from_the_reference_layer():
    """tests/golden/stem_*.npz: the reference's Network.forward volume fed to its own ConvBR_3d(2C, C, 3, 1, 1) in
    eval mode (CPU, fp32)."""
    import glob
    import os

    import numpy as np

    from rag_b200.fused_stem import cv_stem_forward
    from tests.conftest import GOLDEN

    paths = sorted(glob.glob(os.path.join(GOLDEN, "stem_b*.npz")))
    assert paths
    for path in paths:
        z = np.load(path)
        t = lambda k: torch.from_numpy(np.asarray(z[k], dtype=np.float32)).cuda()  # noqa: E731
        scale = t("bn_weight") * torch.rsqrt(t("bn_var") + float(z["bn_eps"]))
        shift = t("bn_bias") - t("bn_mean") * scale
        out = cv_stem_forward(t("x"), t("y"), t("weight"), scale, shift, True, int(z["maxdisp"])).cpu().numpy()
        assert np.abs(out - z["out"]).max() <= 1e-5 * np.abs(z["out"]).max()


def _torch_moments(x, y, w, md):
    """fp64 moments of the fp32 (TF32 off) convolution of the materialised volume, per output channel."""
    from rag_b200.functional import cost_volume

    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        z = F.conv3d(cost_volume(x, y, md), w, None, 1, 1).double()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    return z.mean(dim=(0, 2, 3, 4)), z.var(dim=(0, 2, 3, 4), unbiased=False), z.numel() // z.shape[1]


@pytest.mark.parametrize("shape", [(2, 5, 12, 24), (1, 7, 40, 48), (3, 4, 36, 192), (2, 6, 416, 96)], ids=str)
def test_batch_stats_without_the_volume(shape):
    """First piece of the training path (DESIGN.md section 10): the batch mean / variance a training-mode BatchNorm3d
    after the stem would use, from the collapsed row maps, against the moments of the real convolution output."""
    from rag_b200.fused_stem import cv_stem_batch_stats

    b, hf, wf, md = shape
    g = torch.Generator().manual_seed(sum(shape))
    x = torch.randn(b, 12, hf, wf, generator=g).cuda()
    y = torch.randn(b, 12, hf, wf, generator=g).cuda()
    w = (torch.randn(12, 24, 3, 3, 3, generator=g) * 0.1).cuda()
    mean, var, n = cv_stem_batch_stats(x, y, w, md)
    rmean, rvar, rn = _torch_moments(x, y, w, md)
    assert n == rn
    std = rvar.sqrt()
    assert ((mean - rmean).abs() <= 1e-5 * std + 1e-7).all(), (mean - rmean).abs().max().item()
    assert ((var - rvar).abs() <= 1e-5 * rvar).all(), ((var - rvar).abs() / rvar).max().item()
    m2, v2, _ = cv_stem_batch_stats(x, y, w, md)
    assert torch.equal(mean, m2) and torch.equal(var, v2)          # fixed-order reduction: bitwise repeatable


def test_batch_stats_match_the_reference_running_stat_update():
    """tests/golden/trainstem_*.npz: the reference's ConvBR_3d in train() updated its running statistics from the batch
    moments (momentum 0.1, unbiased variance); ours must reproduce that update."""
    import os

    import numpy as np

    from rag_b200.fused_stem import cv_stem_batch_stats
    from tests.conftest import GOLDEN

    z = np.load(os.path.join(GOLDEN, "trainstem_b2_c12_h5_w12_md24.npz"))
    x, y, w = (torch.from_numpy(z[k]).cuda() for k in ("x", "y", "weight"))
    mean, var, n = cv_stem_batch_stats(x, y, w, int(z["maxdisp"]))
    mom = float(z["bn_momentum"])
    mean1 = (1 - mom) * torch.from_numpy(z["bn_mean0"]).double() + mom * mean.cpu()
    var1 = (1 - mom) * torch.from_numpy(z["bn_var0"]).double() + mom * var.cpu() * n / (n - 1)
    np.testing.assert_allclose(mean1.numpy(), z["bn_mean1"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(var1.numpy(), z["bn_var1"], rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------------------
# training: fused forward + volume-free backward (csrc/cv_stem_train.cu, rag_b200.fused_stem.FusedStemFn)
# ---------------------------------------------------------------------------------------------------------------------
def _mx(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def ref_stem_masked(x, y, layer, maxdisp, mask):
    """The reference composition with the ReLU decision GIVEN (mask = out > 0 of the run under test) and the pre-activation
    returned next to the output.  A gradient through a ReLU is discontinuous in its input: two evaluations that differ by
    one ulp disagree on the handful of elements whose pre-activation is ~0 (7e7 elements at B=4 288x576 -> a few flips, each
    worth O(1) in max-norm), which says nothing about either evaluation's arithmetic.  So: arithmetic is compared with the
    mask fixed, and the mask itself is checked separately (it may differ from the fp64 one only where |pre| is rounding noise)."""
    pre = layer.bn(layer.conv(O.cost_volume_ref(x, y, maxdisp)))
    return pre * mask.to(pre.dtype), pre


def test_training_stem_matches_the_reference_golden():
    """tests/golden/trainstem_*.npz: the reference's own ConvBR_3d(2C, C, 3, 1, 1) in train() on the volume its
    Network.forward builds -- output, gradients w.r.t. both feature maps, the conv weight and the BatchNorm affine
    parameters, running statistics after the step (CPU fp32).  1e-5 max-norm (SURVEY.md section 8a H-3 reading)."""
    import os

    import numpy as np

    from rag_b200.fused_stem import VirtualCostVolume, stem_forward
    from tests.conftest import GOLDEN

    z = np.load(os.path.join(GOLDEN, "trainstem_b2_c12_h5_w12_md24.npz"))
    t = lambda k: torch.from_numpy(z[k]).cuda()  # noqa: E731
    md = int(z["maxdisp"])
    layer = ConvBR_3d(24, 12).cuda().train()
    layer.bn.eps, layer.bn.momentum = float(z["bn_eps"]), float(z["bn_momentum"])
    with torch.no_grad():
        layer.conv.weight.copy_(t("weight")); layer.bn.weight.copy_(t("bn_weight")); layer.bn.bias.copy_(t("bn_bias"))
        layer.bn.running_mean.copy_(t("bn_mean0")); layer.bn.running_var.copy_(t("bn_var0"))
    x, y = t("x").requires_grad_(True), t("y").requires_grad_(True)
    v0 = (layer.bn.running_mean._version, layer.bn.running_var._version)
    out = stem_forward(layer, VirtualCostVolume(x, y, md))
    assert out.grad_fn is not None and "FusedStemFn" in type(out.grad_fn).__name__
    assert layer.bn.running_mean._version > v0[0] and layer.bn.running_var._version > v0[1]      # written in place, as F.batch_norm marks it
    out.backward(t("gout"))
    tol = 1e-5
    assert _mx(out.detach(), t("out")) <= tol
    for got, key in ((x.grad, "gx"), (y.grad, "gy"), (layer.conv.weight.grad, "gweight"), (layer.bn.weight.grad, "gbn_weight"),
                     (layer.bn.bias.grad, "gbn_bias")):
        assert _mx(got, t(key)) <= tol, f"{key}: {_mx(got, t(key)):.3e}"
    np.testing.assert_allclose(layer.bn.running_mean.cpu().numpy(), z["bn_mean1"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(layer.bn.running_var.cpu().numpy(), z["bn_var1"], rtol=1e-5, atol=1e-6)
    assert int(layer.bn.num_batches_tracked) == 1


TRAIN_SHAPES = [
    # (B, Hf, Wf, maxdisp, O)
    (2, 6, 40, 48, 12),       # Df = 16
    (1, 5, 96, 192, 12),      # Df = 64
    (1, 3, 12, 48, 12),       # Wf < Df: mostly masked
    (2, 4, 416, 288, 5),      # config-5 width (4 column chunks), O != C, Df = 96
    (1, 4, 16, 9, 12),        # Df = 3: no interior d
    (1, 9, 132, 96, 32),      # Wf just over one 128-column chunk, O = 32
]


@pytest.mark.parametrize("shape", TRAIN_SHAPES, ids=str)
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_training_stem_forward_backward_vs_fp64(shape, mode):
    """Fused layer vs the materialised composition evaluated in fp64 on the GPU (volume -> Conv3d -> BatchNorm3d -> ReLU, autograd)
    and vs the same composition in fp32 (what the reference runs): ours must be within 1e-5 max-norm of fp64 on every gradient,
    i.e. no further from the truth than the fp32 reference is."""
    from rag_b200.fused_stem import VirtualCostVolume, stem_forward

    b, hf, wf, md, o = shape
    g = gen(hash((shape, mode)) % 997)
    layer = ConvBR_3d(24, o).cuda()
    with torch.no_grad():
        layer.bn.weight.copy_(0.5 + torch.rand(o, generator=g)); layer.bn.bias.copy_(0.3 * torch.randn(o, generator=g))
        layer.bn.running_mean.copy_(0.2 * torch.randn(o, generator=g)); layer.bn.running_var.copy_(0.5 + torch.rand(o, generator=g))
    layer.train(mode == "train")
    x0, y0 = randn((b, 12, hf, wf), g).cuda(), randn((b, 12, hf, wf), g).cuda()
    gout = randn((b, o, int(md / 3), hf, wf), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)           # some exact zeros upstream
    state = copy.deepcopy(layer.state_dict())

    def run(fn, dtype):
        lay = copy.deepcopy(layer).to(dtype)
        lay.load_state_dict({k: v.to(dtype) if v.is_floating_point() else v for k, v in state.items()})
        x, y = x0.to(dtype).clone().requires_grad_(True), y0.to(dtype).clone().requires_grad_(True)
        out = fn(lay, x, y)
        pre = None
        if isinstance(out, tuple):
            out, pre = out
        out.backward(gout.to(dtype))
        return [out.detach(), x.grad, y.grad, lay.conv.weight.grad, lay.bn.weight.grad, lay.bn.bias.grad, lay.bn.running_mean, lay.bn.running_var], pre

    ours, _ = run(lambda lay, x, y: stem_forward(lay, VirtualCostVolume(x, y, md)), torch.float32)
    mask = ours[0] > 0
    ref64, pre64 = run(lambda lay, x, y: ref_stem_masked(x, y, lay, md, mask), torch.float64)
    ref32, _ = run(lambda lay, x, y: ref_stem_masked(x, y, lay, md, mask), torch.float32)
    flips = (pre64.detach() > 0) != mask
    assert not flips.any() or pre64.detach()[flips].abs().max().item() <= 1e-5, "the ReLU decision differs from fp64 beyond rounding noise"
    names = ["out", "gx", "gy", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
    for n, a, r32, r64 in zip(names, ours, ref32, ref64):
        e_ours, e_ref = _mx(a, r64), _mx(r32, r64)
        assert e_ours <= 1e-5, f"{n}: ours vs fp64 {e_ours:.3e} (fp32 reference vs fp64: {e_ref:.3e})"


def test_training_stem_partial_gradients_and_determinism():
    """Frozen weight (only the feature maps want a gradient), frozen features (only the layer's parameters), and bitwise
    repeatability of the whole backward (fixed-order reductions, no atomics)."""
    from rag_b200.fused_stem import VirtualCostVolume, stem_forward

    g = gen(5)
    md = 96
    layer = ConvBR_3d(24, 12).cuda().train()
    x0, y0 = randn((2, 12, 7, 64), g).cuda(), randn((2, 12, 7, 64), g).cuda()
    gout = randn((2, 12, 32, 7, 64), g).cuda()
    state = copy.deepcopy(layer.state_dict())

    def run(req_in, req_par):
        layer.load_state_dict(state)
        layer.zero_grad(set_to_none=True)
        for p in layer.parameters():
            p.requires_grad_(req_par)
        x, y = x0.clone().requires_grad_(req_in), y0.clone().requires_grad_(req_in)
        out = stem_forward(layer, VirtualCostVolume(x, y, md))
        out.backward(gout)
        return x.grad, y.grad, layer.conv.weight.grad, layer.bn.weight.grad, layer.bn.bias.grad

    full = run(True, True)
    again = run(True, True)
    for a, b_ in zip(full, again):
        assert torch.equal(a, b_)
    only_in = run(True, False)
    assert torch.equal(only_in[0], full[0]) and torch.equal(only_in[1], full[1]) and only_in[2] is None and only_in[3] is None
    only_par = run(False, True)
    assert only_par[0] is None and all(torch.equal(a, b_) for a, b_ in zip(only_par[2:], full[2:]))
    for p in layer.parameters():
        p.requires_grad_(True)


def test_training_stem_at_the_training_config_without_the_volume():
    """BASELINE config 3 (B=4, 288x576): parity with the PyTorch CUDA layers on the materialised volume (fp32, TF32 off) and
    the memory the step needs: the fused path must never hold a [B,24,Df,Hf,Wf]-sized tensor (453 MB here)."""
    from rag_b200 import functional as F_
    from rag_b200.fused_stem import VirtualCostVolume, stem_forward

    b, hf, wf, md, o = 4, 96, 192, 192, 12
    g = gen(6)
    layer = ConvBR_3d(24, o).cuda().train()
    x0, y0 = randn((b, 12, hf, wf), g).cuda(), randn((b, 12, hf, wf), g).cuda()
    gout = randn((b, o, 64, hf, wf), g).cuda()
    state = copy.deepcopy(layer.state_dict())
    vol_bytes = b * 24 * 64 * hf * wf * 4

    def run(fn):
        layer.load_state_dict(state)
        layer.zero_grad(set_to_none=True)
        x, y = x0.clone().requires_grad_(True), y0.clone().requires_grad_(True)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = fn(x, y)
        out.backward(gout)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        res = [out.detach().clone(), x.grad, y.grad, layer.conv.weight.grad.clone(), layer.bn.weight.grad.clone(), layer.bn.bias.grad.clone(),
               layer.bn.running_mean.clone(), layer.bn.running_var.clone()]
        del out
        return res, peak

    ref, ref_peak = run(lambda x, y: ConvBR_3d.forward(layer, F_.cost_volume(x, y, md)))
    ours, our_peak = run(lambda x, y: stem_forward(layer, VirtualCostVolume(x, y, md)))
    names = ["out", "gx", "gy", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
    for n in (0, 6, 7):                                     # forward quantities: directly comparable
        assert _mx(ours[n], ref[n]) <= 1e-5, f"{names[n]}: {_mx(ours[n], ref[n]):.3e}"
    # backward: the ReLU decisions of the two fp32 forwards disagree on a few of the 7e7 elements (pre-activation ~ 0), each worth
    # O(1e-2) of max-norm in gx/gy -- so the arithmetic is compared with the mask FIXED to ours, against fp64 (see ref_stem_masked)
    mask = ours[0] > 0
    n_flip = int(((ref[0] > 0) != mask).sum())
    assert n_flip <= 200, n_flip
    lay64 = copy.deepcopy(layer).double()
    lay64.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in state.items()})
    x64, y64 = x0.double().requires_grad_(True), y0.double().requires_grad_(True)
    out64, pre64 = ref_stem_masked(x64, y64, lay64, md, mask)
    out64.backward(gout.double())
    flips = (pre64.detach() > 0) != mask
    assert not flips.any() or pre64.detach()[flips].abs().max().item() <= 1e-5
    want = [out64.detach(), x64.grad, y64.grad, lay64.conv.weight.grad, lay64.bn.weight.grad, lay64.bn.bias.grad]
    errs = {n: _mx(a, r) for n, a, r in zip(names, ours, want)}
    for n, e in errs.items():
        assert e <= 1e-5, f"{n}: {e:.3e} vs fp64 with the same ReLU mask"
    print(f"\ntraining stem at B=4 288x576 vs fp64 (mask fixed): {errs}; ReLU decisions differing from the fp32 cuDNN forward: {n_flip} of {mask.numel()}")
    del lay64, x64, y64, out64, pre64, want
    # out (226 MB) + the recomputed pre-activation (226 MB) + maps/partials: well under the volume + conv output + their gradients
    assert our_peak < 0.45 * ref_peak, (our_peak, ref_peak)
    assert our_peak < 3 * vol_bytes // 2 + (64 << 20), (our_peak, vol_bytes)
    print(f"\ntraining stem at B=4 288x576: peak extra memory fused {our_peak / 2**20:.0f} MiB vs materialised {ref_peak / 2**20:.0f} MiB")


def test_training_stem_falls_back_where_the_kernels_do_not_apply():
    """Widths that are not a multiple of 4, a layer without ReLU or without BatchNorm: stem_forward must materialise the volume
    and run the reference layer (same result as the reference composition, gradients through autograd), never raise."""
    from rag_b200 import _cabi
    from rag_b200.fused_stem import VirtualCostVolume, stem_forward

    g = gen(12)
    for (wf, bn, relu) in [(38, True, True), (40, True, False), (40, False, True)]:
        layer = ConvBR_3d(24, 12, bn=bn, relu=relu).cuda().train()
        x0, y0 = randn((1, 12, 4, wf), g).cuda(), randn((1, 12, 4, wf), g).cuda()
        x, y = x0.clone().requires_grad_(True), y0.clone().requires_grad_(True)
        state = copy.deepcopy(layer.state_dict())
        out = stem_forward(layer, VirtualCostVolume(x, y, 30))
        assert "FusedStemFn" not in type(out.grad_fn).__name__
        out.sum().backward()
        layer.load_state_dict(state)
        xr, yr = x0.clone().requires_grad_(True), y0.clone().requires_grad_(True)
        ref = ref_stem(xr, yr, layer, 30)
        ref.sum().backward()
        assert _mx(out.detach(), ref.detach()) <= 1e-5 and _mx(x.grad, xr.grad) <= 1e-4 and _mx(y.grad, yr.grad) <= 1e-4
    assert _cabi.launch_count() > 0
