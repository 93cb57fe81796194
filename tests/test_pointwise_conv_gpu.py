"""The Matching Net's pointwise ConvBR_3d layers on csrc/conv3d_pw.cu (rag_b200/pointwise_conv.py) against fp64 compositions
of the reference layer: Conv3d(C -> O, 1x1x1, bias=False) -> BatchNorm3d -> ReLU (operations_3d.py:31-47).

Tolerance: max-norm relative 1e-5 of fp64, the bar of tests/test_matching_conv_gpu.py (our kernels sum the C products of an
output, and the weight gradient's voxels, in another order than cuDNN, all in fp32 with an fp64 final pass)."""
import copy
import zlib

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests._util import gen, randn

pytestmark = pytest.mark.gpu
PAIRS = [(1, 1), (5, 3), (7, 29), (12, 4), (24, 12), (48, 24), (64, 32)]


class ConvBR_3d(nn.Module):
    """Same fields / forward as the reference's ConvBR_3d (operations_3d.py:31-47); pointwise by default."""

    def __init__(self, c_in, c_out, kernel=1, stride=1, pad=0, bn=True, relu=True, bias=False, affine=True):
        super().__init__()
        self.relu = relu
        self.use_bn = bn
        self.conv = nn.Conv3d(c_in, c_out, kernel, stride=stride, padding=pad, bias=bias)
        self.bn = nn.BatchNorm3d(c_out, affine=affine)

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


@pytest.fixture(autouse=True)
def _small_inputs_on_the_kernels(monkeypatch):
    """The kernels are tested at small sizes too: the volume floor of the routing (pointwise_conv.MIN_VOXELS) is off here,
    and test_small_volumes_stay_on_cudnn checks it."""
    from rag_b200 import pointwise_conv

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)


def _mx(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def _layer(c, o, g, k=1, pad=0):
    lay = ConvBR_3d(c, o, k, 1, pad).cuda()
    with torch.no_grad():
        lay.bn.weight.copy_(0.5 + torch.rand(o, generator=g)); lay.bn.bias.copy_(0.3 * torch.randn(o, generator=g))
        lay.bn.running_mean.copy_(0.2 * torch.randn(o, generator=g)); lay.bn.running_var.copy_(0.5 + torch.rand(o, generator=g))
    return lay


# (B, D, H, W): D*H*W % 4 == 0, and S not a multiple of the forward's 512-voxel CTA or the backward's 256-voxel tile
FWD_SHAPES = [(2, 1, 1, 4), (2, 3, 5, 12), (3, 2, 9, 20), (1, 10, 5, 132)]


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", FWD_SHAPES, ids=str)
def test_forward_vs_fp64(pair, shape):
    from rag_b200.pointwise_conv import conv3d_pw_forward, convbr_forward, qualifies

    c, o = pair
    b, d, h, w = shape
    g = gen(hash((pair, shape)) % 1009)
    x = randn((b, c, d, h, w), g).cuda()
    wt = randn((o, c, 1, 1, 1), g).cuda() * 0.3
    z = conv3d_pw_forward(x, wt)
    assert _mx(z, F.conv3d(x.double(), wt.double())) <= 1e-5
    # eval-mode BatchNorm folded + ReLU against the mirror layer in fp64
    lay = _layer(c, o, g).eval()
    lay64 = copy.deepcopy(lay).double()
    with torch.no_grad():
        assert qualifies(lay, x)
        out = convbr_forward(lay, x)
        pre = lay64.bn(lay64.conv(x.double()))
    assert ((out.double() - F.relu(pre)).abs().max() / pre.abs().max()).item() <= 1e-5


def test_forward_full_level3_shape():
    """One full level-3 layer at B=4 288x576: [4,12,64,96,192] -> 4."""
    from rag_b200.pointwise_conv import conv3d_pw_forward

    g = gen(5)
    x = randn((4, 12, 64, 96, 192), g).cuda()
    wt = randn((4, 12, 1, 1, 1), g).cuda() * 0.3
    z = conv3d_pw_forward(x, wt)
    assert _mx(z, F.conv3d(x.double(), wt.double())) <= 1e-5


def _run(layer, x0, gout, fn, dtype, req_x=True, only_bn=False):
    lay = copy.deepcopy(layer).to(dtype)
    if only_bn:
        lay.conv.weight.requires_grad_(False)
    x = x0.detach().to(dtype).clone().requires_grad_(req_x)
    out = fn(lay, x)
    pre = None
    if isinstance(out, tuple):
        out, pre = out
    out.backward(gout.to(dtype))
    return [out.detach(), x.grad, lay.conv.weight.grad, lay.bn.weight.grad, lay.bn.bias.grad,
            lay.bn.running_mean.clone(), lay.bn.running_var.clone()], pre


def _masked(lay, x, mask):
    """The reference composition with the ReLU decision GIVEN (mask = out > 0 of the run under test)."""
    pre = lay.bn(lay.conv(x))
    return pre * mask.to(pre.dtype), pre


TRAIN_SHAPES = [(2, 3, 9, 36), (1, 10, 12, 68), (3, 5, 7, 8)]   # (B, D, H, W); D >= 3 and 8 <= W for the BatchNorm helpers


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", TRAIN_SHAPES, ids=str)
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_training_vs_fp64(pair, shape, mode):
    from rag_b200.pointwise_conv import pointwise_forward

    c, o = pair
    b, d, h, w = shape
    g = gen(zlib.crc32(repr((pair, shape, mode)).encode()) % 991)      # not hash(): a str's hash changes from run to run
    layer = _layer(c, o, g).train(mode == "train")
    x0 = randn((b, c, d, h, w), g).cuda()
    gout = randn((b, o, d, h, w), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)
    ours, _ = _run(layer, x0, gout, pointwise_forward, torch.float32)
    mask = ours[0] > 0
    ref64, pre64 = _run(layer, x0, gout, lambda lay, x: _masked(lay, x, mask), torch.float64)
    flips = (pre64.detach() > 0) != mask
    assert not flips.any() or pre64.detach()[flips].abs().max().item() <= 1e-5, "ReLU decision differs from fp64 beyond rounding"
    names = ["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
    for n, a, r in zip(names, ours, ref64):
        if n == "gweight" and c == 1:
            # one input channel: each weight's gradient is one dot product over all B*D*H*W voxels, so its relative error
            # measures cancellation rather than the kernel (under batch statistics the layer is even invariant to the weight's
            # scale: the exact gradient is ~0, eps alone keeps it off zero); bound it by the summed |gz x| instead
            lay64, x64 = copy.deepcopy(layer).double(), x0.double()
            z64 = lay64.conv(x64).detach().requires_grad_(True)
            (lay64.bn(z64) * mask.double()).backward(gout.double())
            bound = 1e-5 * (z64.grad.abs() * x64.abs()).sum().item()
            assert (a.double() - r).abs().max().item() <= bound, n
            continue
        assert _mx(a, r) <= 1e-5, f"{n}: {_mx(a, r):.3e}"
    # only the BatchNorm parameters trainable, the input not requiring grad: no convolution backward at all
    from rag_b200 import _cabi

    n0 = _cabi.launch_count()
    ours2, _ = _run(layer, x0, gout, pointwise_forward, torch.float32, req_x=False, only_bn=True)
    # forward: conv + (batch statistics: moments (2)) + finalize + normalise; backward: sums (2) + consts
    assert _cabi.launch_count() - n0 == (5 if mode == "train" else 3) + 3
    assert ours2[1] is None and ours2[2] is None
    for i in (3, 4):
        assert _mx(ours2[i], ref64[i]) <= 1e-5
    # the input not requiring grad, the weight trainable: gweight still right
    ours3, _ = _run(layer, x0, gout, pointwise_forward, torch.float32, req_x=False)
    assert ours3[1] is None and torch.equal(ours3[2], ours[2])          # the same kernel, with the data gradient skipped


# (pair, (B, D, H, W)) where the fused backward's fixed grid of G CTAs walks each CTA over several 256-voxel tiles (t =
# blockIdx.x, +G, ...): the weight-gradient sums are carried across tiles and the tile buffers reused, as at the routed shapes
MULTI_TILE = [((64, 32), (2, 16, 48, 128)), ((12, 4), (2, 32, 128, 128)), ((24, 12), (4, 32, 64, 96))]


@pytest.mark.parametrize("case", MULTI_TILE, ids=str)
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_training_many_tiles_per_cta(case, mode):
    from rag_b200 import _cabi
    from rag_b200.pointwise_conv import pointwise_forward

    (c, o), (b, d, h, w) = case
    grid = _cabi.lib().rag_conv3d_pw_bwd_workspace_bytes(b, c, o, d, h, w) // (4 * o * c)   # one partial per CTA and weight
    n_tiles = b * -(-(d * h * w) // 256)
    assert n_tiles >= 4 * grid, (n_tiles, grid)
    g = gen(hash((case, mode)) % 997)
    layer = _layer(c, o, g).train(mode == "train")
    x0 = randn((b, c, d, h, w), g).cuda()
    gout = randn((b, o, d, h, w), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)
    ours, _ = _run(layer, x0, gout, pointwise_forward, torch.float32)
    mask = ours[0] > 0
    ref64, pre64 = _run(layer, x0, gout, lambda lay, x: _masked(lay, x, mask), torch.float64)
    flips = (pre64.detach() > 0) != mask
    assert not flips.any() or pre64.detach()[flips].abs().max().item() <= 1e-5, "ReLU decision differs from fp64 beyond rounding"
    for n, a, r in zip(["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"], ours, ref64):
        assert _mx(a, r) <= 1e-5, f"{n}: {_mx(a, r):.3e}"
    again, _ = _run(layer, x0, gout, pointwise_forward, torch.float32)
    for n, u, v in zip(["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"], ours, again):
        assert torch.equal(u, v), n


def test_momentum_none_and_version_bumps():
    """momentum=None (cumulative average) and the running buffers' version counters move as F.batch_norm moves them."""
    from rag_b200.pointwise_conv import pointwise_forward

    g = gen(7)
    lay = _layer(24, 12, g).train()
    lay.bn.momentum = None
    ref = copy.deepcopy(lay)
    x = randn((2, 24, 4, 6, 16), g).cuda()
    for step in range(3):
        v0 = (lay.bn.running_mean._version, lay.bn.running_var._version)
        with torch.no_grad():
            out = pointwise_forward(lay, x + step)
            rout = ref(x + step)
        assert lay.bn.running_mean._version > v0[0] and lay.bn.running_var._version > v0[1]
        assert _mx(out, rout) <= 1e-5
    assert int(lay.bn.num_batches_tracked) == int(ref.bn.num_batches_tracked) == 3
    assert torch.allclose(lay.bn.running_mean, ref.bn.running_mean, rtol=1e-5, atol=1e-6)
    assert torch.allclose(lay.bn.running_var, ref.bn.running_var, rtol=1e-5, atol=1e-6)


def test_backward_is_bitwise_repeatable_and_counted():
    from rag_b200 import _cabi
    from rag_b200.pointwise_conv import pointwise_forward, qualifies

    g = gen(11)
    layer = _layer(48, 24, g).train()
    x0 = randn((2, 48, 16, 24, 48), g).cuda()
    gout = randn((2, 24, 16, 24, 48), g).cuda()
    assert qualifies(layer, x0.clone().requires_grad_(True))
    n0 = _cabi.launch_count()
    a, _ = _run(layer, x0, gout, pointwise_forward, torch.float32)
    launches = _cabi.launch_count() - n0
    # fwd conv + moments (2) + finalize + normalise | bwd sums (2) + consts + fused backward + weight-gradient final
    assert launches == 10, launches
    b_, _ = _run(layer, x0, gout, pointwise_forward, torch.float32)
    for u, v in zip(a, b_):
        assert torch.equal(u, v)
    layer.eval()
    with torch.no_grad():
        n0 = _cabi.launch_count()
        e1 = pointwise_forward(layer, x0)
        assert _cabi.launch_count() - n0 == 1
        assert torch.equal(e1, pointwise_forward(layer, x0))


def test_routing_launches_and_fallthrough_parity():
    """Qualifying layers run the kernels; excluded ones take none and give the fallthrough's result bit for bit."""
    from rag_b200 import _cabi
    from rag_b200.fused_stem import stem_forward
    from rag_b200.matching_conv import matching_forward
    from rag_b200.pointwise_conv import pointwise_forward, pointwise_matching_forward

    g = gen(13)
    x = randn((2, 48, 6, 10, 40), g).cuda()
    good = _layer(48, 24, g).eval()
    x12 = randn((2, 12, 6, 10, 40), g).cuda()
    excluded = {                                  # name: (layer, its input)
        "3x3x3 (48,24)": (ConvBR_3d(48, 24, 3, 1, 1).cuda().eval(), x),
        "stride 2": (ConvBR_3d(48, 24, 1, 2, 0).cuda().eval(), x),
        "padding 1": (ConvBR_3d(48, 24, 1, 1, 1).cuda().eval(), x),
        "bias": (ConvBR_3d(48, 24, bias=True).cuda().eval(), x),
        "O > 32": (ConvBR_3d(48, 33).cuda().eval(), x),
        "no bn": (ConvBR_3d(48, 24, bn=False).cuda().eval(), x),
        "affine-free bn": (ConvBR_3d(48, 24, affine=False).cuda().eval(), x),
        "fp64": (ConvBR_3d(48, 24).cuda().double().eval(), x.double()),
        "S % 4 != 0": (ConvBR_3d(48, 24).cuda().eval(), randn((1, 48, 3, 3, 3), g).cuda()),
    }
    with torch.no_grad():
        n0 = _cabi.launch_count()
        out = pointwise_forward(good, x)
        assert _cabi.launch_count() - n0 == 1
        assert _mx(out, stem_forward(good, x.clone())) <= 1e-5
        for name, (lay, xi) in excluded.items():
            n0 = _cabi.launch_count()
            out = pointwise_forward(lay, xi)
            assert _cabi.launch_count() - n0 == 0, name
            assert torch.equal(out, stem_forward(lay, xi.clone())), name
        # a 3x3x3 interior layer: no conv3d_cc launch under the pointwise-only binding, its usual one under both flags
        cc = _layer(12, 12, g, k=3, pad=1).eval()
        n0 = _cabi.launch_count()
        out = pointwise_forward(cc, x12)
        assert _cabi.launch_count() - n0 == 0
        assert torch.equal(out, stem_forward(cc, x12.clone()))
        n0 = _cabi.launch_count()
        out = pointwise_matching_forward(cc, x12)
        assert _cabi.launch_count() - n0 == 1
        assert torch.equal(out, matching_forward(cc, x12))
    # train(): batch statistics through the kernels, same result as the flag-off (cuDNN) path within the tolerance
    l1, l2 = copy.deepcopy(good).train(), copy.deepcopy(good).train()
    v0 = (l1.bn.running_mean._version, l1.bn.running_var._version)
    with torch.no_grad():
        o1, o2 = pointwise_forward(l1, x), stem_forward(l2, x.clone())
    assert l1.bn.running_mean._version > v0[0] and l1.bn.running_var._version > v0[1]
    assert _mx(o1, o2) <= 1e-5
    assert torch.allclose(l1.bn.running_mean, l2.bn.running_mean, rtol=1e-5, atol=1e-6)
    assert torch.allclose(l1.bn.running_var, l2.bn.running_var, rtol=1e-5, atol=1e-6)
    assert int(l1.bn.num_batches_tracked) == int(l2.bn.num_batches_tracked) == 1


def test_small_volumes_stay_on_cudnn(monkeypatch):
    """Below MIN_VOXELS (B*D*H*W) a qualifying layer takes the fallthrough; at and above it, the kernel."""
    from rag_b200 import _cabi, pointwise_conv
    from rag_b200.fused_stem import stem_forward
    from rag_b200.pointwise_conv import pointwise_forward, qualifies

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 2 ** 17)
    g = gen(23)
    lay = _layer(48, 24, g).eval()
    small = randn((4, 48, 16, 24, 48), g).cuda()        # last_12_3d at B=4 288x576: 73,728 voxels
    big = randn((2, 48, 16, 64, 64), g).cuda()          # 131,072 voxels
    with torch.no_grad():
        assert not qualifies(lay, small) and qualifies(lay, big)
        n0 = _cabi.launch_count()
        out = pointwise_forward(lay, small)
        assert _cabi.launch_count() - n0 == 0
        assert torch.equal(out, stem_forward(lay, small.clone()))
        n0 = _cabi.launch_count()
        pointwise_forward(lay, big)
        assert _cabi.launch_count() - n0 == 1


def test_cuda_graph_capture_replays_bit_exact():
    from rag_b200.pointwise_conv import pointwise_forward

    g = gen(17)
    layer = _layer(24, 12, g).eval()
    x = randn((2, 24, 8, 12, 64), g).cuda().requires_grad_(True)
    gout = randn((2, 12, 8, 12, 64), g).cuda()

    def step():
        layer.zero_grad(set_to_none=True)
        x.grad = None
        out = pointwise_forward(layer, x)
        out.backward(gout)
        return out

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = step().detach().clone()
        e_gx, e_gw = x.grad.clone(), layer.conv.weight.grad.clone()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    layer.zero_grad(set_to_none=True)
    x.grad = None
    with torch.cuda.graph(graph):
        out = pointwise_forward(layer, x)
        out.backward(gout)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out.detach(), eager)
    assert torch.equal(x.grad, e_gx) and torch.equal(layer.conv.weight.grad, e_gw)


GUARD = 4096
CANARY = -12345.678


def _window(n):
    buf = torch.full((n + 2 * GUARD,), CANARY, device="cuda")
    return buf, buf[GUARD:GUARD + n]


def _intact(buf, n):
    return bool((buf[:GUARD] == CANARY).all()) and bool((buf[GUARD + n:] == CANARY).all())


@pytest.mark.parametrize("pair", [(5, 3), (48, 24), (64, 32)], ids=str)
def test_guard_bands(pair):
    """out, gin and gw through the raw ABI, each inside canary bands; the backward's consts are those of an identity
    BatchNorm without ReLU (a = scale = 1, every other entry 0 except rstd = 1, shift = +inf so the ReLU never clamps), so
    the gradient at the convolution output is g itself."""
    from rag_b200 import _cabi

    L = _cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    c, o = pair
    b, d, h, w = 2, 3, 9, 68
    g = gen(19)
    x = randn((b, c, d, h, w), g).cuda()
    gz = randn((b, o, d, h, w), g).cuda()
    z = torch.zeros_like(gz)
    wt = randn((o, c, 1, 1, 1), g).cuda()
    consts = torch.tensor([1.0, 0.0, 0.0, 1.0, float("inf"), 0.0, 1.0], device="cuda").repeat(o, 1).contiguous()
    ob, out = _window(b * o * d * h * w)
    gb, gin = _window(b * c * d * h * w)
    wb, gw = _window(o * c)
    ws = torch.empty(int(L.rag_conv3d_pw_bwd_workspace_bytes(b, c, o, d, h, w)) // 4, device="cuda")
    assert L.rag_conv3d_pw_fwd(x.data_ptr(), wt.data_ptr(), None, None, 1, out.data_ptr(), b, c, o, d, h, w, st) == 0
    assert L.rag_conv3d_pw_bwd(gz.data_ptr(), z.data_ptr(), consts.data_ptr(), x.data_ptr(), wt.data_ptr(), gin.data_ptr(),
                               gw.data_ptr(), ws.data_ptr(), b, c, o, d, h, w, st) == 0
    torch.cuda.synchronize()
    assert _intact(ob, out.numel()) and _intact(gb, gin.numel()) and _intact(wb, gw.numel())
    x64, gz64, w64 = x.double(), gz.double(), wt.double()
    assert _mx(out.view(b, o, d, h, w), F.relu(F.conv3d(x64, w64))) <= 1e-5
    x64.requires_grad_(True); w64.requires_grad_(True)
    F.conv3d(x64, w64).backward(gz64)
    assert _mx(gin.view(b, c, d, h, w), x64.grad) <= 1e-5
    assert _mx(gw.view(o, c, 1, 1, 1), w64.grad) <= 1e-5


def test_pointwise_convs_on_the_real_network():
    """install(..., fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True) on the reference's own Network:
    the pointwise kernels are launched in eval and in training; eval forward within 1e-3 px of the unpatched network;
    training gradients as close to the fp64 network as the unpatched fp32 reference is, within a factor 4 (the criterion of
    test_matching_conv_gpu.test_matching_convs_on_the_real_network).  Skips without oracle/_ref."""
    import os
    import sys
    from copy import deepcopy

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle import refimport as R

    if not R.available():
        pytest.skip("the unmodified reference is not installed in oracle/_ref")
    from rag_b200 import _cabi
    from rag_b200 import network as N

    ref = R.import_reference()
    N.uninstall()
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(3)
    net = ref.rag_model.Network(R.make_genotype(ref, 3), "cuda").cuda().train()
    g = torch.Generator().manual_seed(6)
    H, W = 96, 192
    left, right, w = (torch.randn(2, 3, H, W, generator=g).cuda(), torch.randn(2, 3, H, W, generator=g).cuda(),
                      torch.randn(2, H, W, generator=g).cuda())
    call = lambda: net.forward(left, right, 0, net.arch_init)  # noqa: E731
    for m in net.modules():
        if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
            m.momentum = None
    with torch.no_grad():
        for _ in range(2):
            call()
    net.eval()
    seen = {}
    h = net.last_3_3d[0].register_forward_hook(lambda m, i, o: seen.__setitem__("c", o.detach()))
    with torch.no_grad():
        call()
    h.remove()
    with torch.no_grad():
        net.last_3_3d[0].conv.weight.mul_(1.0 / seen["c"].std().item())
        ref_out = call()

    def launches(fn):
        n0 = _cabi.launch_count()
        r = fn()
        return r, _cabi.launch_count() - n0

    def fwd():
        with torch.no_grad():
            return call()

    # the test's network is small: the autouse fixture has lifted the routing's volume floor, so its pointwise layers qualify
    flags = dict(fuse_stem=True, upsample=True, matching_convs=True)
    try:
        N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, **flags)
        _, base_eval = launches(fwd)
        N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, pointwise_convs=True, **flags)
        assert ref.operations_3d.ConvBR_3d.forward.__module__ == "rag_b200.pointwise_conv"
        out, n_eval = launches(fwd)
        assert n_eval > base_eval, f"no pointwise ConvBR_3d took the kernels in eval() ({n_eval} vs {base_eval} launches)"
        assert (out - ref_out).abs().max().item() <= 1e-3
        net.train()
        state = deepcopy(net.state_dict())

        def fwd_bwd():
            net.load_state_dict(state)
            net.zero_grad(set_to_none=True)
            (call() * w).sum().backward()
            return {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}

        got_g, n_train = launches(fwd_bwd)
        N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, **flags)
        _, base_train = launches(fwd_bwd)
        assert n_train > base_train, f"no pointwise ConvBR_3d took the kernels in train() ({n_train} vs {base_train} launches)"
        N.uninstall()
        ref_g = fwd_bwd()
        net64 = deepcopy(net).double()
        net64.load_state_dict({k: (v.double() if v.is_floating_point() else v) for k, v in state.items()})
        net64.zero_grad(set_to_none=True)
        (net64.forward(left.double(), right.double(), 0, net64.arch_init) * w.double()).sum().backward()
        g64 = {n: p.grad for n, p in net64.named_parameters() if p.grad is not None}
        assert set(g64) == set(got_g) == set(ref_g)

        def errs(gg):
            e = sorted(((gg[n].double() - g64[n]).norm() / g64[n].norm().clamp_min(1e-30)).item() for n in g64)
            return e[len(e) // 2], e[-1]

        (ref_med, ref_max), (got_med, got_max) = errs(ref_g), errs(got_g)
        assert got_med <= 4 * ref_med + 1e-5 and got_max <= 4 * ref_max + 1e-4
    finally:
        N.uninstall()
        torch.backends.cuda.matmul.allow_tf32 = old_tf32
