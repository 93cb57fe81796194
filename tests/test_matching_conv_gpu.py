"""The Matching Net's interior ConvBR_3d layers on csrc/conv3d_cc.cu (rag_b200/matching_conv.py) against fp64 compositions
of the reference layer: Conv3d(C -> O, 3, pad 1, bias=False) -> BatchNorm3d -> ReLU (operations_3d.py:31-47).

Tolerance: max-norm relative 1e-5 of fp64, the bar of tests/test_fused_stem_gpu.py (our kernels sum the 27*C products of an
output, and the weight gradient's positions, in another order than cuDNN, all in fp32 with an fp64 final pass)."""
import copy

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests._util import gen, randn

pytestmark = pytest.mark.gpu
PAIRS = [(4, 4), (8, 8), (12, 12)]


class ConvBR_3d(nn.Module):
    """Same fields / forward as the reference's ConvBR_3d (operations_3d.py:31-47)."""

    def __init__(self, c_in, c_out, kernel=3, stride=1, pad=1, bn=True, relu=True, bias=False, affine=True):
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


def _mx(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def _layer(c, o, g):
    lay = ConvBR_3d(c, o).cuda()
    with torch.no_grad():
        lay.bn.weight.copy_(0.5 + torch.rand(o, generator=g)); lay.bn.bias.copy_(0.3 * torch.randn(o, generator=g))
        lay.bn.running_mean.copy_(0.2 * torch.randn(o, generator=g)); lay.bn.running_var.copy_(0.5 + torch.rand(o, generator=g))
    return lay


TAIL_SHAPES = [(2, 1, 11, 36), (3, 2, 9, 20), (2, 3, 17, 68), (1, 10, 5, 132)]   # (B, D, H, W): tails in every dimension


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", TAIL_SHAPES, ids=str)
def test_forward_vs_fp64(pair, shape):
    from rag_b200.matching_conv import conv3d_cc_forward

    c, o = pair
    b, d, h, w = shape
    g = gen(hash((pair, shape)) % 1009)
    x = randn((b, c, d, h, w), g).cuda()
    wt = randn((o, c, 3, 3, 3), g).cuda() * 0.2
    z = conv3d_cc_forward(x, wt)
    ref = F.conv3d(x.double(), wt.double(), padding=1)
    assert _mx(z, ref) <= 1e-5
    # eval-mode BatchNorm folded + ReLU against the mirror layer in fp64
    lay = _layer(c, o, g).eval()
    from rag_b200.matching_conv import convbr_forward, qualifies

    lay64 = copy.deepcopy(lay).double()
    with torch.no_grad():
        assert qualifies(lay, x)
        out = convbr_forward(lay, x)
        pre = lay64.bn(lay64.conv(x.double()))
    # relative to the pre-activation's max-norm: the ReLU can zero the largest values of a small tensor
    assert ((out.double() - F.relu(pre)).abs().max() / pre.abs().max()).item() <= 1e-5


@pytest.mark.parametrize("pair", [(4, 4)], ids=str)
def test_forward_full_level3_shape(pair):
    """One full level-3 op at B=4 288x576: [4,4,64,96,192]."""
    from rag_b200.matching_conv import conv3d_cc_forward

    c, o = pair
    g = gen(5)
    x = randn((4, c, 64, 96, 192), g).cuda()
    wt = randn((o, c, 3, 3, 3), g).cuda() * 0.2
    z = conv3d_cc_forward(x, wt)
    ref = F.conv3d(x.double(), wt.double(), padding=1)
    assert _mx(z, ref) <= 1e-5


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
    """The reference composition with the ReLU decision GIVEN (mask = out > 0 of the run under test): two correct fp32
    forwards may disagree on elements whose pre-activation is ~0; the mask itself is checked separately."""
    pre = lay.bn(lay.conv(x))
    return pre * mask.to(pre.dtype), pre


TRAIN_SHAPES = [(2, 3, 9, 36), (1, 10, 12, 68), (3, 5, 7, 8)]   # (B, D, H, W); D >= 3 and 8 <= W for the BatchNorm helpers


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", TRAIN_SHAPES, ids=str)
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_training_vs_fp64(pair, shape, mode):
    from rag_b200.matching_conv import matching_forward

    c, o = pair
    b, d, h, w = shape
    g = gen(hash((pair, shape, mode)) % 991)
    layer = _layer(c, o, g).train(mode == "train")
    x0 = randn((b, c, d, h, w), g).cuda()
    gout = randn((b, o, d, h, w), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)
    ours, _ = _run(layer, x0, gout, matching_forward, torch.float32)
    mask = ours[0] > 0
    ref64, pre64 = _run(layer, x0, gout, lambda lay, x: _masked(lay, x, mask), torch.float64)
    flips = (pre64.detach() > 0) != mask
    assert not flips.any() or pre64.detach()[flips].abs().max().item() <= 1e-5, "ReLU decision differs from fp64 beyond rounding"
    names = ["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
    for n, a, r in zip(names, ours, ref64):
        assert _mx(a, r) <= 1e-5, f"{n}: {_mx(a, r):.3e}"
    # only the BatchNorm parameters trainable, the input not requiring grad
    ours2, _ = _run(layer, x0, gout, matching_forward, torch.float32, req_x=False, only_bn=True)
    assert ours2[1] is None and ours2[2] is None
    for i in (3, 4):
        assert _mx(ours2[i], ref64[i]) <= 1e-5


def test_backward_is_bitwise_repeatable_and_routed():
    from rag_b200 import _cabi
    from rag_b200.matching_conv import matching_forward, qualifies

    g = gen(11)
    layer = _layer(12, 12, g).train()
    x0 = randn((2, 12, 16, 24, 96), g).cuda()
    gout = randn((2, 12, 16, 24, 96), g).cuda()
    assert qualifies(layer, x0.clone().requires_grad_(True))
    n0 = _cabi.launch_count()
    a, _ = _run(layer, x0, gout, matching_forward, torch.float32)
    launches = _cabi.launch_count() - n0
    # fwd conv + moments (2) + finalize + normalise | bwd sums (2) + consts + gz + data gradient + weight gradient (2)
    assert launches == 12, launches
    b_, _ = _run(layer, x0, gout, matching_forward, torch.float32)
    for u, v in zip(a, b_):
        assert torch.equal(u, v)


def test_routing_launches_and_flag_off_parity():
    """Qualifying layers run the kernels (one launch in eval()); excluded ones none; outputs match the flag-off path."""
    from rag_b200 import _cabi
    from rag_b200.fused_stem import stem_forward
    from rag_b200.matching_conv import matching_forward

    g = gen(13)
    x = randn((2, 12, 6, 10, 40), g).cuda()
    good = _layer(12, 12, g).eval()
    x5 = randn((2, 5, 6, 10, 40), g).cuda()
    excluded = {                                  # name: (layer, its input)
        "1x1": (ConvBR_3d(12, 12, 1, 1, 0).cuda().eval(), x),
        "stride 2": (ConvBR_3d(12, 12, 3, 2, 1).cuda().eval(), x),
        "bias": (ConvBR_3d(12, 12, bias=True).cuda().eval(), x),
        "(12,5)": (ConvBR_3d(12, 5).cuda().eval(), x),
        "(5,5)": (ConvBR_3d(5, 5).cuda().eval(), x5),
        "no bn": (ConvBR_3d(12, 12, bn=False).cuda().eval(), x),
        "affine-free bn": (ConvBR_3d(12, 12, affine=False).cuda().eval(), x),
        "fp64": (ConvBR_3d(12, 12).cuda().double().eval(), x.double()),
    }
    with torch.no_grad():
        n0 = _cabi.launch_count()
        out = matching_forward(good, x)
        assert _cabi.launch_count() - n0 == 1
        ref = stem_forward(good, x.clone())
        assert _mx(out, ref) <= 1e-5
        for name, (lay, xi) in excluded.items():
            n0 = _cabi.launch_count()
            out = matching_forward(lay, xi)
            assert _cabi.launch_count() - n0 == 0, name
            assert torch.equal(out, stem_forward(lay, xi.clone())), name
    # train(): batch statistics through the kernels, same result as the flag-off (cuDNN) path within the tolerance
    l1, l2 = copy.deepcopy(good).train(), copy.deepcopy(good).train()
    v0 = (l1.bn.running_mean._version, l1.bn.running_var._version)
    with torch.no_grad():
        o1, o2 = matching_forward(l1, x), stem_forward(l2, x.clone())
    assert l1.bn.running_mean._version > v0[0] and l1.bn.running_var._version > v0[1]      # written in place, as F.batch_norm marks it
    assert _mx(o1, o2) <= 1e-5
    assert torch.allclose(l1.bn.running_mean, l2.bn.running_mean, rtol=1e-5, atol=1e-6)
    assert torch.allclose(l1.bn.running_var, l2.bn.running_var, rtol=1e-5, atol=1e-6)
    assert int(l1.bn.num_batches_tracked) == int(l2.bn.num_batches_tracked) == 1


def test_cuda_graph_capture_replays_bit_exact():
    from rag_b200.matching_conv import matching_forward

    g = gen(17)
    layer = _layer(8, 8, g).eval()
    x = randn((2, 8, 8, 12, 64), g).cuda().requires_grad_(True)
    gout = randn((2, 8, 8, 12, 64), g).cuda()

    def step():
        layer.zero_grad(set_to_none=True)
        x.grad = None
        out = matching_forward(layer, x)
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
        out = matching_forward(layer, x)
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


@pytest.mark.parametrize("pair", PAIRS, ids=str)
def test_guard_bands(pair):
    from rag_b200 import _cabi

    L = _cabi.lib()
    st = torch.cuda.current_stream().cuda_stream
    c, o = pair
    b, d, h, w = 2, 3, 9, 68
    g = gen(19)
    x = randn((b, c, d, h, w), g).cuda()
    gz = randn((b, o, d, h, w), g).cuda()
    wt = randn((o, c, 3, 3, 3), g).cuda()
    ob, out = _window(b * o * d * h * w)
    gb, gin = _window(b * c * d * h * w)
    wb, gw = _window(o * c * 27)
    ws = torch.empty(int(L.rag_conv3d_cc_bwd_workspace_bytes(b, c, o, d, h, w)) // 4, device="cuda")
    assert L.rag_conv3d_cc_fwd(x.data_ptr(), wt.data_ptr(), None, None, 1, out.data_ptr(), b, c, o, d, h, w, st) == 0
    assert L.rag_conv3d_cc_bwd(gz.data_ptr(), x.data_ptr(), wt.data_ptr(), gin.data_ptr(), gw.data_ptr(), ws.data_ptr(), b, c, o, d, h, w, st) == 0
    torch.cuda.synchronize()
    assert _intact(ob, out.numel()) and _intact(gb, gin.numel()) and _intact(wb, gw.numel())
    x64, gz64, w64 = x.double(), gz.double(), wt.double()
    assert _mx(out.view(b, o, d, h, w), F.relu(F.conv3d(x64, w64, padding=1))) <= 1e-5
    x64.requires_grad_(True); w64.requires_grad_(True)
    F.conv3d(x64, w64, padding=1).backward(gz64)
    assert _mx(gin.view(b, c, d, h, w), x64.grad) <= 1e-5
    assert _mx(gw.view(o, c, 3, 3, 3), w64.grad) <= 1e-5


def test_matching_convs_on_the_real_network():
    """install(..., fuse_stem=True, upsample=True, matching_convs=True) on the reference's own Network: eval forward within
    1e-3 px of the unpatched network; training gradients as close to the fp64 network as the unpatched fp32 reference is,
    within a factor 4 (the criterion of test_fuse_stem_on_the_real_network).  Skips without oracle/_ref."""
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

    try:
        # the same eval forward without matching_convs: the launches of ours it does not have are the interior layers'
        N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, fuse_stem=True, upsample=True)
        _, base_eval = launches(fwd)
        N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, fuse_stem=True, upsample=True, matching_convs=True)
        assert ref.operations_3d.ConvBR_3d.forward.__module__ == "rag_b200.matching_conv"
        out, n_eval = launches(fwd)
        assert n_eval > base_eval, f"no interior ConvBR_3d took the kernels in eval() ({n_eval} vs {base_eval} launches)"
        assert (out - ref_out).abs().max().item() <= 1e-3
        net.train()
        state = deepcopy(net.state_dict())

        def fwd_bwd():
            net.load_state_dict(state)
            net.zero_grad(set_to_none=True)
            (call() * w).sum().backward()
            return {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}

        got_g, n_train = launches(fwd_bwd)
        N.install(ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d, fuse_stem=True, upsample=True)
        _, base_train = launches(fwd_bwd)
        assert n_train > base_train, f"no interior ConvBR_3d took the kernels in train() ({n_train} vs {base_train} launches)"
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
