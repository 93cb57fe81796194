"""The interior ConvBR_3d layers on the tensor cores in TF32 (csrc/conv3d_cc_tf32.cu; ``install(..., matching_convs=True,
matching_tf32=True)``) against fp64, with cuDNN TF32 as the bar.

TF32 keeps 10 mantissa bits of each operand, so these results are ~1e-4 of fp64 instead of the fp32 kernels' ~1e-6.  The bar
is what a user of the reference gets by default: each max-norm relative error against fp64 must be at most RATIO times the
error of the same computation on cuDNN with ``allow_tf32 = True``.  Where cuDNN picks an fp32 algorithm on a small shape, its
error says nothing about TF32, so the bar is never below RATIO times the error of the fp64 convolution of the TF32-rounded
operands (the rounding alone).  Both errors are printed.

ReLU decisions: TF32 and fp64 disagree on pre-activations within ~1e-3 of the max-norm, so the training comparisons pin the
ReLU to ours (as tests/test_matching_conv_gpu.py does) and allow a flip only where |pre| <= FLIP_REL of the max."""
import copy

import pytest
import torch
import torch.nn.functional as F

from tests._util import gen, randn
from tests.test_matching_conv_gpu import ConvBR_3d, _intact, _layer, _mx, _window

pytestmark = pytest.mark.gpu
PAIRS = [(4, 4), (8, 8), (12, 12)]
RATIO = 2.0
FLIP_REL = 2e-3
# (B, D, H, W): B = 1 with D and H tails and a W that leaves a partial column tile; the narrowest and widest W; the level-3
# training crop (B=4 288x576 at 1/3 resolution)
SHAPES = [(1, 11, 13, 68), (2, 3, 9, 8), (1, 4, 5, 1016), (4, 64, 96, 192)]
TRAIN_SHAPES = [(1, 11, 13, 68), (2, 3, 9, 8), (1, 4, 5, 1016), (2, 64, 96, 192)]


@pytest.fixture(autouse=True)
def _tf32_on():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.fixture
def tf32_mode():
    from rag_b200 import matching_conv

    matching_conv.set_tf32(True)
    yield
    matching_conv.set_tf32(False)


def _rna(t):
    """t rounded to TF32 (10-bit mantissa), to nearest, ties away from zero: the kernels' operand rounding."""
    i = t.float().contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _bar(cudnn_err, rounding_err):
    return RATIO * max(cudnn_err, rounding_err)


def _tf32(fn):
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = True
    try:
        return fn()
    finally:
        torch.backends.cudnn.allow_tf32 = old


def _check(what, ours, cudnn, rounding):
    print(f"\n{what}: ours {ours:.2e}  cuDNN TF32 {cudnn:.2e}  TF32 rounding alone {rounding:.2e}")
    assert ours <= _bar(cudnn, rounding), f"{what}: {ours:.3e} > {RATIO} x max({cudnn:.3e}, {rounding:.3e})"


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_forward_and_data_gradient_vs_fp64(pair, shape):
    from rag_b200 import _cabi
    from rag_b200.matching_conv import conv3d_cc_forward

    c, o = pair
    b, d, h, w = shape
    g = gen(hash((pair, shape)) % 1013)
    x = randn((b, c, d, h, w), g).cuda()
    gz = randn((b, o, d, h, w), g).cuda()
    wt = randn((o, c, 3, 3, 3), g).cuda() * 0.2
    x64, w64, gz64 = x.double(), wt.double(), gz.double()
    # forward, raw z
    ref = F.conv3d(x64, w64, padding=1)
    z = conv3d_cc_forward(x, wt, tf32=True)
    _check(f"z {pair} {shape}", _mx(z, ref), _mx(_tf32(lambda: F.conv3d(x, wt, padding=1)), ref),
           _mx(F.conv3d(_rna(x).double(), _rna(wt).double(), padding=1), ref))
    # the eval fold with ReLU, relative to the pre-activation's max-norm (the ReLU is 1-Lipschitz: no flip tolerance needed)
    lay = _layer(c, o, g).eval()
    from rag_b200.batchnorm import eval_fold

    scale, shift = eval_fold(lay.bn)
    pre = lay.double().bn(F.conv3d(x64, w64, padding=1)).detach()
    lay.float()
    out = conv3d_cc_forward(x, wt, scale.detach(), shift.detach(), relu=True, tf32=True)
    with torch.no_grad():
        cud = _tf32(lambda: F.relu(lay.bn(F.conv3d(x, wt, padding=1))))
    m = pre.abs().max()
    rel = lambda a: ((a.double() - F.relu(pre)).abs().max() / m).item()  # noqa: E731
    r64 = F.relu(lay.double().bn(F.conv3d(_rna(x).double(), _rna(wt).double(), padding=1)))
    lay.float()
    _check(f"eval fold {pair} {shape}", rel(out), rel(cud), rel(r64))
    # data gradient
    x64.requires_grad_(True)
    F.conv3d(x64, w64, padding=1).backward(gz64)
    gin = torch.empty_like(x)
    L = _cabi.lib()
    _cabi.check(L.rag_conv3d_cc_tf32_bwd_data(gz.data_ptr(), wt.data_ptr(), gin.data_ptr(), b, c, o, d, h, w,
                                              torch.cuda.current_stream().cuda_stream), "bwd_data")
    xc = x.clone().requires_grad_(True)
    _tf32(lambda: F.conv3d(xc, wt, padding=1).backward(gz))
    xr = _rna(x).double().requires_grad_(True)
    F.conv3d(xr, _rna(wt).double(), padding=1).backward(_rna(gz).double())
    _check(f"gx {pair} {shape}", _mx(gin, x64.grad), _mx(xc.grad, x64.grad), _mx(xr.grad, x64.grad))


def _train(layer, x0, gout, fn, dtype, tf32_cudnn):
    lay = copy.deepcopy(layer).to(dtype)
    x = x0.detach().to(dtype).clone().requires_grad_(True)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = tf32_cudnn
    try:
        out = fn(lay, x)
        pre = None
        if isinstance(out, tuple):
            out, pre = out
        out.backward(gout.to(dtype))
    finally:
        torch.backends.cudnn.allow_tf32 = old
    return [out.detach(), x.grad, lay.conv.weight.grad, lay.bn.weight.grad, lay.bn.bias.grad,
            lay.bn.running_mean.clone(), lay.bn.running_var.clone()], pre


def _pinned(mask):
    def fn(lay, x):
        pre = lay.bn(lay.conv(x))
        return pre * mask.to(pre.dtype), pre
    return fn


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", TRAIN_SHAPES, ids=str)
def test_training_vs_fp64(pair, shape, tf32_mode):
    """ConvBR3dFn in TF32 mode: out, gx, gw, dgamma, dbeta and both running statistics."""
    from rag_b200.matching_conv import matching_forward

    c, o = pair
    b, d, h, w = shape
    g = gen(hash((pair, shape, "train")) % 997)
    layer = _layer(c, o, g).train()
    x0 = randn((b, c, d, h, w), g).cuda()
    gout = randn((b, o, d, h, w), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)
    ours, _ = _train(layer, x0, gout, matching_forward, torch.float32, True)
    cud, _ = _train(layer, x0, gout, lambda lay, x: F.relu(lay.bn(lay.conv(x))), torch.float32, True)
    ref64, pre64 = _train(layer, x0, gout, _pinned(ours[0] > 0), torch.float64, False)
    cref64, _ = _train(layer, x0, gout, _pinned(cud[0] > 0), torch.float64, False)
    # the TF32 rounding alone: the same fp64 composition on the rounded input and weight
    rlayer = copy.deepcopy(layer)
    with torch.no_grad():
        rlayer.conv.weight.copy_(_rna(rlayer.conv.weight))
    rnd64, _ = _train(rlayer, _rna(x0), gout, _pinned(ours[0] > 0), torch.float64, False)
    pre = pre64.detach()
    flips = (pre > 0) != (ours[0] > 0)
    assert not flips.any() or (pre[flips].abs().max() / pre.abs().max()).item() <= FLIP_REL
    names = ["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
    for n, a, cu, r, cr, rr in zip(names, ours, cud, ref64, cref64, rnd64):
        # the running statistics are fp32 values either way: their floor is one rounding of the stored value
        _check(f"{n} {pair} {shape}", _mx(a, r), max(_mx(cu, cr), 1e-7), _mx(rr, r))


def _launch_pair(L, x, wt, gz, out, gin, b, c, o, d, h, w):
    st = torch.cuda.current_stream().cuda_stream
    assert L.rag_conv3d_cc_tf32_fwd(x.data_ptr(), wt.data_ptr(), None, None, 1, out.data_ptr(), b, c, o, d, h, w, st) == 0
    assert L.rag_conv3d_cc_tf32_bwd_data(gz.data_ptr(), wt.data_ptr(), gin.data_ptr(), b, c, o, d, h, w, st) == 0


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", [(2, 3, 9, 68), (1, 9, 17, 200)], ids=str)
def test_repeatable_captured_and_guarded(pair, shape):
    """Two runs give the same bits, a CUDA-graph replay too, and nothing outside out / gin is written."""
    from rag_b200 import _cabi

    L = _cabi.lib()
    c, o = pair
    b, d, h, w = shape
    g = gen(23)
    x, gz, wt = randn((b, c, d, h, w), g).cuda(), randn((b, o, d, h, w), g).cuda(), randn((o, c, 3, 3, 3), g).cuda()
    ob, out = _window(b * o * d * h * w)
    gb, gin = _window(b * c * d * h * w)
    _launch_pair(L, x, wt, gz, out, gin, b, c, o, d, h, w)
    torch.cuda.synchronize()
    assert _intact(ob, out.numel()) and _intact(gb, gin.numel())
    first = (out.clone(), gin.clone())
    _launch_pair(L, x, wt, gz, out, gin, b, c, o, d, h, w)
    torch.cuda.synchronize()
    assert torch.equal(out, first[0]) and torch.equal(gin, first[1])
    out.zero_(), gin.zero_()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s), torch.cuda.graph(graph):
        _launch_pair(L, x, wt, gz, out, gin, b, c, o, d, h, w)
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, first[0]) and torch.equal(gin, first[1])
    assert _intact(ob, out.numel()) and _intact(gb, gin.numel())
    ref = F.relu(F.conv3d(x.double(), wt.double(), padding=1))
    assert _mx(out.view(b, o, d, h, w), ref) <= 1e-3


class _Spy:
    """Counts the calls of the named library entries (the ctypes attributes of the loaded library, replaced for the test)."""

    def __init__(self, monkeypatch, names):
        from rag_b200 import _cabi

        L = _cabi.lib()
        self.calls = {n: 0 for n in names}
        for n in names:
            real = getattr(L, n)

            def spy(*a, _n=n, _real=real):
                self.calls[_n] += 1
                return _real(*a)
            monkeypatch.setattr(L, n, spy)


ENTRIES = ("rag_conv3d_cc_fwd", "rag_conv3d_cc_bwd", "rag_conv3d_cc_tf32_fwd", "rag_conv3d_cc_tf32_bwd_data")


def _step(layer, x0, gout):
    from rag_b200.matching_conv import matching_forward

    lay = copy.deepcopy(layer)
    x = x0.clone().requires_grad_(True)
    out = matching_forward(lay, x)
    out.backward(gout)
    with torch.no_grad():
        ev = matching_forward(copy.deepcopy(layer).eval(), x0)
    return [out.detach(), x.grad, lay.conv.weight.grad, lay.bn.weight.grad, lay.bn.running_var.clone(), ev]


def test_routing(monkeypatch):
    """Flag off, or flag on with allow_tf32 off: the fp32 kernels' bits.  Flag and allow_tf32 on: the TF32 entries, no fp32
    forward or fp32 data gradient.  Layers that do not qualify: the fuse_stem binding, as without the flag."""
    from rag_b200 import matching_conv
    from rag_b200.fused_stem import stem_forward

    g = gen(29)
    layer = _layer(12, 12, g).train()
    x0, gout = randn((2, 12, 6, 10, 40), g).cuda(), randn((2, 12, 6, 10, 40), g).cuda()
    base = _step(layer, x0, gout)
    layer4 = _layer(4, 4, g).train()
    x4, gout4 = randn((2, 4, 6, 10, 40), g).cuda(), randn((2, 4, 6, 10, 40), g).cuda()
    base4 = _step(layer4, x4, gout4)
    try:
        matching_conv.set_tf32(True)
        torch.backends.cudnn.allow_tf32 = False
        for a, b_ in zip(_step(layer, x0, gout), base):
            assert torch.equal(a, b_)
        torch.backends.cudnn.allow_tf32 = True
        spy = _Spy(monkeypatch, ENTRIES)
        got = _step(layer, x0, gout)
        # train forward + eval forward on TF32; the backward's fp32 call carries the weight gradient only
        assert spy.calls == {"rag_conv3d_cc_fwd": 0, "rag_conv3d_cc_bwd": 1, "rag_conv3d_cc_tf32_fwd": 2,
                             "rag_conv3d_cc_tf32_bwd_data": 1}, spy.calls
        assert not torch.equal(got[0], base[0])
        assert _mx(got[0], base[0]) <= 1e-2
        # 4 -> 4 stays on the fp32 kernels (the shape rule of matching_conv.use_tf32): same bits
        for a, b_ in zip(_step(layer4, x4, gout4), base4):
            assert torch.equal(a, b_)
        x5 = randn((2, 5, 6, 10, 40), g).cuda()
        for lay, xi in ((ConvBR_3d(12, 12, 1, 1, 0).cuda().eval(), x0), (ConvBR_3d(5, 5).cuda().eval(), x5),
                        (ConvBR_3d(12, 12, bias=True).cuda().eval(), x0)):
            before = dict(spy.calls)
            with torch.no_grad():
                out = matching_conv.matching_forward(lay, xi)
                assert torch.equal(out, stem_forward(lay, xi.clone()))
            assert spy.calls == before
    finally:
        matching_conv.set_tf32(False)


def test_training_step_of_the_stand_in(monkeypatch):
    """Every install() flag plus matching_tf32=True on the stand-in network, under torch.use_deterministic_algorithms(True):
    two steps give the same bits, the 12 -> 12 and 8 -> 8 layers take the TF32 entries, and pred and every parameter gradient are no further from fp64 than the plain module tree
    under cuDNN TF32 (max(3 x its error, 2e-5), the criterion of tests/test_training_step_gpu.py)."""
    from rag_b200 import network as N
    from rag_b200 import pointwise_conv
    from tests._stand_in import ReluPins, _stand_in, ref_forward
    from tests._util import sparse_grad
    from tests.test_training_step_gpu import MAXDISP, _compare, _prepare, _run, _state

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)
    mine, ref = _stand_in(), _stand_in()
    state = _state(ref[0], 4, 41)
    g = gen(1031)
    b, h, w = 2, 48, 96
    batches = [(randn((b, 3, h, w), g).cuda(), randn((b, 3, h, w), g).cuda(), sparse_grad((b, h, w), g, keep=0.7).cuda())]
    pins = ReluPins()
    spy = _Spy(monkeypatch, ENTRIES)
    N.uninstall()
    det = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        rag_model, ops3d, cells = mine
        N.install(rag_model, None, ops3d, fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True,
                  resample=True, resample_modules=(cells,), matching_tf32=True)
        runs = []
        for i in range(2):
            net = _prepare(rag_model.Network(MAXDISP, k=4, level12=True), state, False, torch.float32)
            if i == 0:
                with pins.record(net):
                    runs.append(_run(net, lambda n, l, r: n(l, r, 0), batches, torch.float32))
            else:
                runs.append(_run(net, lambda n, l, r: n(l, r, 0), batches, torch.float32))
    finally:
        N.uninstall()
        torch.use_deterministic_algorithms(det)
    assert spy.calls["rag_conv3d_cc_tf32_fwd"] > 0 and spy.calls["rag_conv3d_cc_tf32_bwd_data"] > 0
    ours, again = runs
    assert torch.equal(ours[0], again[0])
    for n in ours[1]:
        assert (ours[1][n] is None and again[1][n] is None) or torch.equal(ours[1][n], again[1][n]), n

    def plain(dtype):
        r = _prepare(ref[0].Network(MAXDISP, k=4, level12=True), state, False, dtype)
        with pins.replay(r, ref[1]):
            return _run(r, ref_forward, batches, dtype)

    r32 = plain(torch.float32)                    # cuDNN TF32: allow_tf32 is on (fixture)
    r64 = plain(torch.float64)
    pins.flips(rel=FLIP_REL)
    rows = _compare(ours, r32, r64)
    for n, e_ours, e_ref in rows:
        print(f"  {n:32s} ours {e_ours:.2e}  cuDNN TF32 {e_ref:.2e}")
    bad = [(n, e_ours, e_ref) for n, e_ours, e_ref in rows if e_ours > max(3.0 * e_ref, 2e-5)]
    assert not bad, bad
