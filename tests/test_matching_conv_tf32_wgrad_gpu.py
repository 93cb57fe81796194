"""The TF32 weight gradient of the interior ConvBR_3d layers (csrc/conv3d_cc_tf32.cu, ``rag_conv3d_cc_tf32_bwd_weight``;
``install(..., matching_tf32=True, matching_tf32_wgrad=True)``) against fp64, with cuDNN TF32 as the bar.

The bar is that of tests/test_matching_conv_tf32_gpu.py: each max-norm relative error against fp64 must be at most its RATIO
times the larger of cuDNN TF32's own error (``torch.nn.grad.conv3d_weight`` with ``allow_tf32`` on) and the error of the fp64
weight gradient of the TF32-rounded operands (the rounding alone).  Both errors are printed."""
import copy

import pytest
import torch
import torch.nn.functional as F

from tests._util import gen, randn
from tests.test_matching_conv_gpu import _intact, _layer, _mx, _window
from tests.test_matching_conv_tf32_gpu import FLIP_REL, _check, _pinned, _rna, _Spy, _step, _tf32, _train

pytestmark = pytest.mark.gpu
PAIRS = [(8, 8), (12, 12)]

# the kernel's grid, restated from conv3d_cc_tf32.cu (kTwGroups, kTwHt, kTwWt; tw_launch)
TW_GROUPS, TW_HT, TW_WT = 296, 4, 32


def _grid(b, h, w):
    n_tiles = b * -(-h // TW_HT) * -(-w // TW_WT)
    return min(TW_GROUPS, n_tiles), n_tiles


# (B, D, H, W): W = 8 / 12 (one k-step, and a partial one) with odd H and D = 3 / 9; W = 68 (a 4-column last tile); W = 200
# with 476 tiles on 296 CTAs (two rounds, the last partial); the level-3 training crop (B=4 288x576), 576 tiles
SHAPES = [(1, 3, 7, 8), (2, 9, 13, 12), (1, 9, 5, 68), (4, 3, 67, 200), (4, 64, 96, 192)]
TRAIN_SHAPES = [(2, 3, 9, 8), (1, 11, 13, 68), (4, 3, 67, 200), (2, 64, 96, 192)]
ENTRIES = ("rag_conv3d_cc_fwd", "rag_conv3d_cc_bwd", "rag_conv3d_cc_tf32_fwd", "rag_conv3d_cc_tf32_bwd_data",
           "rag_conv3d_cc_tf32_bwd_weight")


def test_grid_of_the_shapes():
    """The shapes above reach what they claim: a CTA with two tiles and a partial last round."""
    g, n = _grid(4, 67, 200)
    assert (g, n) == (296, 476) and n % g and n // g == 1
    g, n = _grid(4, 96, 192)
    assert (g, n) == (296, 576) and n % g
    assert _grid(1, 7, 8) == (2, 2)


@pytest.fixture(autouse=True)
def _tf32_on():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.fixture
def tf32_modes():
    from rag_b200 import matching_conv

    matching_conv.set_tf32(True)
    matching_conv.set_tf32_wgrad(True)
    yield
    matching_conv.set_tf32(False)
    matching_conv.set_tf32_wgrad(False)


def _bwd_weight(L, gz, x, gw, ws, b, c, o, d, h, w):
    return L.rag_conv3d_cc_tf32_bwd_weight(gz.data_ptr(), x.data_ptr(), gw.data_ptr(), ws.data_ptr(), b, c, o, d, h, w,
                                           torch.cuda.current_stream().cuda_stream)


def _ws(L, b, c, o, d, h, w):
    return torch.empty(int(L.rag_conv3d_cc_tf32_bwd_weight_workspace_bytes(b, c, o, d, h, w)) // 4, device="cuda")


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_weight_gradient_vs_fp64(pair, shape):
    from rag_b200 import _cabi

    L = _cabi.lib()
    c, o = pair
    b, d, h, w = shape
    g = gen(600 + 10 * PAIRS.index(pair) + SHAPES.index(shape))
    x = randn((b, c, d, h, w), g).cuda()
    gz = randn((b, o, d, h, w), g).cuda()
    wshape = (o, c, 3, 3, 3)
    ref = torch.nn.grad.conv3d_weight(x.double(), wshape, gz.double(), padding=1)
    gw = torch.empty(wshape, device="cuda")
    _cabi.check(_bwd_weight(L, gz, x, gw, _ws(L, b, c, o, d, h, w), b, c, o, d, h, w), "rag_conv3d_cc_tf32_bwd_weight")
    cud = _tf32(lambda: torch.nn.grad.conv3d_weight(x, wshape, gz, padding=1))
    rnd = torch.nn.grad.conv3d_weight(_rna(x).double(), wshape, _rna(gz).double(), padding=1)
    _check(f"gw {pair} {shape}", _mx(gw, ref), _mx(cud, ref), _mx(rnd, ref))


def _gz_rounding(layer, x0, gout, mask):
    """The rounding alone for the two gradients that round the gradient gz at the convolution output as well: the fp64 data
    gradient of the TF32-rounded w and gz, and the fp64 weight gradient of the rounded x and gz, against the fp64
    composition's own gx and gw."""
    lay = copy.deepcopy(layer).double()
    x = x0.double().requires_grad_(True)
    z = lay.conv(x)
    z.retain_grad()
    (lay.bn(z) * mask.double()).backward(gout.double())
    gz = _rna(z.grad).double()
    gx = torch.nn.grad.conv3d_input(x.shape, _rna(lay.conv.weight.detach()).double(), gz, padding=1)
    gw = torch.nn.grad.conv3d_weight(_rna(x0).double(), lay.conv.weight.shape, gz, padding=1)
    return {"gx": _mx(gx, x.grad), "gweight": _mx(gw, lay.conv.weight.grad)}


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", TRAIN_SHAPES, ids=str)
def test_training_vs_fp64(pair, shape, tf32_modes):
    """ConvBR3dFn with both flags: out, gx, gw, dgamma, dbeta and both running statistics, the ReLU pinned to ours."""
    from rag_b200.matching_conv import matching_forward

    c, o = pair
    b, d, h, w = shape
    g = gen(700 + 10 * PAIRS.index(pair) + TRAIN_SHAPES.index(shape))
    layer = _layer(c, o, g).train()
    x0 = randn((b, c, d, h, w), g).cuda()
    gout = randn((b, o, d, h, w), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)
    ours, _ = _train(layer, x0, gout, matching_forward, torch.float32, True)
    cud, _ = _train(layer, x0, gout, lambda lay, x: F.relu(lay.bn(lay.conv(x))), torch.float32, True)
    ref64, pre64 = _train(layer, x0, gout, _pinned(ours[0] > 0), torch.float64, False)
    cref64, _ = _train(layer, x0, gout, _pinned(cud[0] > 0), torch.float64, False)
    rlayer = copy.deepcopy(layer)
    with torch.no_grad():
        rlayer.conv.weight.copy_(_rna(rlayer.conv.weight))
    rnd64, _ = _train(rlayer, _rna(x0), gout, _pinned(ours[0] > 0), torch.float64, False)
    pre = pre64.detach()
    flips = (pre > 0) != (ours[0] > 0)
    assert not flips.any() or (pre[flips].abs().max() / pre.abs().max()).item() <= FLIP_REL
    gz_rnd = _gz_rounding(layer, x0, gout, ours[0] > 0)
    names = ["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
    for n, a, cu, r, cr, rr in zip(names, ours, cud, ref64, cref64, rnd64):
        _check(f"{n} {pair} {shape}", _mx(a, r), max(_mx(cu, cr), 1e-7), max(_mx(rr, r), gz_rnd.get(n, 0.0)))


@pytest.mark.parametrize("pair", PAIRS, ids=str)
@pytest.mark.parametrize("shape", [(2, 3, 9, 68), (4, 3, 67, 200)], ids=str)
def test_repeatable_captured_and_guarded(pair, shape):
    """Two runs give the same bits, a CUDA-graph replay too, and nothing outside gw and the workspace is written."""
    from rag_b200 import _cabi

    L = _cabi.lib()
    c, o = pair
    b, d, h, w = shape
    g = gen(31)
    x, gz = randn((b, c, d, h, w), g).cuda(), randn((b, o, d, h, w), g).cuda()
    n = o * c * 27
    wb, gw = _window(n)
    nws = int(L.rag_conv3d_cc_tf32_bwd_weight_workspace_bytes(b, c, o, d, h, w)) // 4
    sb, ws = _window(nws)
    assert _bwd_weight(L, gz, x, gw, ws, b, c, o, d, h, w) == 0
    torch.cuda.synchronize()
    assert _intact(wb, n) and _intact(sb, nws)
    first = gw.clone()
    assert _bwd_weight(L, gz, x, gw, ws, b, c, o, d, h, w) == 0
    torch.cuda.synchronize()
    assert torch.equal(gw, first)
    gw.zero_(), ws.zero_()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s), torch.cuda.graph(graph):
        assert _bwd_weight(L, gz, x, gw, ws, b, c, o, d, h, w) == 0
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gw, first)
    assert _intact(wb, n) and _intact(sb, nws)
    ref = torch.nn.grad.conv3d_weight(x.double(), (o, c, 3, 3, 3), gz.double(), padding=1)
    assert _mx(gw.view(o, c, 3, 3, 3), ref) <= 1e-3


def test_routing(monkeypatch):
    """Both flags: one TF32 weight-gradient call per backward and no rag_conv3d_cc_bwd; everything but gw has the bits of
    matching_tf32 alone.  4 -> 4 stays on rag_conv3d_cc_bwd.  The new flag off: the call counts of matching_tf32 alone."""
    from rag_b200 import matching_conv

    g = gen(37)
    layer = _layer(12, 12, g).train()
    x0, gout = randn((2, 12, 6, 10, 40), g).cuda(), randn((2, 12, 6, 10, 40), g).cuda()
    layer4 = _layer(4, 4, g).train()
    x4, gout4 = randn((2, 4, 6, 10, 40), g).cuda(), randn((2, 4, 6, 10, 40), g).cuda()
    base4 = _step(layer4, x4, gout4)
    try:
        matching_conv.set_tf32(True)
        spy = _Spy(monkeypatch, ENTRIES)
        tf32_only = _step(layer, x0, gout)
        # as tests/test_matching_conv_tf32_gpu.py::test_routing: train forward + eval forward on TF32, the fp32 weight gradient
        assert spy.calls == {"rag_conv3d_cc_fwd": 0, "rag_conv3d_cc_bwd": 1, "rag_conv3d_cc_tf32_fwd": 2,
                             "rag_conv3d_cc_tf32_bwd_data": 1, "rag_conv3d_cc_tf32_bwd_weight": 0}, spy.calls
        matching_conv.set_tf32_wgrad(True)
        torch.backends.cudnn.allow_tf32 = False           # read at call time: the fp32 kernels
        spy.calls = dict.fromkeys(ENTRIES, 0)
        _step(layer, x0, gout)
        assert spy.calls["rag_conv3d_cc_tf32_bwd_weight"] == 0 and spy.calls["rag_conv3d_cc_fwd"] == 2
        torch.backends.cudnn.allow_tf32 = True
        spy.calls = dict.fromkeys(ENTRIES, 0)
        got = _step(layer, x0, gout)
        assert spy.calls == {"rag_conv3d_cc_fwd": 0, "rag_conv3d_cc_bwd": 0, "rag_conv3d_cc_tf32_fwd": 2,
                             "rag_conv3d_cc_tf32_bwd_data": 1, "rag_conv3d_cc_tf32_bwd_weight": 1}, spy.calls
        for i, (a, b_) in enumerate(zip(got, tf32_only)):      # out, gx, gw, dgamma, running_var, eval out
            if i == 2:
                assert not torch.equal(a, b_) and _mx(a, b_) <= 1e-2
            else:
                assert torch.equal(a, b_), i
        # 4 -> 4 stays on the fp32 kernels: same bits, the fp32 weight gradient
        spy.calls = dict.fromkeys(ENTRIES, 0)
        for a, b_ in zip(_step(layer4, x4, gout4), base4):
            assert torch.equal(a, b_)
        assert spy.calls["rag_conv3d_cc_bwd"] == 1 and spy.calls["rag_conv3d_cc_tf32_bwd_weight"] == 0
    finally:
        matching_conv.set_tf32(False)
        matching_conv.set_tf32_wgrad(False)


def test_training_step_of_the_stand_in(monkeypatch):
    """Every install() flag plus both TF32 flags on the stand-in network, under torch.use_deterministic_algorithms(True):
    two seeded steps give the same pred, gradients and running statistics; the 12 -> 12 and 8 -> 8 layers take the TF32
    weight gradient; pred and every parameter gradient are no further from fp64 than the plain module tree under cuDNN TF32
    (max(3 x its error, 2e-5), the criterion of tests/test_training_step_gpu.py)."""
    from rag_b200 import network as N
    from rag_b200 import pointwise_conv
    from tests._stand_in import ReluPins, _stand_in, ref_forward
    from tests._util import sparse_grad
    from tests.test_training_step_gpu import MAXDISP, _compare, _prepare, _run, _state

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)
    mine, ref = _stand_in(), _stand_in()
    state = _state(ref[0], 4, 43)
    g = gen(1033)
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
                  resample=True, resample_modules=(cells,), matching_tf32=True, matching_tf32_wgrad=True)
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
    assert spy.calls["rag_conv3d_cc_tf32_bwd_weight"] > 0 and spy.calls["rag_conv3d_cc_tf32_bwd_data"] > 0
    ours, again = runs
    assert torch.equal(ours[0], again[0])
    for i in (1, 2):
        for n in ours[i]:
            assert (ours[i][n] is None and again[i][n] is None) or torch.equal(ours[i][n], again[i][n]), n

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
