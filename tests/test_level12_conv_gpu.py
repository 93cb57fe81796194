"""The level-12 interior ConvBR_3d layer, ``ConvBR_3d(16, 16, 3, 1, 1)``, on the rag_conv3d_cc16_* entries of
csrc/conv3d_cc.cu (``install(..., matching_convs=True, level12_convs=True)``) against fp64 compositions of the reference layer.

The bar is that of tests/test_matching_conv_gpu.py: max-norm relative 1e-5 of fp64.  In training, each tensor must also be
no further from fp64 than RATIO times the error of the same composition in fp32 on cuDNN (TF32 off), or FLOOR; both errors
are printed.  The floor is there because the data gradient sums its 432 products per element in order, in fp32: on some
shapes that is up to ~7x cuDNN's error, still under 1e-5."""
import copy

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests._util import gen, randn
from tests.test_matching_conv_gpu import _fp32_convs, _intact, _layer, _masked, _mx, _run, _window  # noqa: F401
from tests.test_matching_conv_tf32_gpu import _Spy, _step

pytestmark = pytest.mark.gpu
RATIO, FLOOR = 4.0, 5e-6
ENTRIES = ("rag_conv3d_cc_fwd", "rag_conv3d_cc_bwd", "rag_conv3d_cc16_fwd", "rag_conv3d_cc16_bwd", "rag_conv3d_cc_tf32_fwd",
           "rag_conv3d_cc_tf32_bwd_data", "rag_conv3d_cc_tf32_bwd_weight")

# the weight gradient's grid, restated from conv3d_cc.cu (kCcWgGroups, kCcWgHT, kCc16WT, kCc16WgDT; cc_launch_wgrad)
WG_GROUPS, WG_HT, WG_WT = 296, 2, 32

# (B, D, H, W) of the level-12 op: training crops 192x384 and 288x576 at B=4, eval 480x960 at B=8, KITTI 384x1248 at B=4,
# maxdisp 288 at 288x576
LEVEL12_SHAPES = [(4, 16, 16, 32), (4, 16, 24, 48), (8, 16, 40, 80), (4, 16, 32, 104), (4, 24, 24, 48)]
# ragged: tails of the 8 x 32 tile in h and w, D = 1 / 2, one plane per CTA and several
RAGGED_SHAPES = [(2, 1, 11, 36), (3, 2, 9, 20), (2, 3, 17, 68), (1, 10, 5, 132), (1, 9, 7, 8)]
TRAIN_SHAPES = [(2, 3, 9, 36), (1, 10, 12, 68), (3, 5, 7, 8), (4, 16, 24, 48)]
# 378 tiles on 296 CTAs (a partial second round); 594 tiles (two rounds and a partial third); the 288x576 crop, 1536 tiles
WRAP_SHAPES = [(2, 9, 13, 68), (3, 11, 17, 40), (4, 16, 24, 48)]


def _wg_grid(b, d, h, w):
    n_tiles = b * d * -(-h // WG_HT) * -(-w // WG_WT)
    return min(WG_GROUPS, n_tiles), n_tiles


def test_grid_of_the_wrap_shapes():
    assert _wg_grid(2, 9, 13, 68) == (296, 378)
    assert _wg_grid(3, 11, 17, 40) == (296, 594) and 594 // 296 == 2 and 594 % 296
    assert _wg_grid(4, 16, 24, 48) == (296, 1536) and 1536 % 296


@pytest.fixture
def level12(monkeypatch):
    """The flag on, and the routing's volume floor lifted, so that the kernels are checked at small shapes too."""
    from rag_b200 import matching_conv

    monkeypatch.setattr(matching_conv, "LEVEL12_MIN_VOXELS", 0)
    matching_conv.set_level12(True)
    yield
    matching_conv.set_level12(False)


def _seed(*key):
    return sum((i + 1) * v for i, v in enumerate(str(key).encode())) % 1009


@pytest.mark.parametrize("shape", RAGGED_SHAPES + LEVEL12_SHAPES, ids=str)
def test_forward_and_eval_fold_vs_fp64(shape, level12):
    from rag_b200.matching_conv import conv3d_cc_forward, convbr_forward, level12_qualifies

    b, d, h, w = shape
    g = gen(_seed("fwd", shape))
    x = randn((b, 16, d, h, w), g).cuda()
    wt = randn((16, 16, 3, 3, 3), g).cuda() * 0.2
    z = conv3d_cc_forward(x, wt)
    assert _mx(z, F.conv3d(x.double(), wt.double(), padding=1)) <= 1e-5
    lay = _layer(16, 16, g).eval()
    lay64 = copy.deepcopy(lay).double()
    from rag_b200 import _cabi

    with torch.no_grad():
        assert not level12_qualifies(lay, x)                    # the eval forward is routed to cuDNN (faster there)
        n0 = _cabi.launch_count()
        out = convbr_forward(lay, x)
        assert _cabi.launch_count() - n0 == 1                   # the eval fold: one launch
        pre = lay64.bn(lay64.conv(x.double()))
    assert ((out.double() - F.relu(pre)).abs().max() / pre.abs().max()).item() <= 1e-5


@pytest.mark.parametrize("shape", WRAP_SHAPES, ids=str)
def test_weight_and_data_gradient_vs_fp64(shape):
    from rag_b200 import _cabi

    L = _cabi.lib()
    b, d, h, w = shape
    g = gen(_seed("wg", shape))
    x = randn((b, 16, d, h, w), g).cuda()
    gz = randn((b, 16, d, h, w), g).cuda()
    wt = randn((16, 16, 3, 3, 3), g).cuda()
    gin, gw = torch.empty_like(x), torch.empty_like(wt)
    ws = torch.empty(int(L.rag_conv3d_cc16_bwd_workspace_bytes(b, 16, 16, d, h, w)) // 4, device="cuda")
    _cabi.check(L.rag_conv3d_cc16_bwd(gz.data_ptr(), x.data_ptr(), wt.data_ptr(), gin.data_ptr(), gw.data_ptr(), ws.data_ptr(),
                                      b, 16, 16, d, h, w, torch.cuda.current_stream().cuda_stream), "rag_conv3d_cc16_bwd")
    x64, w64 = x.double().requires_grad_(True), wt.double().requires_grad_(True)
    F.conv3d(x64, w64, padding=1).backward(gz.double())
    e_gw, e_gx = _mx(gw, w64.grad), _mx(gin, x64.grad)
    gw32 = torch.nn.grad.conv3d_weight(x, wt.shape, gz, padding=1)
    print(f"\n{shape} grid {_wg_grid(*shape)}: gw {e_gw:.2e} (cuDNN fp32 {_mx(gw32, w64.grad):.2e}), gx {e_gx:.2e}")
    assert e_gw <= 1e-5 and e_gx <= 1e-5


@pytest.mark.parametrize("shape", TRAIN_SHAPES, ids=str)
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_training_vs_fp64(shape, mode, level12):
    """ConvBR3dFn on the cc16 entries: out, gx, gw, dgamma, dbeta and both running statistics, the ReLU pinned to ours;
    train() BatchNorm, and eval() BatchNorm behind trainable layers."""
    from rag_b200.matching_conv import matching_forward

    b, d, h, w = shape
    g = gen(_seed("train", shape, mode))
    torch.manual_seed(_seed("train", shape))                    # the conv weight's default initialisation
    layer = _layer(16, 16, g).train(mode == "train")
    x0 = randn((b, 16, d, h, w), g).cuda()
    gout = randn((b, 16, d, h, w), g).cuda()
    gout = gout * (torch.rand(gout.shape, generator=g).cuda() < 0.7)
    ours, _ = _run(layer, x0, gout, matching_forward, torch.float32)
    mask = ours[0] > 0
    ref64, pre64 = _run(layer, x0, gout, lambda lay, x: _masked(lay, x, mask), torch.float64)
    fp32, _ = _run(layer, x0, gout, lambda lay, x: _masked(lay, x, mask), torch.float32)
    flips = (pre64.detach() > 0) != mask
    assert not flips.any() or pre64.detach()[flips].abs().max().item() <= 1e-5, "ReLU decision differs from fp64 beyond rounding"
    names = ["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
    errs = {n: (_mx(a, r), _mx(f, r)) for n, a, f, r in zip(names, ours, fp32, ref64)}
    print(f"\n{shape} {mode}: ours / cuDNN fp32 vs fp64: " + ", ".join(f"{n} {e:.2e} / {e32:.2e}" for n, (e, e32) in errs.items()))
    for n, (e, e32) in errs.items():
        assert e <= 1e-5 and e <= max(RATIO * e32, FLOOR), f"{n}: ours {e:.3e}, cuDNN fp32 {e32:.3e}"


@pytest.mark.parametrize("shape", [(2, 3, 9, 68), (4, 16, 24, 48)], ids=str)
def test_repeatable_captured_and_guarded(shape):
    """Two runs give the same bits, on a second stream and in a CUDA-graph replay too; nothing outside the outputs and the
    workspace is written."""
    from rag_b200 import _cabi

    L = _cabi.lib()
    b, d, h, w = shape
    g = gen(_seed("rep", shape))
    x, gz = randn((b, 16, d, h, w), g).cuda(), randn((b, 16, d, h, w), g).cuda()
    wt = randn((16, 16, 3, 3, 3), g).cuda() * 0.2
    scale, shift = torch.rand(16, generator=g).cuda() + 0.5, randn((16,), g).cuda()
    nx, nw = x.numel(), 16 * 16 * 27
    nws = int(L.rag_conv3d_cc16_bwd_workspace_bytes(b, 16, 16, d, h, w)) // 4
    bufs = [_window(n) for n in (nx, nx, nw, nws)]           # out, gin, gw, workspace
    (ob, out), (ib, gin), (wb, gw), (sb, ws) = bufs

    def run():
        st = torch.cuda.current_stream().cuda_stream
        assert L.rag_conv3d_cc16_fwd(x.data_ptr(), wt.data_ptr(), scale.data_ptr(), shift.data_ptr(), 1, out.data_ptr(),
                                     b, 16, 16, d, h, w, st) == 0
        assert L.rag_conv3d_cc16_bwd(gz.data_ptr(), x.data_ptr(), wt.data_ptr(), gin.data_ptr(), gw.data_ptr(), ws.data_ptr(),
                                     b, 16, 16, d, h, w, st) == 0

    def intact():
        torch.cuda.synchronize()
        return all(_intact(buf, n) for (buf, _), n in zip(bufs, (nx, nx, nw, nws)))

    run()
    assert intact()
    first = [out.clone(), gin.clone(), gw.clone()]
    for t in (out, gin, gw):
        t.zero_()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()
    torch.cuda.current_stream().wait_stream(s)
    assert intact() and all(torch.equal(a, b_) for a, b_ in zip((out, gin, gw), first))
    for t in (out, gin, gw, ws):
        t.zero_()
    graph = torch.cuda.CUDAGraph()
    s2 = torch.cuda.Stream()
    s2.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s2), torch.cuda.graph(graph):
        run()
    torch.cuda.current_stream().wait_stream(s2)
    graph.replay()
    assert intact() and all(torch.equal(a, b_) for a, b_ in zip((out, gin, gw), first))
    x64, w64 = x.double().requires_grad_(True), wt.double().requires_grad_(True)
    z64 = F.conv3d(x64, w64, padding=1)
    assert _mx(out.view(b, 16, d, h, w), F.relu(z64 * scale.double().view(1, -1, 1, 1, 1) + shift.double().view(1, -1, 1, 1, 1))) <= 1e-5
    z64.backward(gz.double())
    assert _mx(gin.view(x.shape), x64.grad) <= 1e-5 and _mx(gw.view(wt.shape), w64.grad) <= 1e-5


# the shape domain's edges, as tests/test_training_limits_gpu.py states them for the other pairs: (B, D, H, W)
LIMIT_CASES = [(1, 3, 3, 8), (1, 3, 3, 1016), (32767, 3, 1, 8), (1, 3, 65535, 8)]


@pytest.mark.parametrize("shape", LIMIT_CASES, ids=str)
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_training_at_the_limits_vs_fp64(shape, mode, level12):
    from rag_b200.matching_conv import level12_qualifies, matching_forward
    from tests.test_training_limits_gpu import NAMES, _compare

    b, d, h, w = shape
    g = gen(_seed("limit", shape, mode))
    layer = _layer(16, 16, g).train(mode == "train")
    x0 = randn((b, 16, d, h, w), g).cuda()
    gout = randn((b, 16, d, h, w), g).cuda() * (torch.rand((b, 16, d, h, w), generator=g).cuda() < 0.7)
    assert level12_qualifies(layer, x0.clone().requires_grad_(True))
    kind, *_ = _compare(f"conv3d_cc16 {list(shape)} {mode}", NAMES, layer, (x0,), gout, matching_forward,
                        lambda lay, mask, x: _masked(lay, x, mask))
    assert kind == "ConvBR3dFnBackward", kind


PAST = {"W=1020": ((1, 3, 1, None), {3: (1016, 1020)}),
        "D=2": ((1, None, 2, 8), {1: (3, 2)}),
        "B=32768": ((None, 3, 1, 8), {0: (32767, 32768)}),
        "H=65536": ((1, 3, None, 8), {2: (65535, 65536)})}


@pytest.mark.parametrize("which", list(PAST))
def test_one_step_past_each_limit_falls_back(which, level12):
    from rag_b200 import _cabi
    from rag_b200.matching_conv import level12_qualifies, matching_forward
    from tests.test_training_limits_gpu import NAMES, _fallback_matches_the_reference, _past

    shape, at = PAST[which]
    inside, past = _past(shape, at)
    g = gen(_seed("past", which))
    layer = _layer(16, 16, g).train()
    for s, ok in ((inside, True), (past, False)):
        assert level12_qualifies(layer, torch.empty((s[0], 16) + s[1:], device="cuda").requires_grad_(True)) == ok, s
    x0 = randn((past[0], 16) + past[1:], g).cuda()
    gout = randn((past[0], 16) + past[1:], g).cuda()
    n0 = _cabi.launch_count()
    kind = _fallback_matches_the_reference(f"conv3d_cc16 {which} {past}", NAMES, layer, (x0,), gout, matching_forward,
                                           lambda lay, x: lay(x))
    assert _cabi.launch_count() == n0 and kind != "ConvBR3dFnBackward", kind


def test_routing(monkeypatch):
    """With the flag (and the volume floor lifted), 16 -> 16 training calls take the cc16 entries and 4/8/12 layers keep their
    calls and bits; under
    matching_tf32(+_wgrad), 16 -> 16 stays fp32 while 12 -> 12 takes TF32; with the flag off, 16 -> 16 goes to the fuse_stem
    binding and its bits are those of a run without the flag."""
    from rag_b200 import matching_conv
    from rag_b200.fused_stem import stem_forward

    g = gen(41)
    shape = (2, 6, 10, 40)
    lay16 = _layer(16, 16, g).train()
    x16, g16 = randn((2, 16) + shape[1:], g).cuda(), randn((2, 16) + shape[1:], g).cuda()
    others = {c: (_layer(c, c, g).train(), randn((2, c) + shape[1:], g).cuda(), randn((2, c) + shape[1:], g).cuda()) for c in (4, 8, 12)}
    base = {c: _step(*v) for c, v in others.items()}

    def plain16():
        lay = copy.deepcopy(lay16)
        x = x16.clone().requires_grad_(True)
        out = stem_forward(lay, x)
        out.backward(g16)
        with torch.no_grad():
            ev = stem_forward(copy.deepcopy(lay16).eval(), x16)
        return [out.detach(), x.grad, lay.conv.weight.grad, lay.bn.weight.grad, lay.bn.running_var.clone(), ev]

    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)     # the flag-off runs compare cuDNN's bits
    monkeypatch.setattr(matching_conv, "LEVEL12_MIN_VOXELS", 0)
    spy = _Spy(monkeypatch, ENTRIES)
    off = _step(lay16, x16, g16)                               # flag off: no entry at all, the bits of the fuse_stem binding
    assert sum(spy.calls.values()) == 0, spy.calls
    for a, b_ in zip(off, plain16()):
        assert torch.equal(a, b_)
    try:
        matching_conv.set_level12(True)
        on = _step(lay16, x16, g16)
        assert spy.calls == {**dict.fromkeys(ENTRIES, 0), "rag_conv3d_cc16_fwd": 1, "rag_conv3d_cc16_bwd": 1}, spy.calls
        for i in (0, 5):                                       # the train and eval outputs: fp32 rounding apart
            assert _mx(on[i], off[i]) <= 1e-5
        for c, v in others.items():
            spy.calls = dict.fromkeys(ENTRIES, 0)
            for a, b_ in zip(_step(*v), base[c]):
                assert torch.equal(a, b_), c
            assert spy.calls["rag_conv3d_cc16_fwd"] == spy.calls["rag_conv3d_cc16_bwd"] == 0 and spy.calls["rag_conv3d_cc_bwd"] == 1
        # TF32 on: 16 -> 16 keeps the fp32 entries and its bits; 12 -> 12 takes the TF32 ones
        monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", True)
        matching_conv.set_tf32(True)
        matching_conv.set_tf32_wgrad(True)
        spy.calls = dict.fromkeys(ENTRIES, 0)
        for a, b_ in zip(_step(lay16, x16, g16)[:5], on[:5]):   # the eval forward [5] is cuDNN's, TF32 now
            assert torch.equal(a, b_)
        assert spy.calls == {**dict.fromkeys(ENTRIES, 0), "rag_conv3d_cc16_fwd": 1, "rag_conv3d_cc16_bwd": 1}, spy.calls
        spy.calls = dict.fromkeys(ENTRIES, 0)
        _step(*others[12])
        assert spy.calls == {**dict.fromkeys(ENTRIES, 0), "rag_conv3d_cc_tf32_fwd": 2, "rag_conv3d_cc_tf32_bwd_data": 1,
                             "rag_conv3d_cc_tf32_bwd_weight": 1}, spy.calls
    finally:
        matching_conv.set_level12(False)
        matching_conv.set_tf32(False)
        matching_conv.set_tf32_wgrad(False)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    spy.calls = dict.fromkeys(ENTRIES, 0)
    for a, b_ in zip(_step(lay16, x16, g16), off):             # the flag off again: the same bits as before it was on
        assert torch.equal(a, b_)
    assert sum(spy.calls.values()) == 0, spy.calls


def test_volume_floor():
    """Training calls route from LEVEL12_MIN_VOXELS voxels on, not one voxel row under it; eval calls never."""
    from rag_b200.matching_conv import LEVEL12_MIN_VOXELS, level12_qualifies

    g = gen(43)
    layer = _layer(16, 16, g).train()
    w = 64
    at = torch.empty((1, 16, LEVEL12_MIN_VOXELS // (8 * w), 8, w), device="cuda")
    under = torch.empty((1, 16, LEVEL12_MIN_VOXELS // (8 * w), 7, w), device="cuda")
    assert level12_qualifies(layer, at) and not level12_qualifies(layer, under)
    with torch.no_grad():
        assert not level12_qualifies(layer.eval(), at)


def _level12_network(rag_model, ops3d, cells):
    """The stand-in network with a width-16 level-12 cell: the level-3 cell's output down-sampled by 4, a Cell_3d(12, 16)
    (its 3x3x3 ops are ConvBR_3d(16, 16, 3, 1, 1)), a last_12_3d-style pointwise layer 48 -> 12 and upsample_12 into
    last_6_3d's output."""

    class Level12Network(rag_model.Network):
        def __init__(self, maxdisp, k=4):
            super().__init__(maxdisp, k=k)
            self.cell12 = cells.Cell_3d(3 * k, 16)
            self.last_12_3d = ops3d.ConvBR_3d(48, 3 * k, 1, 1, 0)

        def matching(self, cost, task_arch=None, path=None):
            x = self.stem3d1(self.stem3d0(cost))
            x3, x6 = self.cell3d(x)
            y6 = self.last_6_3d(x6)
            d, h, w = x3.shape[2:]
            x12, _ = self.cell12(rag_model.F.interpolate(x3, [d // 4, h // 4, w // 4], mode="trilinear", align_corners=True))
            upsample_12 = rag_model.nn.Upsample(size=y6.size()[2:], mode="trilinear", align_corners=True)
            y6 = y6 + upsample_12(self.last_12_3d(x12))
            upsample_6 = rag_model.nn.Upsample(size=x3.size()[2:], mode="trilinear", align_corners=True)
            return self.last_3_3d(x3 + upsample_6(y6))

    return Level12Network


def test_training_step_of_the_stand_in(monkeypatch):
    """Every install() flag plus level12_convs=True on the stand-in with a width-16 level-12 cell, under
    torch.use_deterministic_algorithms(True): two seeded steps give the same pred, gradients and running statistics; the
    16 -> 16 layers take the cc16 entries; pred and every parameter gradient are within the fp64 bar of
    tests/test_training_step_gpu.py (max(3 x the plain fp32 module tree's error, 2e-5))."""
    from rag_b200 import network as N
    from rag_b200 import pointwise_conv
    from tests._stand_in import ReluPins, _stand_in, ref_forward
    from tests._util import sparse_grad
    from tests.test_training_step_gpu import FLOOR as STEP_FLOOR
    from tests.test_training_step_gpu import MAXDISP, _compare, _prepare, _run as _net_run
    from tests.test_training_step_gpu import RATIO as STEP_RATIO

    from rag_b200 import matching_conv

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)
    monkeypatch.setattr(matching_conv, "LEVEL12_MIN_VOXELS", 0)
    mine, ref = _stand_in(), _stand_in()
    net_mine, net_ref = _level12_network(*mine), _level12_network(*ref)
    g = gen(1051)
    torch.manual_seed(1051)
    state_net = net_ref(MAXDISP)
    with torch.no_grad():
        for m in state_net.modules():
            if isinstance(m, nn.modules.batchnorm._BatchNorm):
                c = m.num_features
                m.weight.copy_(0.5 + torch.rand(c, generator=g)); m.bias.copy_(0.3 * torch.randn(c, generator=g))
                m.running_mean.copy_(0.2 * torch.randn(c, generator=g)); m.running_var.copy_(0.5 + torch.rand(c, generator=g))
    state = copy.deepcopy(state_net.state_dict())
    b, h, w = 2, 48, 192
    batches = [(randn((b, 3, h, w), g).cuda(), randn((b, 3, h, w), g).cuda(), sparse_grad((b, h, w), g, keep=0.7).cuda())]
    pins = ReluPins()
    spy = _Spy(monkeypatch, ENTRIES)
    N.uninstall()
    det = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        rag_model, ops3d, cells = mine
        N.install(rag_model, None, ops3d, fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True,
                  resample=True, resample_modules=(cells,), level12_convs=True)
        runs = []
        for i in range(2):
            net = _prepare(net_mine(MAXDISP), state, False, torch.float32)
            if i == 0:
                with pins.record(net):
                    runs.append(_net_run(net, lambda n, l, r: n(l, r, 0), batches, torch.float32))
            else:
                runs.append(_net_run(net, lambda n, l, r: n(l, r, 0), batches, torch.float32))
    finally:
        N.uninstall()
        torch.use_deterministic_algorithms(det)
    assert spy.calls["rag_conv3d_cc16_fwd"] > 0 and spy.calls["rag_conv3d_cc16_bwd"] > 0, spy.calls
    ours, again = runs
    assert torch.equal(ours[0], again[0])
    for i in (1, 2):
        for n in ours[i]:
            assert (ours[i][n] is None and again[i][n] is None) or torch.equal(ours[i][n], again[i][n]), n

    def plain(dtype):
        r = _prepare(net_ref(MAXDISP), state, False, dtype)
        with pins.replay(r, ref[1]):
            return _net_run(r, ref_forward, batches, dtype)

    r32 = plain(torch.float32)                    # TF32 off (the autouse fixture)
    r64 = plain(torch.float64)
    pins.flips()
    rows = _compare(ours, r32, r64)
    for n, e_ours, e_ref in rows:
        print(f"  {n:32s} ours {e_ours:.2e}  fp32 {e_ref:.2e}")
    bad = [(n, e_ours, e_ref) for n, e_ours, e_ref in rows if e_ours > max(STEP_RATIO * e_ref, STEP_FLOOR)]
    assert not bad, bad
