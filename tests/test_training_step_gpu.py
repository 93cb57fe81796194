"""A whole training step on the kernels against fp64, gradient by gradient.

``install(fuse_stem, upsample, matching_convs, pointwise_convs, resample)`` on the stand-in network of ``tests/_stand_in.py``
(the growable network's structure, with cells): one step (two in the continual-learning configuration) of ours, compared with
the plain forward of the same module tree (``_stand_in.ref_forward``: no install(), the oracle's cost volume and head) in fp32
(ref32) and in fp64 (ref64) on the GPU.  The three load the same state_dict.  Compared: ``pred``, every parameter's gradient
by name, and every BatchNorm's running statistics.  Each error is the relative max-norm against ref64; ours must be no
further from fp64 than plain fp32 is: err_ours <= max(3 err_ref32, 2e-5).  The floor matters where fp32 storage alone sets the
error: a running statistic's error is about one rounding of the stored value (up to 6e-8), and a ref32 that happens to round
closer makes the ratio meaningless (7e-9 against 6e-8 seen on a B200).

TF32 is off for cuDNN and matmul throughout (``_fp32`` below): in ref32 and in ours, whose Feature Net and fallthrough
layers run on cuDNN.

The ReLU decisions of the three runs are pinned to ours (``_stand_in.ReluPins``): fp32 and fp64 disagree on a few
pre-activations near 0, and each disagreement is worth O(1e-2) of max-norm in the gradients, which says nothing about
either run's arithmetic.  Every decision fp64 would take otherwise must be rounding noise (|pre| <= 1e-5 of the max).
The backward is driven by a fixed upstream gradient on ``pred`` with about 30 % exact zeros (what the smooth-L1 loss's mask
produces) rather than by the loss, whose |d| < 1 branch would be one more decision to pin.

The seams this covers and the per-layer tests do not: ``torch.cat``'s backward handing each producer a channel slice
(non-contiguous for B > 1), one layer's output feeding the next with in-place ops between, kernel and cuDNN layers in one
step, routing predicates that could silently send a layer to cuDNN (spies assert each layer's path), and frozen eval-mode
layers beside trainable ones."""
from collections import Counter
from copy import deepcopy

import pytest
import torch
import torch.nn as nn

from tests._stand_in import AUTOGRAD, ReluPins, Routes, _stand_in, ref_forward
from tests._util import gen, randn, sparse_grad

pytestmark = pytest.mark.gpu

MAXDISP = 48
RATIO, FLOOR = 3.0, 2e-5

# every ConvBR_3d of the stand-in (with its level-12 branch) and the path it takes when the kernels apply
KERNEL_PATHS = {"stem3d0": "stem", "stem3d1": "matching", "cell3d.pre": "pointwise", "cell3d.op0": "matching",
                "cell3d.op1": "matching", "cell3d.op2": "matching", "last_6_3d": "pointwise", "last_12_3d": "pointwise",
                "last_3_3d": "last_conv"}

CONFIGS = {
    # name: (k, B, image H x W, frozen, steps, ConvBR_3d layers that fall through to cuDNN)
    "k4": (4, 2, (48, 96), False, 1, ()),
    "k8": (8, 2, (48, 96), False, 1, ()),
    # level-3 W = 36, level-6 W = 18, level-12 W = 9: the level-6 and level-12 layers are not W % 4 == 0
    "mixed": (4, 2, (48, 108), False, 1, ("cell3d.op1", "last_6_3d", "last_12_3d")),
    "frozen": (4, 2, (48, 96), True, 2, ()),
    "b1": (4, 1, (48, 96), False, 1, ()),
    "b3": (4, 3, (48, 96), False, 1, ()),
}
# the continual-learning freeze: an earlier task's layers, requires_grad=False with BatchNorm in eval().  last_6_3d sits behind
# trainable layers, so gradients flow through a frozen eval-mode layer to cell3d.op1.
FROZEN = ("stem2d", "cell2d", "stem3d0", "stem3d1", "last_6_3d")


@pytest.fixture(autouse=True)
def _fp32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _mx(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def _state(rag_model, k, seed):
    """The shared state_dict: default initialisation, BatchNorm parameters and running statistics randomised."""
    g = gen(seed)
    torch.manual_seed(seed)
    net = rag_model.Network(MAXDISP, k=k, level12=True)
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, nn.modules.batchnorm._BatchNorm):
                c = m.num_features
                m.weight.copy_(0.5 + torch.rand(c, generator=g)); m.bias.copy_(0.3 * torch.randn(c, generator=g))
                m.running_mean.copy_(0.2 * torch.randn(c, generator=g)); m.running_var.copy_(0.5 + torch.rand(c, generator=g))
    return deepcopy(net.state_dict())


def _prepare(net, state, frozen, dtype):
    net = net.to("cuda", dtype)
    net.load_state_dict(state)
    net.train()
    if frozen:
        for name in FROZEN:
            layer = getattr(net, name)
            layer.requires_grad_(False)
            for m in layer.modules():
                if isinstance(m, nn.modules.batchnorm._BatchNorm):
                    m.eval()
        net.cell3d.op0.bn.momentum = None             # a trainable layer on the cumulative average
    net.zero_grad(set_to_none=True)
    return net


def _run(net, forward, batches, dtype):
    """The steps (gradients accumulate over them, as without zero_grad between steps); pred of the last one, every
    parameter's gradient and every buffer afterwards."""
    for left, right, gpred in batches:
        pred = forward(net, left.to(dtype), right.to(dtype))
        pred.backward(gpred.to(dtype))
    grads = {n: p.grad.detach().clone() if p.grad is not None else None for n, p in net.named_parameters()}
    return pred.detach(), grads, {n: b.detach().clone() for n, b in net.named_buffers()}


def _compare(ours, r32, r64):
    """[(tensor, err_ours, err_ref32)] against ref64; asserts the None pattern of the gradients, the names and the counters."""
    rows = [("pred", _mx(ours[0], r64[0]), _mx(r32[0], r64[0]))]
    for i in (1, 2):
        assert list(ours[i]) == list(r32[i]) == list(r64[i])
        for n in ours[i]:
            a, b, c = ours[i][n], r32[i][n], r64[i][n]
            assert (a is None) == (b is None) == (c is None), f"{n}: gradient None in one run and not in another"
            if a is None:
                continue
            if n.endswith("num_batches_tracked"):
                assert int(a) == int(b) == int(c), f"{n}: {int(a)} {int(b)} {int(c)}"
                continue
            rows.append((n, _mx(a, c), _mx(b, c)))
    return rows


@pytest.mark.parametrize("config", list(CONFIGS))
def test_training_step_vs_fp64(config, monkeypatch):
    from rag_b200 import network as N
    from rag_b200 import pointwise_conv

    k, b, (h, w), frozen, steps, cudnn = CONFIGS[config]
    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)        # the stand-in is small: its 1x1x1 layers take the kernels
    mine, ref = _stand_in(), _stand_in()                         # install() binds into the first only
    state = _state(ref[0], k, 31 + list(CONFIGS).index(config))
    g = gen(1009 + list(CONFIGS).index(config))
    batches = [(randn((b, 3, h, w), g).cuda(), randn((b, 3, h, w), g).cuda(), sparse_grad((b, h, w), g, keep=0.7).cuda())
               for _ in range(steps)]
    pins = ReluPins()
    N.uninstall()
    try:
        rag_model, ops3d, cells = mine
        N.install(rag_model, None, ops3d, fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True,
                  resample=True, resample_modules=(cells,))
        net = _prepare(rag_model.Network(MAXDISP, k=k, level12=True), state, frozen, torch.float32)
        routes = Routes(monkeypatch, net)
        fns = {}

        def autograd_fn(name):
            def hook(m, args, out):
                fns.setdefault(name, set()).add(type(out.grad_fn).__name__ if out.requires_grad else None)
            return hook

        handles = [m.register_forward_hook(autograd_fn(n)) for n, m in net.named_modules() if n in KERNEL_PATHS]
        with pins.record(net):
            ours = _run(net, lambda n, l, r: n(l, r, 0), batches, torch.float32)
        for hd in handles:
            hd.remove()
    finally:
        N.uninstall()
    monkeypatch.undo()

    # every ConvBR_3d took the path it should, on its autograd function when a gradient was wanted
    want = {n: {p} for n, p in KERNEL_PATHS.items() if n not in cudnn}
    assert routes.layers == want, routes.layers
    for n, p in KERNEL_PATHS.items():
        if n not in cudnn:
            assert all(f is None or f.startswith(AUTOGRAD[p]) for f in fns[n]), (n, fns[n])
            assert frozen and n in ("stem3d0", "stem3d1") or None not in fns[n], (n, fns[n])
    # every resample ran on the kernels: per feature pass 2 bilinear, per matching pass 2 in the cell, 3 -> 12, upsample_12
    # and upsample_6; each backward where its input wants a gradient (not in the frozen Feature Net)
    launches = Counter(f for f, _, _ in routes.resizes)
    assert launches == Counter({"rag_bilinear_resize_fwd": 4 * steps, "rag_bilinear_resize_bwd": 0 if frozen else 4 * steps,
                                "rag_trilinear_resize_fwd": 5 * steps, "rag_trilinear_resize_bwd": 5 * steps}) - Counter(), launches
    fwd = Counter((i, o) for f, i, o in routes.resizes if f.endswith("_fwd") and not (frozen and len(i) == 2))
    assert fwd == Counter((i, o) for f, i, o in routes.resizes if f.endswith("_bwd"))

    def plain(dtype):
        r = _prepare(ref[0].Network(MAXDISP, k=k, level12=True), state, frozen, dtype)
        with pins.replay(r, ref[1]):
            return _run(r, ref_forward, batches, dtype)

    r32 = plain(torch.float32)
    r64 = plain(torch.float64)
    flips = pins.flips()
    rows = _compare(ours, r32, r64)
    worst = max(rows, key=lambda r: r[1] / max(r[2], 1e-30))
    n_pinned = sum(m.numel() for v in pins.masks.values() for m in v)
    print(f"\n{config}: {len(rows)} tensors, {n_pinned} ReLU decisions in {pins.calls()} calls pinned, {flips} differing from fp64 "
          f"(rounding noise); largest err_ours / err_ref32 = {worst[1] / max(worst[2], 1e-30):.2f} on {worst[0]}")
    for n, e_ours, e_ref in rows:
        print(f"  {n:32s} ours {e_ours:.2e}  ref32 {e_ref:.2e}")
    bad = [(n, e_ours, e_ref) for n, e_ours, e_ref in rows if e_ours > max(RATIO * e_ref, FLOOR)]
    assert not bad, f"further from fp64 than max({RATIO} x fp32, {FLOOR}): {bad}"
