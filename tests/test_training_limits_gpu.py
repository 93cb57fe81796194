"""The three training paths at the edges of the shape domain include/rag_b200.h states for them (O <= 32, D >= 3,
8 <= W <= 1016 with W % 4 == 0, B <= 32767, H <= 65535), against fp64 compositions of the reference layer:

* the fused stem (``FusedStemFn``: rag_cv_stem_fwd + csrc/bn3d.cu + rag_cv_stem_bwd) through ``stem_forward``;
* the interior 3x3x3 ConvBR_3d (``ConvBR3dFn``: conv3d_cc + bn3d) through ``matching_forward``;
* the pointwise ConvBR_3d (``PointwiseBR3dFn``: conv3d_pw + bn3d) through ``pointwise_forward``, or through
  ``batchnorm.apply`` directly below ``pointwise_conv.MIN_VOXELS``;
* the BatchNorm kernels alone on a channel whose mean is 100 times its standard deviation.

Each case runs one training step, forward and backward, in train() and in eval() BatchNorm.  Its ReLU decision is pinned to
ours (``ref_stem_masked`` / ``_masked``); a decision fp64 would take otherwise must sit within 1e-5 of zero.  The output,
the input gradients, the weight and affine gradients and both running statistics must be within 1e-5 max-norm relative of
fp64; the error of plain fp32 (cuDNN, TF32 off) is printed beside ours.  Each case asserts that the kernels ran (the
``grad_fn`` type or a launch count) and the launch geometry it was written for (tests/_grids.py restates it from the host
code; tests/test_work_loops_cpu.py checks that against the sources).  One step past each limit, the routing predicate must
refuse the shape and the fallback must give the reference layer's result.

The stem's maps kernel asks for (2U + 5) * Wf * 4 bytes of shared memory, U = the largest of 8, 4, 2, 1 dividing Df: over
48 KB from Wf = 588 at U = 8 and Wf = 948 at U = 4, which the cases straddle."""
import copy
import time
import zlib

import pytest
import torch
import torch.nn.functional as F

from tests import _grids
from tests.test_fused_stem_gpu import ref_stem, ref_stem_masked
from tests.test_matching_conv_gpu import _fp32_convs, _layer, _masked, _mx  # noqa: F401  (_fp32_convs: autouse, TF32 off)
from tests.test_pointwise_conv_gpu import _layer as _pw_layer

pytestmark = pytest.mark.gpu
NAMES_STEM = ["out", "gx", "gy", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]
NAMES = ["out", "gx", "gweight", "ggamma", "gbeta", "running_mean", "running_var"]


@pytest.fixture(autouse=True)
def _measured(request):
    """Frees the case's temporaries and prints its wall time and peak memory."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    print(f"  [{request.node.name}: {time.perf_counter() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB]")
    torch.cuda.empty_cache()


def _seed(case):
    return zlib.crc32(repr(case).encode()) % 997


def _randn(shape, g):
    return torch.randn(shape, generator=g, device="cuda")


def _gout(shape, g):
    return _randn(shape, g) * (torch.rand(shape, generator=g, device="cuda") < 0.7)     # some exact zeros upstream


def _step(fn, layer, inputs, gout, dtype):
    """One forward and backward of ``fn(layer copy, *inputs)`` in ``dtype``: ([out, input grads..., gweight, ggamma, gbeta,
    running_mean, running_var], the pre-activation if ``fn`` returns it, the output's grad_fn type name)."""
    lay = copy.deepcopy(layer).to(dtype)
    xs = [t.to(dtype).clone().requires_grad_(True) for t in inputs]
    out = fn(lay, *xs)
    pre = None
    if isinstance(out, tuple):
        out, pre = out
    kind = type(out.grad_fn).__name__
    out.backward(gout.to(dtype))
    return ([out.detach()] + [x.grad for x in xs] + [lay.conv.weight.grad, lay.bn.weight.grad, lay.bn.bias.grad,
                                                      lay.bn.running_mean.clone(), lay.bn.running_var.clone()],
            None if pre is None else pre.detach(), kind)


def _compare(label, names, layer, inputs, gout, ours_fn, plain_fn, skip=()):
    """Our step against the plain composition in fp64 and in fp32, the ReLU decision pinned to ours; returns the grad_fn
    type name of our output."""
    ours, _, kind = _step(ours_fn, layer, inputs, gout, torch.float32)
    mask = ours[0] > 0
    ref64, pre64, _ = _step(lambda lay, *xs: plain_fn(lay, mask, *xs), layer, inputs, gout, torch.float64)
    flips = (pre64 > 0) != mask
    n_flips = int(flips.sum())
    flip = pre64[flips].abs().max().item() if n_flips else 0.0
    del pre64, flips
    fp32, _, _ = _step(lambda lay, *xs: plain_fn(lay, mask, *xs), layer, inputs, gout, torch.float32)
    errs = {n: (_mx(a, r), _mx(f, r)) for n, a, f, r in zip(names, ours, fp32, ref64) if n not in skip}
    print(f"\n{label}: vs fp64 ours / fp32: " + ", ".join(f"{n} {e:.2e} / {e32:.2e}" for n, (e, e32) in errs.items())
          + f"; {n_flips} ReLU decisions differ from fp64 (largest |pre| {flip:.1e})")
    assert flip <= 1e-5, "a ReLU decision differs from fp64 beyond rounding"
    for n, (e, e32) in errs.items():
        assert e <= 1e-5, f"{n}: ours {e:.3e} (fp32 {e32:.3e})"
    return kind, ours, ref64, mask


# ---------------------------------------------------------------------------------------------------------------------
# the fused stem
# ---------------------------------------------------------------------------------------------------------------------
# (B, Hf, Wf, maxdisp, O): Df = maxdisp / 3; U and the maps kernel's shared memory follow from (Df, Wf)
STEM_CASES = [
    (1, 1, 1016, 192, 12),      # the widest row, U = 8: 85,344 bytes of shared memory in the maps kernel
    (1, 5, 1016, 192, 12),
    (1, 1, 1016, 192, 32),      # O = 32: the weight kernel's 672 threads
    (1, 5, 1016, 192, 32),      # ... and the inputs kernel's 198 KB of shared memory
    (1, 2, 584, 192, 12),       # U = 8: the last width under 48 KB
    (1, 2, 588, 192, 12),       # U = 8: the first width over it
    (1, 2, 944, 108, 12),       # Df = 36, U = 4: the last width under 48 KB
    (1, 2, 948, 108, 12),       # U = 4: the first width over it
    (2, 4, 132, 54, 12),        # Df = 18, U = 2
    (2, 4, 132, 99, 12),        # Df = 33, U = 1
    (2, 6, 8, 48, 12),          # the narrowest row (Wf < Df)
    (32767, 1, 8, 9, 1),        # B at its limit: the inputs kernel's grid z and the weight kernel's grid y are 2B = 65534
    (1, 65535, 8, 9, 1),        # Hf at its limit: the maps and BatchNorm row kernels' grid x
]
STEM_U = {(192, 1016): 8, (192, 584): 8, (192, 588): 8, (108, 944): 4, (108, 948): 4, (54, 132): 2, (99, 132): 1}


def _stem_layer(o, g):
    torch.manual_seed(o)                    # the conv weight's default initialisation
    return _layer(24, o, g)


@pytest.mark.parametrize("case", STEM_CASES, ids=lambda c: "B{}-Hf{}-Wf{}-md{}-O{}".format(*c))
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_stem_training_at_the_limits_vs_fp64(case, mode):
    from rag_b200.fused_stem import VirtualCostVolume, _train_fusable, stem_forward

    b, hf, wf, md, o = case
    df = int(md / 3)
    u, maps_grid, maps_threads, maps_smem = _grids.stem_maps(b, o, df, hf, wf)
    if (md, wf) in STEM_U:
        assert u == STEM_U[(md, wf)]
        assert (maps_smem > _grids.SMEM_DEFAULT) == (u == 8 and wf >= 588 or u == 4 and wf >= 948)
    if o == 32:
        assert _grids.stem_bwd_weight(b, o, hf)[1] == 672 and _grids.stem_bwd_inputs(b, o, hf, wf)[1] > 196 * 1024
    if b == 32767:
        assert _grids.stem_bwd_inputs(b, o, hf, wf)[0][2] == 65534 and _grids.stem_bwd_weight(b, o, hf)[0][1] == 65534
    if hf == 65535:
        assert maps_grid[0] == 65535 and _grids.bn3d_rows(b, o, hf)[0] == 65535
    g = torch.Generator(device="cuda").manual_seed(_seed((case, mode)))
    layer = _stem_layer(o, torch.Generator().manual_seed(_seed(case))).train(mode == "train")
    x0, y0 = _randn((b, 12, hf, wf), g), _randn((b, 12, hf, wf), g)
    gout = _gout((b, o, df, hf, wf), g)
    assert _train_fusable(layer, VirtualCostVolume(x0, y0, md))
    kind, *_ = _compare(f"stem B={b} Hf={hf} Wf={wf} Df={df} O={o} U={u} ({maps_smem} B smem) {mode}", NAMES_STEM, layer, (x0, y0), gout,
                        lambda lay, x, y: stem_forward(lay, VirtualCostVolume(x, y, md)),
                        lambda lay, mask, x, y: ref_stem_masked(x, y, lay, md, mask))
    assert kind == "FusedStemFnBackward", kind


# ---------------------------------------------------------------------------------------------------------------------
# the interior 3x3x3 ConvBR_3d (conv3d_cc)
# ---------------------------------------------------------------------------------------------------------------------
# ((C, O), (B, D, H, W))
CC_CASES = ([((c, c), (1, 3, h, 1016)) for c in (4, 8, 12) for h in (1, 3)]
            + [((12, 12), (32767, 3, 1, 8)),      # B at its limit: the forward's grid z = B * ceil(D/8) = 32767
               ((12, 12), (1, 3, 65535, 8))])     # H at its limit


@pytest.mark.parametrize("pair, shape", CC_CASES, ids=[f"{p[0]}x{p[1]}-" + "x".join(map(str, s)) for p, s in CC_CASES])
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_matching_conv_training_at_the_limits_vs_fp64(pair, shape, mode):
    from rag_b200.matching_conv import matching_forward, qualifies

    c, o = pair
    b, d, h, w = shape
    grid = _grids.cc_fwd(b, d, h, w)
    assert grid[2] == b and _grids.bn3d_rows(b, o, h) == (h, o, b)
    g = torch.Generator(device="cuda").manual_seed(_seed((pair, shape, mode)))
    torch.manual_seed(c)
    layer = _layer(c, o, torch.Generator().manual_seed(_seed((pair, shape)))).train(mode == "train")
    x0 = _randn((b, c, d, h, w), g)
    gout = _gout((b, o, d, h, w), g)
    assert qualifies(layer, x0.clone().requires_grad_(True))
    kind, *_ = _compare(f"conv3d_cc {pair} {list(shape)} grid {grid} {mode}", NAMES, layer, (x0,), gout, matching_forward,
                        lambda lay, mask, x: _masked(lay, x, mask))
    assert kind == "ConvBR3dFnBackward", kind


# ---------------------------------------------------------------------------------------------------------------------
# the pointwise ConvBR_3d (conv3d_pw)
# ---------------------------------------------------------------------------------------------------------------------
PW_CASES = [((1, 1), (1, 3, 2, 1016)), ((64, 32), (1, 3, 2, 1016)),
            ((64, 32), (32767, 3, 1, 8)),        # B at its limit: the forward's grid y = B
            ((64, 32), (1, 3, 65535, 8))]        # H at its limit


@pytest.mark.parametrize("pair, shape", PW_CASES, ids=[f"{p[0]}x{p[1]}-" + "x".join(map(str, s)) for p, s in PW_CASES])
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_pointwise_conv_training_at_the_limits_vs_fp64(pair, shape, mode):
    from rag_b200 import batchnorm
    from rag_b200.pointwise_conv import MIN_VOXELS, PointwiseBR3dFn, pointwise_forward, qualifies

    c, o = pair
    b, d, h, w = shape
    grid = _grids.pw_fwd(b, d, h, w)
    assert grid[1] == b and _grids.bn3d_rows(b, o, h) == (h, o, b)
    g = torch.Generator(device="cuda").manual_seed(_seed((pair, shape, mode)))
    torch.manual_seed(c)
    layer = _pw_layer(c, o, torch.Generator().manual_seed(_seed((pair, shape)))).train(mode == "train")
    x0 = _randn((b, c, d, h, w), g)
    gout = _gout((b, o, d, h, w), g)
    routed = b * d * h * w >= MIN_VOXELS
    assert qualifies(layer, x0.clone().requires_grad_(True)) == routed
    if routed:
        fn = pointwise_forward
    else:                                   # under the routing's volume floor: the autograd function itself
        def fn(lay, x):
            return batchnorm.apply(PointwiseBR3dFn, lay.bn, x, lay.conv.weight)
    # one input and one output channel under batch statistics: the layer is invariant to the weight's scale, so the exact
    # weight gradient is ~0 (eps alone keeps it off zero) and its relative error measures cancellation; bounded below instead
    skip = ("gweight",) if c == 1 and mode == "train" else ()
    kind, ours, ref64, mask = _compare(f"conv3d_pw {pair} {list(shape)} grid {grid} {mode}{'' if routed else ' (direct)'}", NAMES,
                                       layer, (x0,), gout, fn, lambda lay, mask, x: _masked(lay, x, mask), skip)
    assert kind == "PointwiseBR3dFnBackward", kind
    if skip:
        lay64, x64 = copy.deepcopy(layer).double(), x0.double()
        z64 = lay64.conv(x64).detach().requires_grad_(True)
        (lay64.bn(z64) * mask.double()).backward(gout.double())
        assert (ours[2].double() - ref64[2]).abs().max().item() <= 1e-5 * (z64.grad.abs() * x64.abs()).sum().item()


# ---------------------------------------------------------------------------------------------------------------------
# one step past each limit: refused by the routing, the reference layer's result from the fallback
# ---------------------------------------------------------------------------------------------------------------------
def _past(shape, at):
    """(inside, past): ``shape`` with the entries of ``at`` (index -> (inside value, past value)) set."""
    inside, past = list(shape), list(shape)
    for i, (a, p) in at.items():
        inside[i], past[i] = a, p
    return tuple(inside), tuple(past)


def _fallback_matches_the_reference(label, names, layer, inputs, gout, ours_fn, ref_fn):
    ours, _, kind = _step(ours_fn, layer, inputs, gout, torch.float32)
    ref, _, _ = _step(ref_fn, layer, inputs, gout, torch.float32)
    errs = {n: _mx(a, r) for n, a, r in zip(names, ours, ref)}
    print(f"\n{label}: fallback vs the reference layer: " + ", ".join(f"{n} {e:.1e}" for n, e in errs.items()))
    for n, e in errs.items():
        assert e <= 1e-5, f"{n}: {e:.3e}"
    return kind


# (B, Hf, Wf, maxdisp, O) -> the entry past its limit
STEM_PAST = {"Wf=1020": ((1, 1, None, 9, 12), {2: (1016, 1020)}),
             "Df=2": ((1, 2, 8, None, 12), {3: (9, 6)}),
             "O=33": ((1, 2, 8, 9, None), {4: (32, 33)}),
             "B=32768": ((None, 1, 8, 9, 1), {0: (32767, 32768)}),
             "Hf=65536": ((1, None, 8, 9, 1), {1: (65535, 65536)})}


@pytest.mark.parametrize("which", list(STEM_PAST))
def test_stem_one_step_past_each_limit_falls_back(which):
    from rag_b200.fused_stem import VirtualCostVolume, _train_fusable, stem_forward

    shape, at = STEM_PAST[which]
    inside, past = _past(shape, at)
    for s, fusable in ((inside, True), (past, False)):
        b, hf, wf, md, o = s
        x = torch.empty((b, 12, hf, wf), device="cuda")
        assert _train_fusable(_stem_layer(o, torch.Generator().manual_seed(0)).train(), VirtualCostVolume(x, x, md)) == fusable, s
    b, hf, wf, md, o = past
    g = torch.Generator(device="cuda").manual_seed(_seed(past))
    layer = _stem_layer(o, torch.Generator().manual_seed(_seed(past))).train()
    x0, y0 = _randn((b, 12, hf, wf), g), _randn((b, 12, hf, wf), g)
    gout = _gout((b, o, int(md / 3), hf, wf), g)
    kind = _fallback_matches_the_reference(f"stem {which} {past}", NAMES_STEM, layer, (x0, y0), gout,
                                           lambda lay, x, y: stem_forward(lay, VirtualCostVolume(x, y, md)),
                                           lambda lay, x, y: ref_stem(x, y, lay, md))
    assert kind != "FusedStemFnBackward", kind


# ((C, O), (B, D, H, W)) -> the entry past its limit; O = 33 has no conv3d_cc instantiation to step past
CC_PAST = {"W=1020": ((1, 3, 1, None), {3: (1016, 1020)}),
           "D=2": ((1, None, 2, 8), {1: (3, 2)}),
           "B=32768": ((None, 3, 1, 8), {0: (32767, 32768)}),
           "H=65536": ((1, 3, None, 8), {2: (65535, 65536)})}


@pytest.mark.parametrize("which", list(CC_PAST))
def test_matching_conv_one_step_past_each_limit_falls_back(which):
    from rag_b200 import _cabi
    from rag_b200.matching_conv import matching_forward, qualifies

    shape, at = CC_PAST[which]
    inside, past = _past(shape, at)
    torch.manual_seed(4)
    layer = _layer(4, 4, torch.Generator().manual_seed(_seed(past))).train()
    for s, ok in ((inside, True), (past, False)):
        assert qualifies(layer, torch.empty((s[0], 4) + s[1:], device="cuda").requires_grad_(True)) == ok, s
    g = torch.Generator(device="cuda").manual_seed(_seed(past))
    x0 = _randn((past[0], 4) + past[1:], g)
    gout = _gout((past[0], 4) + past[1:], g)
    n0 = _cabi.launch_count()
    kind = _fallback_matches_the_reference(f"conv3d_cc {which} {past}", NAMES, layer, (x0,), gout, matching_forward,
                                           lambda lay, x: lay(x))
    assert _cabi.launch_count() == n0 and kind != "ConvBR3dFnBackward", kind


# ((C, O), (B, D, H, W)) -> the entry past its limit
PW_PAST = {"W=1020": ((4, 4), (1, 3, 1, None), {3: (1016, 1020)}),
           "D=2": ((4, 4), (1, None, 2, 8), {1: (3, 2)}),
           "O=33": ((4, None), (1, 3, 2, 8), {}),
           "B=32768": ((4, 4), (None, 3, 1, 8), {0: (32767, 32768)}),
           "H=65536": ((4, 4), (1, 3, None, 8), {2: (65535, 65536)})}


@pytest.mark.parametrize("which", list(PW_PAST))
def test_pointwise_conv_one_step_past_each_limit_falls_back(which, monkeypatch):
    """The routing's volume floor is lifted here, so that only the limit under test can refuse the shape."""
    from rag_b200 import _cabi, pointwise_conv
    from rag_b200.pointwise_conv import pointwise_forward, qualifies

    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)
    (c, o), shape, at = PW_PAST[which]
    inside, past = _past(shape, at)
    outs = (32, 33) if o is None else (o, o)
    for s, oo, ok in ((inside, outs[0], True), (past, outs[1], False)):
        lay = _pw_layer(c, oo, torch.Generator().manual_seed(0)).train()
        assert qualifies(lay, torch.empty((s[0], c) + s[1:], device="cuda").requires_grad_(True)) == ok, (s, oo)
    o = outs[1]
    torch.manual_seed(o)
    layer = _pw_layer(c, o, torch.Generator().manual_seed(_seed(past))).train()
    g = torch.Generator(device="cuda").manual_seed(_seed(past))
    x0 = _randn((past[0], c) + past[1:], g)
    gout = _gout((past[0], o) + past[1:], g)
    n0 = _cabi.launch_count()
    kind = _fallback_matches_the_reference(f"conv3d_pw {which} {(c, o)} {past}", NAMES, layer, (x0,), gout, pointwise_forward,
                                           lambda lay, x: lay(x))
    assert _cabi.launch_count() == n0 and kind != "PointwiseBR3dFnBackward", kind


# ---------------------------------------------------------------------------------------------------------------------
# the BatchNorm kernels alone, on a channel whose mean is 100 times its standard deviation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 32, 4, 8, 64), (1, 32, 3, 1, 8)], ids=lambda s: "x".join(map(str, s)))
def test_bn3d_on_an_offset_channel_vs_fp64(shape):
    """bn3d forms the variance as E[z^2] - mean^2 from fp64 sums of fp32 partials: fp32 partials of z^2 itself would lose
    (mean/std)^2 times their rounding to that cancellation, so they square z minus a shift.  Forward and backward of ``batchnorm`` (train(), momentum 1, so the running statistics ARE the batch
    statistics) against nn.BatchNorm3d + ReLU in fp64, torch's fp32 BatchNorm printed beside ours; ours must be within
    max(3 x fp32's error, 1e-5) of fp64."""
    from rag_b200 import _cabi, batchnorm

    b, o, d, h, w = shape
    g = torch.Generator(device="cuda").manual_seed(_seed(shape))
    std = 0.5 + torch.rand(o, generator=g, device="cuda")
    z = (std.view(1, o, 1, 1, 1) * (100.0 + _randn(shape, g))).contiguous()
    gout = _gout(shape, g)
    gamma, beta = 0.5 + torch.rand(o, generator=g, device="cuda"), 0.3 * _randn((o,), g)
    rm0, rv0 = 0.2 * _randn((o,), g), 0.5 + torch.rand(o, generator=g, device="cuda")
    assert _grids.bn3d_rows(b, o, h) == (h, o, b)
    rm, rv = rm0.clone(), rv0.clone()
    n0 = _cabi.launch_count()
    out = z.clone()
    bn = batchnorm.forward(z, out, gamma, beta, rm, rv, True, True, 1.0, 1e-5)
    _, ggamma, gbeta, gz = batchnorm.backward(gout, z, bn, True, want_gz=True)
    assert _cabi.launch_count() - n0 == 8             # moments (2), finalize, normalise | sums (2), consts, gz
    mask = out > 0
    ours = [out, gz, ggamma, gbeta, rm, rv]

    def plain(dtype):
        m = torch.nn.BatchNorm3d(o, momentum=1.0).cuda().to(dtype).train()
        with torch.no_grad():
            m.weight.copy_(gamma); m.bias.copy_(beta); m.running_mean.copy_(rm0); m.running_var.copy_(rv0)
        zz = z.to(dtype).clone().requires_grad_(True)
        pre = m(zz)
        (pre * mask.to(dtype)).backward(gout.to(dtype))
        return [(pre * mask.to(dtype)).detach(), zz.grad, m.weight.grad, m.bias.grad, m.running_mean, m.running_var], pre.detach()

    ref64, pre64 = plain(torch.float64)
    fp32, _ = plain(torch.float32)
    flips = (pre64 > 0) != mask
    assert not flips.any() or pre64[flips].abs().max().item() <= 1e-5, "a ReLU decision differs from fp64 beyond rounding"
    names = ["out", "gz", "ggamma", "gbeta", "running_mean", "running_var"]
    errs = {n: (_mx(a, r), _mx(f, r)) for n, a, f, r in zip(names, ours, fp32, ref64)}
    print(f"\nbn3d {list(shape)}, mean = 100 std: vs fp64 ours / torch fp32: " + ", ".join(f"{n} {e:.2e} / {e32:.2e}" for n, (e, e32) in errs.items()))
    for n, (e, e32) in errs.items():
        assert e <= max(3 * e32, 1e-5), f"{n}: ours {e:.3e}, torch fp32 {e32:.3e}"
