"""The drop-in F.grid_sample on the GPU (rag_b200/grid_sample.py, csrc/grid_sample.cu): forward and both gradients against ATen
and an fp64 restatement, bitwise repeatability (runs, streams, CUDA-graph replay, one pixel holding every entry, mostly empty
pixels), non-finite grid values, torch.use_deterministic_algorithms(True) before and after, and a self-supervised training step
on the kernels against fp64.

The fp64 restatement takes its corners (floor) from the fp32 source index the kernels compute -- ((g + 1) * size - 1) / 2 with
one rounding (a fused multiply-add), or ((g + 1) / 2) * (size - 1) -- and its weights from the fp64 index, so a sample within
one rounding of a cell boundary is not counted as error: the grid gradient jumps there.  The gradients' bound is
err_ours <= max(3 err_ATen, 1e-6), err = max-norm relative to fp64."""
from copy import deepcopy

import pytest
import torch
import torch.nn.functional as F

from tests._stand_in import ReluPins, _stand_in, ref_forward
from tests._stand_in_selfsup import loss_module
from tests._util import gen, randn

pytestmark = pytest.mark.gpu

RATIO, FLOOR = 3.0, 1e-6


def _mx(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def _index32(g, size, ac):
    """The kernels' fp32 source index (before clipping)."""
    a = g.float() + 1
    if ac:
        return (a / 2) * float(size - 1)
    return (a.double() * size - 1).float() / 2            # one rounding, as the fused multiply-add


def _ref64(x, grid, padding, ac):
    """F.grid_sample(x, grid, 'bilinear', padding, ac) in fp64 with the corners of the fp32 index: differentiable in x and grid."""
    n, c, hi, wi = x.shape
    out = 0
    ixs = []
    for k, size in ((0, wi), (1, hi)):
        g = grid[..., k]
        i32 = _index32(g.detach(), size, ac)
        i64 = ((g + 1) / 2) * (size - 1) if ac else ((g + 1) * size - 1) / 2
        if padding == "border":                                     # ATen's clip: gradient 0 where i <= 0 or i >= size - 1
            i32 = i32.clamp(0, size - 1)
            i64 = torch.where((i64 <= 0) | (i64 >= size - 1), i64.detach().clamp(0, size - 1), i64)
        ixs.append((torch.floor(i32).long(), i64))
    (x0, ix), (y0, iy) = ixs
    flat = x.reshape(n, c, hi * wi)
    wx = ((x0 + 1) - ix, ix - x0)
    wy = ((y0 + 1) - iy, iy - y0)
    for dx, dy in ((0, 0), (1, 0), (0, 1), (1, 1)):                # nw, ne, sw, se
        xx, yy = x0 + dx, y0 + dy
        w = wx[dx] * wy[dy]
        ok = (xx >= 0) & (xx < wi) & (yy >= 0) & (yy < hi)
        idx = (yy.clamp(0, hi - 1) * wi + xx.clamp(0, wi - 1)).reshape(n, 1, -1).expand(n, c, -1)
        v = flat.gather(2, idx).reshape(n, c, *xx.shape[1:])
        out = out + v * (w * ok).unsqueeze(1)
    return out


def _grid(kind, n, ho, wo, hi, wi, g, ac):
    """Sampling grids [n, ho, wo, 2]."""
    if kind == "random":
        return torch.rand(n, ho, wo, 2, generator=g) * 2.2 - 1.1
    if kind in ("identity", "centres"):
        # identity: each output pixel samples its own input pixel (ho, wo = hi, wi); centres: input pixel centres of a
        # resized grid, points that land exactly on a pixel (and on the edges) in the fp32 index
        xs = torch.randint(0, wi, (n, ho, wo), generator=g) if kind == "centres" else torch.arange(wo).expand(n, ho, wo)
        ys = torch.randint(0, hi, (n, ho, wo), generator=g) if kind == "centres" else torch.arange(ho).view(1, ho, 1).expand(n, ho, wo)
        if kind == "centres":
            xs[:, :, 0], ys[:, 0, :] = 0, 0
            xs[:, :, -1], ys[:, -1, :] = wi - 1, hi - 1
        if ac:
            return torch.stack([2 * xs / (wi - 1) - 1, 2 * ys / (hi - 1) - 1], -1).float()
        return torch.stack([(2 * xs + 1) / wi - 1, (2 * ys + 1) / hi - 1], -1).float()
    if kind == "edges":
        # exactly -1 and 1 (and just inside / outside) on both axes
        vals = torch.tensor([-1.0, 1.0, -1.0 + 1e-7, 1.0 - 1e-7, -1.0 - 1e-7, 1.0 + 1e-7, 0.0])
        return vals[torch.randint(0, len(vals), (n, ho, wo, 2), generator=g)]
    if kind == "stereo":
        # x shifted left by a disparity map (up to a quarter of the width, some samples off the image), y = the row
        xs = torch.arange(wo).view(1, 1, wo).float() - torch.rand(n, ho, wo, generator=g) * wi / 4
        ys = torch.arange(ho).view(1, ho, 1).float().expand(n, ho, wo)
        return torch.stack([2 * xs / (wi - 1) - 1, 2 * ys / (hi - 1) - 1], -1).float()
    if kind in ("upsample", "downsample"):
        xs = torch.linspace(-1, 1, wo).view(1, 1, wo).expand(n, ho, wo)
        ys = torch.linspace(-1, 1, ho).view(1, ho, 1).expand(n, ho, wo)
        return torch.stack([xs, ys], -1).contiguous().float()
    raise ValueError(kind)


# (grid kind, N, C, input H x W, output H x W)
CASES = [("identity", 1, 3, (12, 20), (12, 20)), ("stereo", 3, 3, (16, 40), (16, 40)), ("random", 3, 12, (9, 13), (7, 11)),
         ("random", 1, 32, (24, 32), (10, 14)), ("upsample", 1, 1, (5, 7), (17, 23)), ("downsample", 3, 12, (30, 41), (8, 9)),
         ("centres", 1, 3, (11, 17), (6, 9)), ("edges", 3, 1, (6, 10), (5, 8)), ("stereo", 1, 32, (24, 64), (24, 64))]
MODES = [("zeros", False), ("zeros", True), ("border", False), ("border", True)]


@pytest.mark.parametrize("mode", MODES, ids=lambda m: f"{m[0]}-ac{int(m[1])}")
@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-N{c[1]}C{c[2]}")
def test_forward_and_gradients_vs_aten_and_fp64(case, mode):
    from rag_b200 import _cabi
    from rag_b200.grid_sample import grid_sample

    kind, n, c, (hi, wi), (ho, wo) = case
    padding, ac = mode
    g = gen(1000 + CASES.index(case) * 4 + MODES.index(mode))
    x0 = randn((n, c, hi, wi), g).cuda()
    g0 = _grid(kind, n, ho, wo, hi, wi, g, ac).cuda()
    go = randn((n, c, ho, wo), g).cuda()
    kw = dict(mode="bilinear", padding_mode=padding, align_corners=ac)

    x, grid = x0.clone().requires_grad_(True), g0.clone().requires_grad_(True)
    n0 = _cabi.launch_count()
    out = grid_sample(x, grid, **kw)
    assert _cabi.launch_count() - n0 == 1
    out.backward(go)
    xa, ga = x0.clone().requires_grad_(True), g0.clone().requires_grad_(True)
    ref = _aten(xa, ga, padding, ac)
    ref.backward(go)
    x64, g64 = x0.double().requires_grad_(True), g0.double().requires_grad_(True)
    r64 = _ref64(x64, g64, padding, ac)
    r64.backward(go.double())

    assert out.shape == ref.shape and out.is_contiguous()
    bits = torch.equal(out, ref)
    print(f"\n{kind} N{n} C{c} {padding} ac={ac}: forward {'= ATen bit for bit' if bits else f'vs ATen {_mx(out, ref):.2e}'}; "
          f"ggrid {'= ATen' if torch.equal(grid.grad, ga.grad) else f'vs ATen {_mx(grid.grad, ga.grad):.2e}'}; "
          f"gin vs fp64 ours {_mx(x.grad, x64.grad):.2e} ATen {_mx(xa.grad, x64.grad):.2e}; "
          f"ggrid vs fp64 ours {_mx(grid.grad, g64.grad):.2e} ATen {_mx(ga.grad, g64.grad):.2e}")
    assert _mx(out.detach(), ref.detach()) <= 1e-6
    assert _mx(out.detach(), r64.detach()) <= max(RATIO * _mx(ref.detach(), r64.detach()), FLOOR)
    for name, ours, aten, want in (("gin", x.grad, xa.grad, x64.grad), ("ggrid", grid.grad, ga.grad, g64.grad)):
        e_ours, e_aten = _mx(ours, want), _mx(aten, want)
        assert e_ours <= max(RATIO * e_aten, FLOOR), f"{name}: ours {e_ours:.2e}, ATen {e_aten:.2e}"


def _run(x0, g0, go, padding="zeros", ac=False):
    from rag_b200.grid_sample import grid_sample

    x, grid = x0.clone().requires_grad_(True), g0.clone().requires_grad_(True)
    out = grid_sample(x, grid, padding_mode=padding, align_corners=ac)
    out.backward(go)
    return out.detach(), x.grad, grid.grad


def _same(a, b):
    return all(torch.equal(u, v) for u, v in zip(a, b))


@pytest.mark.parametrize("kind", ["stereo", "one pixel", "mostly outside"])
def test_bitwise_repeatable(kind):
    """Two runs, a second stream and a CUDA-graph replay give the same bits.  'one pixel': every sample reads the same input
    pixel (one segment holds every entry); 'mostly outside': 95 % of the samples are off the image (most pixels empty)."""
    g = gen(77)
    n, c, h, w = 2, 12, 48, 96
    x0 = randn((n, c, h, w), g).cuda()
    go = torch.randn(n, c, h, w, generator=g).mul(torch.exp(3 * torch.randn(n, c, h, w, generator=g))).cuda()   # wide range
    if kind == "stereo":
        g0 = _grid("stereo", n, h, w, h, w, g, True)
    elif kind == "one pixel":
        g0 = torch.full((n, h, w, 2), 0.0)           # align_corners=False: index (size - 1) / 2 -> the centre pixel
        g0[..., 0], g0[..., 1] = (2 * 40 + 1) / w - 1, (2 * 20 + 1) / h - 1
    else:
        g0 = torch.rand(n, h, w, 2, generator=g) * 2 + 1.05
        keep = torch.rand(n, h, w, generator=g) < 0.05
        g0[keep] = torch.rand(int(keep.sum()), 2, generator=g) * 2 - 1
    g0 = g0.cuda()
    first = _run(x0, g0, go)
    assert _same(first, _run(x0, g0, go))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        other = _run(x0, g0, go)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    assert _same(first, other)
    if kind == "one pixel":
        assert (first[1][:, :, 20, 40] != 0).all()
    # CUDA graph: forward and backward captured, replayed
    from rag_b200.grid_sample import grid_sample

    x, grid = x0.clone().requires_grad_(True), g0.clone().requires_grad_(True)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                        # warm-up outside the capture
        grid_sample(x, grid, align_corners=False).backward(go)
    torch.cuda.current_stream().wait_stream(s)
    x.grad = grid.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = grid_sample(x, grid, align_corners=False)
        out.backward(go)
    graph.replay()
    torch.cuda.synchronize()
    assert _same(first, (out.detach(), x.grad, grid.grad))


def _aten(x, grid, padding, ac):
    """ATen's own grid_sampler_2d kernel.  F.grid_sample sends zeros padding with align_corners=True on CUDA to cuDNN's sampler
    instead (when cuDNN accepts the tensors); the kernels' contract is ATen's kernel."""
    return torch.grid_sampler_2d(x, grid, 0, {"zeros": 0, "border": 1}[padding], ac)


def test_non_finite_grid_values_match_aten():
    """NaN and +-inf grid entries (and ones beyond the int range) read nothing out of bounds and give the values of ATen's own
    kernel.  cuDNN's sampler, which F.grid_sample uses for zeros padding with align_corners=True, differs there: a NaN grid
    entry makes its output NaN, where ATen's kernel and ours treat the sample as out of range (0)."""
    g = gen(5)
    n, c, h, w = 2, 3, 8, 12
    x0 = randn((n, c, h, w), g).cuda()
    go = randn((n, c, h, w), g).cuda()
    g0 = torch.rand(n, h, w, 2, generator=g) * 2 - 1
    bad = [float("nan"), float("inf"), -float("inf"), 3e9, -3e9, 1e38]
    for i, v in enumerate(bad):
        g0[0, i, 2, i % 2] = v
        g0[1, i, 5, 0] = g0[1, i, 5, 1] = v
    g0 = g0.cuda()
    for padding, ac in MODES:
        ours = _run(x0, g0, go, padding, ac)
        xa, ga = x0.clone().requires_grad_(True), g0.clone().requires_grad_(True)
        ref = _aten(xa, ga, padding, ac)
        ref.backward(go)
        fg = F.grid_sample(x0, g0, padding_mode=padding, align_corners=ac)
        print(f"\n{padding} ac={ac}: NaN outputs: ours {int(ours[0].isnan().sum())}, ATen kernel {int(ref.isnan().sum())}, "
              f"F.grid_sample {int(fg.isnan().sum())}")
        for a, b, name in zip(ours, (ref.detach(), xa.grad, ga.grad), ("out", "gin", "ggrid")):
            assert torch.equal(a.isnan(), b.isnan()), (padding, ac, name)
            fin = ~b.isnan()
            assert _mx(a[fin], b[fin]) <= 1e-6, (padding, ac, name, _mx(a[fin], b[fin]))


def test_routing_on_the_device():
    """Routed calls launch the kernels; every other call is F.grid_sample itself (bit-identical, no launch)."""
    from rag_b200 import _cabi
    from rag_b200.grid_sample import grid_sample

    g = gen(13)
    x, grid = randn((2, 3, 6, 8), g).cuda(), (torch.rand(2, 5, 7, 2, generator=g) * 2 - 1).cuda()
    for kw in (dict(align_corners=True), dict(padding_mode="border", align_corners=False)):
        n0 = _cabi.launch_count()
        out = grid_sample(x, grid, **kw)
        assert _cabi.launch_count() - n0 == 1 and _mx(out, F.grid_sample(x, grid, **kw)) <= 1e-6
    through = [(x, grid, dict(mode="nearest", align_corners=True)), (x, grid, dict(mode="bicubic", align_corners=True)),
               (x, grid, dict(padding_mode="reflection", align_corners=True)), (x.double(), grid.double(), dict(align_corners=True)),
               (x.contiguous(memory_format=torch.channels_last), grid, dict(align_corners=True)),
               (x[:, :, :, ::2], grid, dict(align_corners=True)),
               (randn((1, 2, 4, 6, 8), g).cuda(), (torch.rand(1, 3, 5, 7, 3, generator=g) * 2 - 1).cuda(), dict(align_corners=True))]
    for xx, gg, kw in through:
        n0 = _cabi.launch_count()
        out = grid_sample(xx, gg, **kw)
        assert _cabi.launch_count() - n0 == 0, kw
        assert torch.equal(out, F.grid_sample(xx, gg, **kw)), kw


def test_deterministic_mode_before_and_after():
    """With the mode on, ATen's grid_sample backward raises (what the feature fixes); the drop-in runs under it and gives the
    bits it gives without it.  Both align_corners: F.grid_sample takes cuDNN's sampler for zeros padding with
    align_corners=True and ATen's kernel otherwise; what each does under the mode is printed."""
    g = gen(17)
    x0 = randn((2, 3, 24, 48), g).cuda()
    go = randn((2, 3, 24, 48), g).cuda()
    raised = {}
    for ac in (True, False):
        g0 = _grid("stereo", 2, 24, 48, 24, 48, g, ac).cuda()
        free = _run(x0, g0, go, "zeros", ac)
        was = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
        try:
            torch.use_deterministic_algorithms(True)
            for name, fn in (("F.grid_sample", lambda x: F.grid_sample(x, g0, align_corners=ac)),
                             ("ATen kernel", lambda x: _aten(x, g0, "zeros", ac))):
                xa = x0.clone().requires_grad_(True)
                try:
                    fn(xa).backward(go)
                    raised[(name, ac)] = False
                except RuntimeError as e:
                    assert "deterministic" in str(e)
                    raised[(name, ac)] = True
            moded = _run(x0, g0, go, "zeros", ac)
        finally:
            torch.use_deterministic_algorithms(was[0], warn_only=was[1])
        assert _same(free, moded), ac
    print(f"\nbackward raises under deterministic mode: {raised}")
    if not any(raised.values()):
        pytest.skip("this torch raises for no grid_sample backward under deterministic mode; the drop-in was checked")


# ---------------------------------------------------------------------------------------------------------------------
# A self-supervised training step on the kernels under torch.use_deterministic_algorithms(True)
# ---------------------------------------------------------------------------------------------------------------------
MAXDISP = 48


def _selfsup_step(net, forward, loss_mod, left, right):
    pred = forward(net, left, right)
    loss = loss_mod.photometric(left, right, pred)
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}
    return loss.detach(), pred.detach(), grads


def test_selfsup_training_step_deterministic_and_vs_fp64(monkeypatch):
    """install(every flag, grid_sample=True) on the stand-in network with the stand-in self-supervised loss, under
    deterministic mode: two seeded steps are bit-identical, every grid_sample call took the kernels, and pred and every
    parameter gradient are within max(3 err_fp32, 1e-6) of fp64 (plain forward of the same module tree, ReLU decisions pinned)."""
    from rag_b200 import grid_sample as G
    from rag_b200 import network as N
    from rag_b200 import pointwise_conv

    old_tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    monkeypatch.setattr(pointwise_conv, "MIN_VOXELS", 0)
    mine, ref = _stand_in(), _stand_in()
    loss_mine, loss_ref = loss_module(), loss_module()
    g = gen(41)
    left, right = torch.rand(2, 3, 48, 96, generator=g).cuda(), torch.rand(2, 3, 48, 96, generator=g).cuda()
    calls = []
    orig_apply = G.GridSampleFn.apply

    def spy(*a):
        calls.append(tuple(a[0].shape))
        return orig_apply(*a)

    was = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    pins = ReluPins()
    N.uninstall()
    try:
        rag_model, ops3d, cells = mine
        N.install(rag_model, None, ops3d, fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True,
                  resample=True, resample_modules=(cells,), grid_sample=True, grid_sample_modules=(loss_mine,))
        torch.manual_seed(9)
        net = rag_model.Network(MAXDISP, k=4, level12=True).cuda().train()
        state = deepcopy(net.state_dict())
        monkeypatch.setattr(G.GridSampleFn, "apply", spy)
        n_fwd = {"n": 0}
        plain_gs = F.grid_sample
        monkeypatch.setattr(F, "grid_sample", lambda *a, **k: (n_fwd.__setitem__("n", n_fwd["n"] + 1), plain_gs(*a, **k))[1])
        torch.use_deterministic_algorithms(True)
        results = []
        for step in range(2):
            net.load_state_dict(state)
            net.zero_grad(set_to_none=True)
            if step == 0:
                with pins.record(net):
                    results.append(_selfsup_step(net, lambda m, l, r: m(l, r, 0), loss_mine, left, right))
            else:
                results.append(_selfsup_step(net, lambda m, l, r: m(l, r, 0), loss_mine, left, right))
    finally:
        torch.use_deterministic_algorithms(was[0], warn_only=was[1])
        N.uninstall()
    monkeypatch.undo()
    assert calls == [(2, 3, 48, 96)] * 2 and n_fwd["n"] == 0, (calls, n_fwd)      # every warp on the kernels
    (l1, p1, g1), (l2, p2, g2) = results
    assert torch.equal(l1, l2) and torch.equal(p1, p2) and set(g1) == set(g2)
    assert all(torch.equal(g1[k], g2[k]) for k in g1), [k for k in g1 if not torch.equal(g1[k], g2[k])]
    assert torch.isfinite(l1) and all(torch.isfinite(v).all() for v in g1.values())

    def plain(dtype):
        net_r = ref[0].Network(MAXDISP, k=4, level12=True).to("cuda", dtype).train()
        net_r.load_state_dict(state)
        with pins.replay(net_r, ref[1]):
            return _selfsup_step(net_r, ref_forward, loss_ref, left.to(dtype), right.to(dtype))

    try:
        r32, r64 = plain(torch.float32), plain(torch.float64)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_tf32
    flips = pins.flips()
    rows = [("pred", _mx(p1, r64[1]), _mx(r32[1], r64[1]))]
    assert set(g1) == set(r32[2]) == set(r64[2])
    rows += [(k, _mx(g1[k], r64[2][k]), _mx(r32[2][k], r64[2][k])) for k in g1]
    print(f"\n{len(rows)} tensors, {flips} ReLU decisions differing from fp64 (rounding noise); loss {l1.item():.6f}")
    for k, a, b in rows:
        print(f"  {k:32s} ours {a:.2e}  fp32 {b:.2e}")
    bad = [(k, a, b) for k, a, b in rows if a > max(RATIO * b, FLOOR)]
    assert not bad, f"further from fp64 than max({RATIO} x fp32, {FLOOR}): {bad}"
