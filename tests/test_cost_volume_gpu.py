"""GPU parity of the cost-volume kernels against the oracle and the golden vectors.  Bit-exact."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import rag_oracle as O
from tests._util import gen, randn, wide_grad

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def F_():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from rag_b200 import functional

    return functional


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "cv_*.npz"))), ids=os.path.basename)
def test_golden(F_, path):
    z = np.load(path)
    md = int(z["maxdisp"])
    x = torch.from_numpy(z["x"]).cuda().requires_grad_(True)
    y = torch.from_numpy(z["y"]).cuda().requires_grad_(True)
    cost = F_.cost_volume(x, y, md)
    assert torch.equal(cost.cpu(), torch.from_numpy(z["cost"]))
    cost.backward(torch.from_numpy(z["gcost"]).cuda())
    assert torch.equal(x.grad.cpu(), torch.from_numpy(z["gx"]))
    assert torch.equal(y.grad.cpu(), torch.from_numpy(z["gy"]))


SHAPES = [
    # (B, C, Hf, Wf, maxdisp)   covers V=4/2/1 paths, Wf<Df, ragged tiles, Df not multiple of 4
    (1, 12, 96, 192, 192),   # config 1/3 (288x576)
    (2, 12, 20, 320, 192),   # config 2 width
    (1, 12, 8, 416, 288),    # config 5 width, maxdisp 288
    (2, 3, 7, 294, 192),     # literal ceil(880/3) width: Wf % 4 == 2
    (1, 2, 5, 37, 30),       # odd width, Df = 10
    (1, 4, 3, 10, 48),       # Wf < Df
    (3, 1, 1, 4, 3),         # Df = 1
    (1, 12, 33, 64, 100),    # Df = 33 (not a multiple of 4), ragged row tile
    (2, 5, 11, 36, 48),      # ragged row tiles (Hf % R != 0), Df = 16
    (1, 2, 6, 64, 192),      # Df == Wf (last disparity keeps a single column)
    (1, 12, 4, 1024, 192),   # widest row the slim persistent geometry takes (256 vectors: one row per tile)
    (2, 3, 5, 8, 96),        # Wf < Df on the lean kernels
    (1, 2, 1, 12, 6),        # Hf = 1, Df = 2
    (2, 12, 3, 96, 195),     # Df = 65: one disparity past the last full disparity chunk
    (1, 1, 50, 44, 96),      # C = 1, 11 vectors per row: many ragged rows per tile
    (1, 5, 17, 132, 120),    # Df = 40, Hf prime
    (3, 2, 2, 4, 192),       # Wf = 4: one vector per row, Df = 64 >> Wf
]


@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_forward_bit_exact(F_, shape):
    b, c, hf, wf, md = shape
    g = gen(hash(shape) % 1000)
    x, y = randn((b, c, hf, wf), g), randn((b, c, hf, wf), g)
    ref = O.cost_volume_ref(x, y, md)
    # None = default with a workspace (persistent lean kernel), "plain" = the stateless entry point without one
    for variant in (None, "plain", 0) + ((1, 3, 5) if wf % 4 == 0 else ()):
        if variant == "plain":
            out = F_.cost_volume_forward(x.cuda(), y.cuda(), int(md / 3), workspace=False)
        else:
            out = F_.cost_volume_forward(x.cuda(), y.cuda(), int(md / 3), variant=variant)
        assert torch.equal(out.cpu(), ref), f"variant {variant}"


@pytest.mark.parametrize("shape", SHAPES, ids=str)
def test_backward_bit_exact(F_, shape):
    b, c, hf, wf, md = shape
    g = gen(1 + hash(shape) % 1000)
    gc = wide_grad((b, 2 * c, int(md / 3), hf, wf), g)
    gx_ref, gy_ref = O.cost_volume_grad_closed(gc.numpy(), c)
    # 2 = persistent grid, 3 = the shared-memory cp.async ring (RAG_CV_BWD_SLIM)
    for variant in (None, 0, 1) + ((2, 3) if wf % 4 == 0 else ()):
        gx, gy = F_.cost_volume_backward(gc.cuda(), c, variant=variant)
        assert np.array_equal(gx.cpu().numpy(), gx_ref), f"gx variant {variant}"
        assert np.array_equal(gy.cpu().numpy(), gy_ref), f"gy variant {variant}"


def test_backward_matches_autograd_of_reference_loop(F_):
    """The closed-form oracle is itself pinned to autograd of the literal loop on CPU; here the
    kernel is compared to autograd of the same literal loop run by PyTorch on the GPU."""
    g = gen(5)
    b, c, hf, wf, md = 1, 12, 6, 48, 96
    x = randn((b, c, hf, wf), g).cuda().requires_grad_(True)
    y = randn((b, c, hf, wf), g).cuda().requires_grad_(True)
    gc = wide_grad((b, 2 * c, md // 3, hf, wf), g).cuda()
    O.cost_volume_ref(x, y, md).backward(gc)
    gx, gy = F_.cost_volume_backward(gc, c)
    assert torch.equal(gx, x.grad) and torch.equal(gy, y.grad)


def test_full_size_properties(F_):
    """BASELINE config 2 per-GPU size (B=8, 480x960 -> 160x320, Df=64): size-independent checks.
    forward: every d-plane equals the shifted/masked input (checked with torch ops on the GPU);
    backward: linearity + ones-gradient closed form (count of valid d per column)."""
    b, c, hf, wf, df = 8, 12, 160, 320, 64
    g = gen(11)
    x, y = randn((b, c, hf, wf), g).cuda(), randn((b, c, hf, wf), g).cuda()
    cost = F_.cost_volume_forward(x, y, df)
    assert cost.shape == (b, 2 * c, df, hf, wf)
    for d in (0, 1, 2, 3, 4, 5, 31, 62, 63):
        assert torch.equal(cost[:, :c, d, :, d:], x[..., d:])
        assert torch.equal(cost[:, c:, d, :, d:], y[..., : wf - d])
        assert not cost[:, :, d, :, :d].any()
    # checksum of checksums: sum over the volume == sum_d of the valid input part (fp64)
    tot = cost.double().sum().item()
    exp = sum(x[..., d:].double().sum().item() + y[..., : wf - d].double().sum().item() for d in range(df))
    assert abs(tot - exp) <= 1e-6 * max(1.0, abs(exp))
    del cost
    ones = torch.ones((b, 2 * c, df, hf, wf), device="cuda")
    gx, gy = F_.cost_volume_backward(ones, c)
    w = torch.arange(wf, device="cuda")
    cnt_x = torch.clamp(w + 1, max=df).float()
    cnt_y = torch.clamp(wf - w, max=df).float()
    assert torch.equal(gx, cnt_x.expand_as(gx)) and torch.equal(gy, cnt_y.expand_as(gy))


def test_empty_and_maximum_sizes(F_):
    """Empty batch (the reference's zero-fill of an empty tensor) and BASELINE config 4's size:
    32 pairs at 480x960 -> a 10 GB volume; config 5's largest: 384x1248 at maxdisp 288."""
    e = F_.cost_volume_forward(torch.zeros(0, 12, 4, 8, device="cuda"), torch.zeros(0, 12, 4, 8, device="cuda"), 64)
    assert e.shape == (0, 24, 64, 4, 8)
    gx, gy = F_.cost_volume_backward(torch.zeros(0, 24, 64, 4, 8, device="cuda"), 12)
    assert gx.shape == (0, 12, 4, 8) and gy.shape == (0, 12, 4, 8)
    for (b, c, hf, wf, df) in ((32, 12, 160, 320, 64), (4, 12, 128, 416, 96)):
        g = gen(b)
        x, y = randn((b, c, hf, wf), g).cuda(), randn((b, c, hf, wf), g).cuda()
        cost = F_.cost_volume_forward(x, y, df)
        for d in (0, 7, df - 1):
            assert torch.equal(cost[:, :c, d, :, d:], x[..., d:]) and torch.equal(cost[:, c:, d, :, d:], y[..., : wf - d])
            assert not cost[:, :, d, :, :d].any()
        assert torch.equal(cost[b - 1, c + 3, 5, hf - 1, 5:], y[b - 1, 3, hf - 1, : wf - 5])
        del cost
        torch.cuda.empty_cache()


def test_autograd_module_and_hygiene(F_):
    import copy
    import pickle

    from rag_b200.modules import CostVolume

    m = CostVolume(192)
    assert len(m.state_dict()) == 0 and len(list(m.parameters())) == 0
    m2 = pickle.loads(pickle.dumps(copy.deepcopy(m)))
    g = gen(3)
    x = randn((2, 12, 4, 80), g).cuda().requires_grad_(True)
    y = randn((2, 12, 4, 80), g).cuda().requires_grad_(True)
    out = m2(x, y)
    out.sum().backward()
    assert x.grad is not None and y.grad is not None
    # non-contiguous inputs are accepted (made contiguous), like the reference's slice copies
    xt = randn((2, 12, 80, 4), g).cuda().transpose(2, 3)
    assert torch.equal(m(xt, xt).cpu(), O.cost_volume_ref(xt.cpu().contiguous(), xt.cpu().contiguous(), 192))


def test_errors_are_loud(F_):
    with pytest.raises(RuntimeError):
        F_.cost_volume(torch.zeros(1, 2, 3, 4), torch.zeros(1, 2, 3, 4))  # CPU tensors
    with pytest.raises(RuntimeError):
        F_.cost_volume(torch.zeros(1, 2, 3, 4, device="cuda", dtype=torch.float16), torch.zeros(1, 2, 3, 4, device="cuda", dtype=torch.float16))
    with pytest.raises(RuntimeError):
        F_.cost_volume(torch.zeros(1, 2, 3, 4, device="cuda"), torch.zeros(1, 2, 3, 5, device="cuda"))
    with pytest.raises(RuntimeError):
        F_.cost_volume_forward(torch.zeros(1, 2, 3, 4, device="cuda"), torch.zeros(1, 2, 3, 4, device="cuda"), 4, variant=99)
    # retired ids (2: lean persistent 256 x 2, 4: TMA bulk stores) are refused, with a workspace and on a lean-capable shape
    for v in (2, 4):
        with pytest.raises(RuntimeError, match="unknown variant"):
            F_.cost_volume_forward(torch.zeros(1, 2, 3, 4, device="cuda"), torch.zeros(1, 2, 3, 4, device="cuda"), 4, variant=v)


def test_deterministic(F_):
    g = gen(9)
    gc = wide_grad((2, 24, 64, 12, 96), g).cuda()
    a = F_.cost_volume_backward(gc, 12)
    b = F_.cost_volume_backward(gc, 12)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
