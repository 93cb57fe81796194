"""GPU parity of the rows adjacent to the hot path: loss + metric sums, input staging, the network
drop-in functions, the path router and the host-buffer pipeline."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import rag_oracle as O
from tests import _grids
from tests._mirror_net import MirrorNet, arch
from tests._util import gen, randn

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def test_metrics_golden(dev):
    from rag_b200 import metrics as M

    z = np.load(os.path.join(GOLDEN, "metrics_b3_h12_w20.npz"))
    est, gt = torch.from_numpy(z["est"]).to(dev), torch.from_numpy(z["gt"]).to(dev)
    sums = M.loss_metric_sums(est, gt, float(z["maxdisp"]))
    vec = M.metrics_from_sums(sums).cpu().numpy()
    for i, k in enumerate(M.KEYS):
        assert abs(vec[i] - float(z[k])) <= 2e-6 * max(1.0, abs(float(z[k]))), k


def test_metrics_vs_oracle_and_skip_rules(dev):
    from rag_b200 import metrics as M

    g = gen(31)
    b, h, w, md = 4, 48, 96, 192
    gt = torch.rand(b, h, w, generator=g) * 260 - 30
    gt[1] = torch.where(torch.rand(h, w, generator=g) < 0.98, torch.full((h, w), 250.0), gt[1])  # skipped image
    est = gt + 3 * torch.randn(b, h, w, generator=g)
    ref = O.loss_and_metrics_ref(est, gt, md)
    sums = M.loss_metric_sums(est.to(dev), gt.to(dev), md)
    # integer sums are exact
    mask = (gt < md) & (gt > 0)
    assert torch.equal(sums[:, 0].cpu(), mask.flatten(1).sum(1).double())
    assert torch.equal(sums[:, 1].cpu(), (gt > 0).flatten(1).sum(1).double())
    vec = M.metrics_from_sums(sums).cpu().numpy()
    for i, k in enumerate(M.KEYS):
        assert abs(vec[i] - ref[k]) <= 2e-6 * max(1.0, abs(ref[k])), k
    # every image skipped -> metrics are 0, loss still defined
    gt2 = torch.full((2, 8, 8), 250.0)
    gt2[:, 0, 0] = 5.0
    s2 = M.loss_metric_sums(torch.zeros(2, 8, 8, device=dev), gt2.to(dev), md)
    v2 = M.metrics_from_sums(s2).cpu().numpy()
    assert np.all(v2[1:] == 0) and abs(v2[0] - 4.5) < 1e-6
    # deterministic
    assert torch.equal(sums, M.loss_metric_sums(est.to(dev), gt.to(dev), md))


def test_masked_smooth_l1_forward_backward(dev):
    from rag_b200 import metrics as M

    g = gen(32)
    gt = (torch.rand(3, 24, 40, generator=g) * 260 - 30).to(dev)
    est = (gt + 2 * torch.randn(3, 24, 40, generator=g).to(dev)).requires_grad_(True)
    loss, sums = M.masked_smooth_l1(est, gt, 192)
    (loss * 2.5).backward()
    est2 = est.detach().clone().requires_grad_(True)
    mask = (gt < 192) & (gt > 0)
    ref = F.smooth_l1_loss(est2[mask], gt[mask], reduction="mean")
    (ref * 2.5).backward()
    assert abs(loss.item() - ref.item()) <= 1e-6 * abs(ref.item())
    assert torch.allclose(est.grad, est2.grad, rtol=1e-6, atol=1e-12)
    assert not est.grad[~mask].any()


def test_normalize_pad_golden_bit_exact(dev):
    from rag_b200.staging import normalize_pad

    z = np.load(os.path.join(GOLDEN, "stage_h10_w14.npz"))
    img = torch.from_numpy(z["img"])[None].to(dev)
    out = normalize_pad(img, 10 + int(z["top_pad"]), 14 + int(z["right_pad"]))
    assert np.array_equal(out[0].cpu().numpy(), z["out"])
    # reference-size case against the oracle restatement: 400x880 -> 480x960, batch of 2
    rng = np.random.RandomState(3)
    big = rng.randint(0, 256, size=(2, 400, 880, 3), dtype=np.uint8)
    out = normalize_pad(torch.from_numpy(big).to(dev), 480, 960).cpu().numpy()
    for i in range(2):
        assert np.array_equal(out[i], O.normalize_pad_ref(big[i], 80, 80))


def _oracle_forward(net, left, right, task_arch, md):
    x, y = net.feature(left, task_arch), net.feature(right, task_arch)
    return O.disp_head_ref(net.matching(O.cost_volume_ref(x, y, md), task_arch), md)


def test_network_dropin_forward_backward(dev):
    from rag_b200 import network as N
    from rag_b200.modules import Disp

    torch.manual_seed(0)
    md = 48
    net = MirrorNet(Disp(md), md).to(dev)
    g = gen(33)
    left, right = randn((2, 3, 36, 60), g).to(dev), randn((2, 3, 36, 60), g).to(dev)
    for fwd, args in ((N.network_forward, (0, arch(1))), (N.network_search_forward, (0, None)), (N.basic_network_forward, (None, None))):
        net.zero_grad()
        if fwd is N.basic_network_forward:
            class _B(MirrorNet):  # BasicNetwork.feature/matching take (x, ops)
                pass
            out = fwd(net, left, right, None, None)
            ta = None
        else:
            out = fwd(net, left, right, *args)
            ta = args[1] if isinstance(args[1], dict) else None
        assert out.shape == (2, 36, 60)
        ref = _oracle_forward(net, left, right, ta, md)
        assert (out - ref).abs().max().item() <= 1e-4
        w = randn((2, 36, 60), g).to(dev)
        (out * w).sum().backward()
        got = [p.grad.clone() for p in net.parameters() if p.grad is not None]
        net.zero_grad()
        (_oracle_forward(net, left, right, ta, md) * w).sum().backward()
        want = [p.grad.clone() for p in net.parameters() if p.grad is not None]
        assert len(got) == len(want) and len(got) > 0
        for a, b_ in zip(got, want):
            assert (a - b_).abs().max().item() <= 2e-4 * max(1.0, b_.abs().max().item())


def test_network_works_with_reference_style_disp_attribute(dev):
    """``install()`` leaves already-built networks with the reference's own Disp object in ``self.disp``;
    the patched forward must still take the fused path (it keys on maxdisp, not on the module)."""
    from rag_b200 import network as N

    class RefStyleDisp(torch.nn.Module):  # stands in for the reference's Disp instance
        def forward(self, x):
            raise AssertionError("the reference head must not be called")

    net = MirrorNet(RefStyleDisp(), 48).to(dev)
    out = N.network_forward(net, randn((1, 3, 18, 24), gen(1)).to(dev), randn((1, 3, 18, 24), gen(2)).to(dev), 0)
    assert out.shape == (1, 18, 24)


def test_path_router(dev):
    from rag_b200 import network as N
    from rag_b200.modules import Disp

    torch.manual_seed(1)
    md = 48
    net = MirrorNet(Disp(md), md, n_paths=3).to(dev).eval()
    net.forward = lambda l, r, t, ta=None, path=None: N.network_forward(net, l, r, t, ta, path)
    g = gen(34)
    left, right = randn((5, 3, 18, 36), g).to(dev), randn((5, 3, 18, 36), g).to(dev)
    ids = [2, 0, 2, 1, 0]
    out = N.PathRouter(net, [arch(0), arch(1), arch(2)]).route(left, right, ids)
    for i, u in enumerate(ids):
        with torch.no_grad():
            one = N.network_forward(net, left[i:i + 1], right[i:i + 1], u, arch(u))
        assert torch.equal(out[i], one[0])
    with pytest.raises(IndexError):
        N.PathRouter(net, [arch(0)]).route(left, right, ids)


def test_host_pipeline_matches_oracle(dev):
    from rag_b200.pipeline import HostPipeline

    g = gen(35)
    md = 96
    x, y = randn((2, 12, 8, 32), g), randn((2, 12, 8, 32), g)
    cl = randn((2, 1, 32, 8, 32), g)
    pipe = HostPipeline(md, dev)
    slots = []
    for i in range(5):                              # more steps than slots: the double buffering wraps around
        slot = pipe.acquire(x.shape, cl.shape)
        assert slot.x.is_pinned() and slot.h_in.is_pinned() and slot.x.data_ptr() == slot.h_in.data_ptr()
        slot.x.copy_(x * (i + 1)), slot.y.copy_(y), slot.cost_lr.copy_(cl * (i + 1))
        pipe.submit(slot, keep_volume=True)
        slots.append(slot)
    pipe.drain()
    ref = O.disp_head_ref(cl * 5, md)
    assert (slots[-1].result["disp"] - ref).abs().max().item() <= 1e-4
    assert torch.equal(slots[-1].keep.cpu(), O.cost_volume_ref(x * 5, y, md))
    assert slots[-1].h2d_bytes == 4 * (2 * x.numel() + cl.numel()) and slots[-1].d2h_bytes == 4 * ref.numel()
    assert torch.equal(pipe.run(x * 5, y, cl * 5), slots[-1].result["disp"])


def test_host_train_pipeline_matches_the_functions(dev):
    from rag_b200 import functional as F_
    from rag_b200.pipeline import HostTrainPipeline

    g = gen(36)
    md = 96
    x, y = randn((2, 12, 8, 32), g), randn((2, 12, 8, 32), g)
    cl = randn((2, 1, 32, 8, 32), g)
    gd = randn((2, 24, 96), g)
    gcost = randn((2, 24, 32, 8, 32), g).to(dev)
    pipe = HostTrainPipeline(md, dev)
    for _ in range(3):
        slot = pipe.acquire(x.shape, cl.shape)
        slot.x.copy_(x), slot.y.copy_(y), slot.cost_lr.copy_(cl), slot.gdisp.copy_(gd)
        pipe.submit(slot, gcost)
    pipe.drain()
    disp, stats = F_.disp_head_forward(cl.to(dev), md, True)
    gcl = F_.disp_head_backward(cl.to(dev), gd.to(dev), disp, stats, md)
    gx, gy = F_.cost_volume_backward(gcost, 12)
    r = slot.result
    assert torch.equal(r["disp"], disp.cpu()) and torch.equal(r["gcost_lr"], gcl.cpu())
    assert torch.equal(r["gx"], gx.cpu()) and torch.equal(r["gy"], gy.cpu())
    gx_ref, gy_ref = O.cost_volume_grad_closed(gcost.cpu().numpy(), 12)
    assert np.array_equal(r["gx"].numpy(), gx_ref) and np.array_equal(r["gy"].numpy(), gy_ref)


# (id prefix, (B, C, Hf, Wf, maxdisp, steps)).  The small shape gives every persistent CTA at most one item; at the bench's
# training shape (B=4 288x576) the co-resident head kernels loop over tiles / CTA-tasks (fewer steps there bound the memory)
OVERLAP_SHAPES = [("", (2, 12, 9, 64, 96, 10)), ("B4-288x576-", (4, 12, 96, 192, 192, 3))]
OVERLAP_CASES = [(p, s, k) for p, s in OVERLAP_SHAPES for k in ("launch-order", "coresident", "slim-volume")]


@pytest.mark.parametrize("shape, schedule", [(s, k) for _, s, k in OVERLAP_CASES], ids=[p + k for p, _, k in OVERLAP_CASES])
def test_overlapped_train_path_matches_the_serial_functions(dev, shape, schedule):
    """Every schedule of the two-stream training step (rag_b200.pipeline.SCHEDULES: persistent / co-resident kernel
    variants) gives the bits of the plain serial calls."""
    from rag_b200 import functional as F_
    from rag_b200.pipeline import OverlappedTrainPath

    b, c, hf, wf, md, steps = shape
    dl = md // 3
    if shape == OVERLAP_SHAPES[1][1]:
        print(f"\npersistent head forward: {_grids.loops(*_grids.head_fwd(b, hf, wf, dev))}; "
              f"backward: {_grids.loops(*_grids.head_bwd(b, dl, hf, wf, dev))}")
    g = gen(37)
    op = OverlappedTrainPath(md, dev, schedule=schedule)
    x, y = randn((b, c, hf, wf), g).to(dev), randn((b, c, hf, wf), g).to(dev)
    cl = randn((b, 1, dl, hf, wf), g).to(dev)
    gd = randn((b, 3 * hf, 3 * wf), g).to(dev)
    gcost = randn((b, 2 * c, dl, hf, wf), g).to(dev)
    outs = [op.step(x, y, cl, gcost, gd) for _ in range(steps)]
    op.join()
    torch.cuda.synchronize()
    disp, stats = F_.disp_head_forward(cl, md, True)
    want = (F_.cost_volume_forward(x, y, md // 3, variant=0), disp, F_.disp_head_backward(cl, gd, disp, stats, md)) + F_.cost_volume_backward(gcost, c, variant=1)
    for o in outs:
        for a, b_ in zip(o, want):
            assert torch.equal(a, b_)
