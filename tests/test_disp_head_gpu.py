"""GPU parity of the disparity-head kernels.

Tolerances (BASELINE.json north_star): disparity within 1e-4 px absolute; gradient within 1e-5
relative in max-norm.  The reference's OWN fp32 result deviates from an exact (fp64) evaluation of
its formula by up to ~9e-5 px at maxdisp=192 / sigma=1 (sequential fp32 sum of p_k*k at magnitude
~100; SURVEY.md section 8a H-1), so the comparison is made three ways:
  (1) against the fp64 evaluation of the reference formula: <= 3e-5 px  (the kernel's own error; mean ~3e-6);
  (2) against the fp32 reference run by PyTorch on CPU and on this GPU: <= 1e-4 px on the golden
      and seeded cases below (deterministic inputs, so this is a hard assert, not a statistic);
  (3) at full size, where a few pixels in 10^5 of the reference itself are > 1e-4 from its own
      exact value: >= 99.9% of pixels within 1e-4 and every pixel within 1e-4 + the reference's
      own deviation from fp64 at that pixel.
"""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import rag_oracle as O
from tests._util import gen, maxnorm_rel, randn, sparse_grad

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
TOL_DISP = 1e-4
TOL_GRAD = 1e-5


@pytest.fixture(scope="module")
def F_():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from rag_b200 import functional

    return functional


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "head_*.npz"))), ids=os.path.basename)
def test_golden(F_, path):
    z = np.load(path)
    md = int(z["maxdisp"])
    cost = torch.from_numpy(z["cost"]).cuda().requires_grad_(True)
    disp = F_.disp_head(cost, md)
    out = disp.detach().cpu().numpy().astype(np.float64)
    d64, g64 = O.disp_head_grad_f64(z["cost"][:, 0], z["gdisp"], md)
    # The golden disparity is the reference's fp32 result; its own deviation from the exact value of its formula is part of
    # the fixture (it grows with maxdisp and with sigma: the sequential fp32 sum of p_k*k).  Per pixel the kernel must be
    # within 1e-4 + that deviation, the deviation itself must stay under the cap recorded here (so a regression cannot hide
    # in it), and the kernel's own error against the exact value is bounded separately.
    ref_dev = np.abs(z["disp"].astype(np.float64) - d64)
    cap = 6e-4 if "_s5" in path else (1.5e-4 if "_md288_" in path else 1e-4)
    assert ref_dev.max() <= cap, f"reference vs fp64 {ref_dev.max():.3e} exceeds the recorded cap {cap}"
    assert np.all(np.abs(out - z["disp"]) <= TOL_DISP + ref_dev)
    assert np.abs(out - d64).max() <= (1e-4 if "_s5" in path else 3e-5 * md / 192)
    disp.backward(torch.from_numpy(z["gdisp"]).cuda())
    assert maxnorm_rel(cost.grad.cpu().numpy(), z["gcost"]) <= 2 * TOL_GRAD  # vs fp32 reference (own noise 7.5e-6)
    assert maxnorm_rel(cost.grad.cpu().numpy()[:, 0], g64) <= TOL_GRAD       # vs exact


def test_regression_module_golden(F_):
    from rag_b200.modules import DisparityRegression

    for path in sorted(glob.glob(os.path.join(GOLDEN, "head_*.npz"))):
        z = np.load(path)
        md = int(z["maxdisp"])
        p = torch.from_numpy(z["p"]).cuda().requires_grad_(True)
        out = DisparityRegression(md)(p)
        assert np.abs(out.detach().cpu().numpy() - z["reg"]).max() <= TOL_DISP
        out.sum().backward()
        k = torch.arange(md, device="cuda", dtype=torch.float32).view(1, md, 1, 1)
        assert torch.equal(p.grad, k.expand_as(p.grad).contiguous())


CASES = [
    # (B, Dl, Hl, Wl, maxdisp, sigma)
    (1, 64, 32, 64, 192, 1.0),   # 96x192 output
    (2, 64, 9, 35, 192, 1.0),    # ragged vs warp/CTA tiling (Wl+1 = 36, Hl+1 = 10)
    (1, 96, 8, 40, 288, 1.0),    # maxdisp 288
    (1, 64, 16, 33, 192, 5.0),   # sigma 5 stress
    (1, 48, 6, 10, 192, 1.0),    # depth != maxdisp/3 -> generic kernel
    (1, 1, 2, 2, 3, 1.0),        # smallest x3 case
    (2, 64, 7, 36, 192, 1.0),    # tiled kernel: ragged CTA tiles (Hl % 4 != 0, Wl % 32 != 0)
    (1, 20, 5, 4, 60, 1.0),      # tiled kernel: Dl not a multiple of the 8-bin stage, one 4-wide strip
    (1, 4, 1, 1, 12, 1.0),       # single low-res pixel
]


@pytest.mark.parametrize("case", CASES, ids=str)
def test_forward_parity(F_, case):
    b, dl, hl, wl, md, sigma = case
    cost = randn((b, 1, dl, hl, wl), gen(hash(case) % 997), sigma)
    ref_cpu = O.disp_head_ref(cost, md).numpy()
    ref_gpu = O.disp_head_ref(cost.cuda(), md).cpu().numpy()
    d64, _ = O.disp_head_f64(cost[:, 0].numpy(), md)
    variants = [None, 0] + ([1] if md == 3 * dl else []) + ([2, 3, 4] if md == 3 * dl and wl % 4 == 0 else [])
    for v in variants:
        disp, stats = F_.disp_head_forward(cost.cuda(), md, want_stats=True, variant=v)
        out = disp.cpu().numpy()
        own = np.abs(out - d64).max()
        assert own <= (3e-5 * md / 192 if sigma <= 1 else 1e-4), f"variant {v}: own error {own}"
        # vs the fp32 reference: within 1e-4 px, allowing at each pixel for the reference's OWN deviation
        # from the exact value of its formula (its fp32 sum of p_k*k is good to ~1e-4 at maxdisp 192 and
        # worse at maxdisp 288 / sigma 5); and the bulk of the pixels within 1e-4 outright
        for name, ref in (("CPU", ref_cpu), ("CUDA", ref_gpu)):
            err = np.abs(out - ref)
            assert np.all(err <= TOL_DISP + np.abs(ref - d64)), f"variant {v} vs {name} reference"
            if sigma <= 1:  # the reference's fp32 noise scales with the magnitude of sum p_k*k, i.e. with maxdisp
                assert (err <= TOL_DISP * md / 192).mean() >= 0.995, f"variant {v} vs {name} reference (bulk)"
        disp2, _ = F_.disp_head_forward(cost.cuda(), md, want_stats=False, variant=v)
        assert torch.equal(disp, disp2)


@pytest.mark.parametrize("case", CASES, ids=str)
def test_backward_parity(F_, case):
    b, dl, hl, wl, md, sigma = case
    g = gen(1 + hash(case) % 997)
    cost = randn((b, 1, dl, hl, wl), g, sigma)
    gd = sparse_grad((b, 3 * hl, 3 * wl), g)
    if not gd.any():
        gd[0, 0, 0] = 1.0
    _, gref = O.disp_head_grad_ref(cost, gd, md)
    _, g64 = O.disp_head_grad_f64(cost[:, 0].numpy(), gd.numpy(), md)
    variants = [None, 0] + ([1, 2, 3] if md == 3 * dl else [])
    for vf in ([None, 0] if md != 3 * dl else [None, 0, 1] + ([2, 3] if wl % 4 == 0 else [])):
        disp, stats = F_.disp_head_forward(cost.cuda(), md, want_stats=True, variant=vf)
        for v in variants:
            try:
                gc = F_.disp_head_backward(cost.cuda(), gd.cuda(), disp, stats, md, variant=v)
            except RuntimeError as e:
                if "unknown variant" in str(e):
                    continue
                raise
            out = gc.cpu().numpy()
            assert maxnorm_rel(out[:, 0], g64) <= TOL_GRAD, f"fwd {vf} bwd {v} vs fp64"
            if np.abs(g64).max() > 1e-6 * gd.abs().max().item():   # Dl == 1: the true gradient is 0 and the
                # fp32 reference returns pure rounding noise (~1e-8); nothing to be relative to
                assert maxnorm_rel(out, gref.numpy()) <= 2 * TOL_GRAD, f"fwd {vf} bwd {v} vs fp32 reference"
            else:
                assert np.abs(out).max() <= 1e-6 * gd.abs().max().item()


@pytest.mark.parametrize("sigma", [30.0, 8000.0])
def test_large_magnitude_costs_exercise_the_rescale_path(F_, sigma):
    """An untrained Matching Net emits costs with sigma ~ 8000 (SURVEY.md section 8a H-1): the running maximum
    jumps by far more than the lazy-rescale threshold, the softmax is one-hot.  Every variant must stay
    finite and agree with the fp64 evaluation wherever that is well conditioned (a clear winner bin)."""
    g = gen(int(sigma))
    b, dl, hl, wl, md = 1, 64, 6, 36, 192
    cost = randn((b, 1, dl, hl, wl), g, sigma)
    # monotone ramps force repeated upward moves of the reference exponent
    cost[0, 0, :, 0, :] = -torch.arange(dl, dtype=torch.float32)[:, None] * sigma
    cost[0, 0, :, 1, :] = torch.arange(dl, dtype=torch.float32)[:, None] * sigma
    d64, p64 = O.disp_head_f64(cost[:, 0].numpy(), md)
    gd = sparse_grad((b, 3 * hl, 3 * wl), g, keep=1.0)
    _, g64 = O.disp_head_grad_f64(cost[:, 0].numpy(), gd.numpy(), md)
    # well conditioned = a 1-ulp change of the logits cannot move the result by more than ~1e-4
    top2 = np.sort(p64, axis=1)[:, -2:]
    clear = (top2[:, 1] > 0.999) | (sigma <= 30.0)
    for v in (None, 0, 1, 2, 3, 4):
        disp, stats = F_.disp_head_forward(cost.cuda(), md, want_stats=True, variant=v)
        out = disp.cpu().numpy()
        assert np.isfinite(out).all() and out.min() >= 0 and out.max() <= md - 1, f"variant {v}"
        tol = 2e-3 if sigma <= 30.0 else 1e-2
        assert np.abs(out - d64)[clear].max() <= tol, f"variant {v}: {np.abs(out - d64)[clear].max()}"
        assert torch.isfinite(stats).all()
        for vb in (0, 1, 2, 3):
            gc = F_.disp_head_backward(cost.cuda(), gd.cuda(), disp, stats, md, variant=vb).cpu().numpy()
            assert np.isfinite(gc).all(), f"fwd {v} bwd {vb}"
            if sigma <= 30.0:
                assert maxnorm_rel(gc[:, 0], g64) <= 5e-3, f"fwd {v} bwd {vb}"


def test_backward_with_spatially_coherent_zero_gradient(F_):
    """Sparse ground truth: whole regions with no upstream gradient take the warp-level skip path."""
    g = gen(77)
    b, dl, hl, wl, md = 2, 64, 24, 70, 192
    cost = randn((b, 1, dl, hl, wl), g)
    gd = sparse_grad((b, 3 * hl, 3 * wl), g)
    gd[:, : 3 * hl // 2] = 0          # "sky": no returns in the top half
    gd[1, :, 100:] = 0                # and a blank right part in the second image
    _, g64 = O.disp_head_grad_f64(cost[:, 0].numpy(), gd.numpy(), md)
    disp, stats = F_.disp_head_forward(cost.cuda(), md, want_stats=True)
    out0 = F_.disp_head_backward(cost.cuda(), gd.cuda(), disp, stats, md, variant=0)
    for v in (1, 2, 3):
        out1 = F_.disp_head_backward(cost.cuda(), gd.cuda(), disp, stats, md, variant=v)
        assert maxnorm_rel(out1.cpu().numpy()[:, 0], g64) <= TOL_GRAD
        assert maxnorm_rel(out1.cpu().numpy(), out0.cpu().numpy()) <= TOL_GRAD
        zero = F_.disp_head_backward(cost.cuda(), torch.zeros_like(gd).cuda(), disp, stats, md, variant=v)
        assert not zero.any()


def test_backward_deterministic_and_vs_cuda_autograd(F_):
    g = gen(21)
    cost = randn((2, 1, 64, 8, 24), g).cuda().requires_grad_(True)
    gd = sparse_grad((2, 24, 72), g).cuda()
    d1 = F_.disp_head(cost, 192)
    d1.backward(gd)
    g1 = cost.grad.clone()
    cost.grad = None
    F_.disp_head(cost, 192).backward(gd)
    assert torch.equal(g1, cost.grad)          # bitwise repeatable (two commutative contributions per element)
    _, gref = O.disp_head_grad_ref(cost.detach(), gd, 192)   # PyTorch CUDA autograd (atomicAdd, fp32)
    assert maxnorm_rel(g1.cpu().numpy(), gref.cpu().numpy()) <= 2 * TOL_GRAD


def test_upsample_matches_torch_cuda(F_):
    """Locks the lambda variant: the kernel's upsample vs F.interpolate on this GPU."""
    g = gen(4)
    cost = randn((1, 1, 64, 7, 9), g).cuda()
    ref = torch.nn.functional.interpolate(cost, [192, 21, 27], mode="trilinear", align_corners=False)[:, 0]
    up_fma = F_.upsample_trilinear(cost, 192, True)
    up_mul = F_.upsample_trilinear(cost, 192, False)
    e_fma = (up_fma - ref).abs().max().item()
    e_mul = (up_mul - ref).abs().max().item()
    print(f"upsample vs torch CUDA: fma max|d|={e_fma:.3e} equal={torch.equal(up_fma, ref)}; mul-sub max|d|={e_mul:.3e} equal={torch.equal(up_mul, ref)}")
    assert e_fma <= 2e-6
    assert e_fma <= e_mul


def test_full_size_properties(F_):
    """BASELINE config 2 per-GPU size: B=8, 160x320 low-res -> 480x960, maxdisp 192."""
    b, dl, hl, wl, md = 8, 64, 160, 320, 192
    g = gen(17)
    cost = randn((b, 1, dl, hl, wl), g).cuda()
    disp = F_.disp_head(cost, md)
    assert disp.shape == (b, 3 * hl, 3 * wl)
    assert torch.isfinite(disp).all() and disp.min() >= 0 and disp.max() <= md - 1
    # shift invariance of softmin: adding a constant to the cost leaves the disparity unchanged
    disp_s = F_.disp_head(cost + 3.0, md)
    assert (disp - disp_s).abs().max().item() <= 2e-4
    # batch independence: each pair alone gives the same bits
    one = F_.disp_head(cost[3:4].contiguous(), md)
    assert torch.equal(one[0], disp[3])
    # one pair against the fp32 CUDA reference and its fp64 evaluation
    ref = O.disp_head_ref(cost[:1], md)[0].cpu().numpy().astype(np.float64)
    d64, _ = O.disp_head_f64(cost[:1, 0].cpu().numpy(), md)
    out = disp[0].cpu().numpy().astype(np.float64)
    assert np.abs(out - d64[0]).max() <= 3e-5
    assert np.abs(out - d64[0]).mean() <= 5e-6
    err = np.abs(out - ref)
    assert (err <= TOL_DISP).mean() >= 0.999
    assert np.all(err <= TOL_DISP + np.abs(ref - d64[0]))
    # a one-hot-like cost (one clearly best bin per low-res voxel column) regresses to ~ 3j+1
    hot = torch.full((1, 1, dl, 4, 4), 50.0, device="cuda")
    hot[0, 0, 20] = -50.0
    d = F_.disp_head(hot, md)
    assert (d - 61.0).abs().max().item() < 1e-3


def _reference_head(md):
    """The unmodified reference's Disp (oracle/_ref) when installed, else the oracle port of the same lines."""
    from oracle import refimport as R

    if R.available():
        return R.import_reference().rag_model.Disp(md), "reference"
    return (lambda c: O.disp_head_ref(c, md)), "port"


BASELINE_SIZES = [
    # (name, B, Dl, Hl, Wl, maxdisp)          one pair per batch element is checked against fp64, all against the reference
    ("config 2/4: 480x960", 2, 64, 160, 320, 192),
    ("config 3: B=4 288x576", 4, 64, 96, 192, 192),
    ("config 5: 384x1248 md192", 2, 64, 128, 416, 192),
    ("config 5: 384x1248 md288", 2, 96, 128, 416, 288),
]


@pytest.mark.parametrize("size", BASELINE_SIZES, ids=lambda s: s[0])
def test_forward_and_backward_parity_at_baseline_sizes(F_, size):
    """VERDICT r1 #2: head forward AND backward against the torch-CUDA reference and the fp64 evaluation at the BASELINE
    configurations themselves (fp64 evaluated on the GPU: oracle.disp_head_f64_torch, checked against the numpy evaluator in
    test_oracle_golden).  Forward: own error <= 3e-5*(maxdisp/192) px; per pixel |ours - ref| <= 1e-4 + |ref - fp64| with the
    reference's own deviation capped; >= 99.9 % of pixels within 1e-4*(maxdisp/192).  Backward: 1e-5 max-norm vs fp64."""
    name, b, dl, hl, wl, md = size
    g = gen(len(name) + hl)
    cost = randn((b, 1, dl, hl, wl), g).cuda()
    gd = sparse_grad((b, 3 * hl, 3 * wl), g).cuda()
    head, kind = _reference_head(md)
    cr = cost.clone().requires_grad_(True)
    ref = head(cr)
    ref.backward(gd)
    gref = cr.grad
    co = cost.clone().requires_grad_(True)
    out = F_.disp_head(co, md)
    out.backward(gd)
    scale = md / 192
    worst = {"own": 0.0, "ref_dev": 0.0, "excess": 0.0, "grad": 0.0, "grad_ref": 0.0}
    for i in range(b):                                   # fp64 pair by pair (0.7-1.1 GB of temporaries each)
        d64, g64 = O.disp_head_f64_torch(cost[i:i + 1, 0], md, gd[i:i + 1])
        own = (out[i].detach().double() - d64[0]).abs()
        dev = (ref[i].detach().double() - d64[0]).abs()
        err = (out[i].detach() - ref[i].detach()).abs().double()
        worst["own"] = max(worst["own"], own.max().item())
        worst["ref_dev"] = max(worst["ref_dev"], dev.max().item())
        worst["excess"] = max(worst["excess"], (err - dev).max().item())
        worst["grad"] = max(worst["grad"], ((co.grad[i, 0].double() - g64[0]).abs().max() / g64.abs().max()).item())
        worst["grad_ref"] = max(worst["grad_ref"], ((gref[i, 0].double() - g64[0]).abs().max() / g64.abs().max()).item())
        del d64, g64
    frac = ((out.detach() - ref.detach()).abs() <= TOL_DISP * scale).double().mean().item()
    print(f"\n{name} [{kind}]: own {worst['own']:.2e} px, reference vs fp64 {worst['ref_dev']:.2e}, frac within {TOL_DISP * scale:.1e}: {frac:.6f}, "
          f"grad vs fp64 {worst['grad']:.2e} (reference's own: {worst['grad_ref']:.2e})")
    assert worst["own"] <= 3e-5 * scale
    assert worst["ref_dev"] <= 2e-4 * scale, "the reference's own fp32 deviation exceeds its recorded cap"
    assert worst["excess"] <= TOL_DISP
    assert frac >= 0.999
    assert worst["grad"] <= TOL_GRAD
    assert maxnorm_rel(co.grad.cpu().numpy(), gref.cpu().numpy()) <= 2 * TOL_GRAD


def test_module_hygiene(F_):
    import copy
    import pickle

    from rag_b200.modules import Disp

    m = Disp(192)
    assert len(m.state_dict()) == 0
    assert hasattr(m, "softmax") and hasattr(m, "disparity") and m.maxdisp == 192
    m2 = pickle.loads(pickle.dumps(copy.deepcopy(m)))
    x = randn((1, 1, 64, 4, 6), gen(2)).cuda().requires_grad_(True)
    m2(x).sum().backward()
    assert x.grad is not None and torch.isfinite(x.grad).all()
    with torch.no_grad():
        assert m(x).shape == (1, 12, 18)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 1, 64, 4, 6))  # CPU tensor: no fallback


def test_backward_red_variant_is_bitwise_deterministic(F_):
    """Variant 4 adds the two row parts of every element into a zeroed buffer with red.global.add: two
    commutative contributions, so the result must not depend on arrival order -- bitwise equal run to run and
    equal to the scratch + combine variant (which adds the same two numbers) up to the sign of a zero."""
    g = gen(404)
    b, dl, hl, wl, md = 2, 64, 40, 96, 192
    cost = randn((b, 1, dl, hl, wl), g).cuda()
    gd = sparse_grad((b, 3 * hl, 3 * wl), g).cuda()
    disp, stats = F_.disp_head_forward(cost, md, want_stats=True)
    ref = F_.disp_head_backward(cost, gd, disp, stats, md, variant=2)
    outs = [F_.disp_head_backward(cost, gd, disp, stats, md, variant=1) for _ in range(5)]
    for o in outs[1:]:
        assert torch.equal(outs[0], o)
    assert torch.equal(outs[0], ref)     # torch.equal treats -0.0 == +0.0
