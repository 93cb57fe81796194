"""Out-of-bounds write check without compute-sanitizer (closed on this pool): every output buffer is a
window inside a larger canary-filled allocation; after the call the canaries on both sides must be
intact.  Calls go straight through the C ABI with raw pointers."""
import pytest
import torch

from tests._util import gen, randn

pytestmark = pytest.mark.gpu
GUARD = 4096  # floats on each side
CANARY = -12345.678


def window(n, dtype=torch.float32):
    buf = torch.full((n + 2 * GUARD,), CANARY, dtype=dtype, device="cuda")
    return buf, buf[GUARD:GUARD + n]


def intact(buf, n):
    return bool((buf[:GUARD] == CANARY).all()) and bool((buf[GUARD + n:] == CANARY).all())


@pytest.fixture(scope="module")
def L():
    assert torch.cuda.is_available()
    from rag_b200 import _cabi

    return _cabi.lib()


def st():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("shape", [(2, 12, 9, 36, 96), (1, 3, 5, 37, 30), (1, 4, 7, 70, 192), (1, 2, 3, 10, 48), (1, 12, 33, 64, 100), (1, 3, 9, 64, 192),
                                   (2, 3, 5, 8, 96), (1, 5, 17, 132, 120), (3, 2, 2, 4, 192)], ids=str)
def test_cost_volume_guards(L, shape):
    b, c, hf, wf, md = shape
    df = int(md / 3)
    g = gen(1)
    x, y = randn((b, c, hf, wf), g).cuda(), randn((b, c, hf, wf), g).cuda()
    n = b * 2 * c * df * hf * wf
    variants = [-1, 0] + ([1, 3, 5] if wf % 4 == 0 else [])
    for v in variants:
        buf, out = window(n)
        wbuf, ws = window(4)                       # the 16-byte work-counter workspace, itself behind guard bands
        assert L.rag_cost_volume_fwd_v(x.data_ptr(), y.data_ptr(), out.data_ptr(), b, c, df, hf, wf, ws.data_ptr(), v, st()) == 0
        torch.cuda.synchronize()
        assert intact(wbuf, 4), f"cv_fwd variant {v} wrote outside its workspace"
        torch.cuda.synchronize()
        assert intact(buf, n), f"cv_fwd variant {v} wrote out of bounds"
        assert not (out == CANARY).any(), f"cv_fwd variant {v} left output elements unwritten"
    gc = randn((b, 2 * c, df, hf, wf), g).cuda()
    m = b * c * hf * wf
    for v in (0, 1) + ((2, 3) if wf % 4 == 0 else ()):
        bx, gx = window(m)
        by, gy = window(m)
        assert L.rag_cost_volume_bwd_v(gc.data_ptr(), gx.data_ptr(), gy.data_ptr(), b, c, df, hf, wf, v, st()) == 0
        torch.cuda.synchronize()
        assert intact(bx, m) and intact(by, m), f"cv_bwd variant {v}"
        assert not (gx == CANARY).any() and not (gy == CANARY).any()


@pytest.mark.parametrize("shape", [(1, 16, 5, 36, 48), (2, 8, 3, 7, 24), (1, 20, 9, 4, 60), (1, 12, 3, 4, 48), (1, 64, 7, 33, 192), (2, 64, 6, 64, 192),
                                   (1, 64, 4, 32, 192), (2, 17, 3, 12, 51), (1, 32, 12, 8, 96)], ids=str)
def test_head_guards(L, shape):
    b, dl, hl, wl, md = shape
    g = gen(2)
    cl = randn((b, 1, dl, hl, wl), g).cuda()
    npx = b * 9 * hl * wl
    x3 = md == 3 * dl
    fv = [0] + ([1] if x3 else []) + ([2, 4] if x3 and wl % 4 == 0 else [])
    for v in fv:
        bd, disp = window(npx)
        bs, stats = window(2 * npx)
        assert L.rag_disp_head_fwd_v(cl.data_ptr(), disp.data_ptr(), stats.data_ptr(), b, dl, hl, wl, md, v, st()) == 0
        torch.cuda.synchronize()
        assert intact(bd, npx) and intact(bs, 2 * npx), f"head_fwd variant {v}"
        assert not (disp == CANARY).any() and not (stats == CANARY).any(), f"head_fwd variant {v} left outputs unwritten"
    gd = randn((b, 3 * hl, 3 * wl), g).cuda()
    nv = b * dl * hl * wl
    for v in [0] + ([1, 2, 3] if x3 else []):
        bg, gcl = window(nv)
        bsc, scr = window(nv)
        assert L.rag_disp_head_bwd_v(cl.data_ptr(), gd.data_ptr(), disp.data_ptr(), stats.data_ptr(), gcl.data_ptr(), scr.data_ptr(), b, dl, hl, wl, md, v, st()) == 0
        torch.cuda.synchronize()
        assert intact(bg, nv) and intact(bsc, nv), f"head_bwd variant {v}"
        if v == 2:
            assert not (scr == CANARY).any(), f"head_bwd variant {v} left scratch elements unwritten"
        else:
            assert (scr == CANARY).all(), f"head_bwd variant {v} must not touch the scratch buffer"
        assert not (gcl == CANARY).any(), f"head_bwd variant {v} left outputs unwritten"
    bu, up = window(b * md * 9 * hl * wl)
    assert L.rag_upsample_trilinear(cl.data_ptr(), up.data_ptr(), b, dl, hl, wl, md, 1, st()) == 0
    torch.cuda.synchronize()
    assert intact(bu, b * md * 9 * hl * wl)


def test_fused_stem_guards(L):
    g = gen(4)
    for (b, c, hf, wf, df, o) in [(1, 12, 4, 40, 16, 12), (2, 12, 3, 38, 10, 5), (1, 12, 3, 16, 2, 12), (1, 5, 3, 20, 8, 4)]:
        x, y = randn((b, c, hf, wf), g).cuda(), randn((b, c, hf, wf), g).cuda()
        w = randn((o, 2 * c, 3, 3, 3), g).cuda()
        n = b * o * df * hf * wf
        for v in (0,) + ((1,) if (c == 12 and df >= 3) else ()) + ((2,) if (c == 12 and df >= 3 and wf % 4 == 0) else ()):
            buf, out = window(n)
            nws = int(L.rag_cv_stem_workspace_bytes(c, o)) // 4
            wbuf, ws = window(max(nws, 4))
            assert L.rag_cv_stem_fwd_v(x.data_ptr(), y.data_ptr(), w.data_ptr(), None, None, 0, out.data_ptr(), b, c, o, df, hf, wf,
                                       ws.data_ptr() if nws else None, v, st()) == 0
            torch.cuda.synchronize()
            assert intact(wbuf, max(nws, 4)), f"cv_stem variant {v} wrote outside its workspace"
            torch.cuda.synchronize()
            assert intact(buf, n), f"cv_stem variant {v} wrote out of bounds"
            assert not (out == CANARY).any(), f"cv_stem variant {v} left outputs unwritten"


def test_misc_guards(L):
    g = gen(3)
    b, h, w = 3, 37, 53
    gt = (torch.rand(b, h, w, generator=g) * 250 - 20).cuda()
    est = (gt + torch.randn(b, h, w, generator=g).cuda())
    nscr = L.rag_loss_metrics_scratch(h, w)
    bs, sums = window(b * 8, torch.float64)
    bc, scr = window(b * nscr, torch.float64)
    assert L.rag_loss_metrics_sums(est.data_ptr(), gt.data_ptr(), sums.data_ptr(), scr.data_ptr(), b, h, w, 192.0, st()) == 0
    bg, gest = window(b * h * w)
    one = torch.ones(1, device="cuda")
    assert L.rag_smooth_l1_bwd(est.data_ptr(), gt.data_ptr(), sums.data_ptr(), one.data_ptr(), gest.data_ptr(), b, h, w, 192.0, st()) == 0
    img = torch.randint(0, 256, (2, 10, 14, 3), dtype=torch.uint8, device="cuda")
    bo, out = window(2 * 3 * 12 * 18)
    assert L.rag_normalize_pad(img.data_ptr(), out.data_ptr(), 2, 10, 14, 2, 4, st()) == 0
    p = torch.softmax(randn((2, 24, 5, 7), g), 1).cuda().contiguous()
    br, reg = window(2 * 5 * 7)
    assert L.rag_disparity_regression_fwd(p.data_ptr(), reg.data_ptr(), 2, 24, 5, 7, st()) == 0
    bp, gp = window(2 * 24 * 5 * 7)
    assert L.rag_disparity_regression_bwd(reg.data_ptr(), gp.data_ptr(), 2, 24, 5, 7, st()) == 0
    torch.cuda.synchronize()
    assert intact(bs, b * 8) and intact(bc, b * nscr) and intact(bg, b * h * w) and intact(bo, 2 * 3 * 12 * 18)
    assert intact(br, 70) and intact(bp, 2 * 24 * 35)


@pytest.mark.parametrize("shape", [(1, 12, 17, 9, 68), (2, 3, 5, 3, 4), (1, 12, 32, 8, 64)], ids=str)
def test_last_conv_guards(L, shape):
    b, c, d, h, w = shape
    g = gen(4)
    x = randn((b, c, d, h, w), g).cuda()
    wt = randn((1, c, 3, 3, 3), g).cuda()
    n = b * d * h * w
    buf, out = window(n)
    assert L.rag_conv3d_c1_fwd(x.data_ptr(), wt.data_ptr(), out.data_ptr(), b, c, d, h, w, st()) == 0
    torch.cuda.synchronize()
    assert intact(buf, n), "conv3d_c1 wrote out of bounds"
    assert not (out == CANARY).any(), "conv3d_c1 left output elements unwritten"
