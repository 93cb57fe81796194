"""The grids of the kernels whose CTAs (or warps) loop over work items, restated from their host launch code, so that a test
can show that its shape makes the loop run more than once and end on an uneven last round.

Each function returns ``(grid, n_items)`` where ``grid`` counts the CTAs (or warps) that share the ``n_items`` items
round-robin.  tests/test_work_loops_cpu.py checks the constants below against the CUDA sources.  Nothing here touches CUDA
at import."""

CC_WG_GROUPS, CC_WG_DT, CC_WG_HT, CC_WT = 296, 8, 2, 64    # conv3d_cc.cu: kCcWgGroups, kCcWgDT, kCcWgHT, kCcWT
LB_GROUPS, WM_DS = 296, 32                                  # last_conv_bwd.cu: kLbGroups, kWmDS
BW_J = 16                                                   # disp_head_x3w.cuh: kBwJ
HEAD_CTAS_PER_SM = 3                                        # disp_head.cu: num_sms() * 3
HEAD_FWD_WARPS = 4                                          # disp_head.cu: the persistent forward's warps (block rows) per tile


def _cdiv(a, b):
    return -(-a // b)


def cc_wgrad(b, d, h, w):
    """conv3d_cc_wgrad_kernel's CTAs and tiles; mirrors cc_launch_wgrad (conv3d_cc.cu)."""
    n_tiles = b * _cdiv(d, CC_WG_DT) * _cdiv(h, CC_WG_HT) * _cdiv(w, CC_WT)
    return min(CC_WG_GROUPS, n_tiles), n_tiles


def c1_bwd_weight(b, d, h, w):
    """conv3d_c1_bwd_weight_march_kernel's warps per channel pair (kLbGroups CTAs of 4 warps) and items; mirrors
    conv3d_c1_bwd (last_conv_bwd.cu)."""
    return LB_GROUPS * 4, b * _cdiv(d, WM_DS) * _cdiv(h, 4) * _cdiv(w, 32)


def _sms(dev):
    import torch

    return torch.cuda.get_device_properties(dev).multi_processor_count


def head_fwd(b, hl, wl, dev):
    """The persistent head forward's CTAs and tiles (variant RAG_HEAD_FWD_SHARED); mirrors disp_head_fwd (disp_head.cu)."""
    n_tiles = b * _cdiv(wl, 32) * _cdiv(hl, HEAD_FWD_WARPS)
    return min(n_tiles, _sms(dev) * HEAD_CTAS_PER_SM), n_tiles


def head_bwd(b, dl, hl, wl, dev):
    """The persistent head backward's CTAs and CTA-tasks (variant RAG_HEAD_BWD_SHARED); mirrors disp_head_bwd
    (disp_head.cu)."""
    n_ct = _cdiv(wl, 31) * _cdiv((hl + 1) * _cdiv(dl, BW_J), 4) * b
    return min(n_ct, _sms(dev) * HEAD_CTAS_PER_SM), n_ct


def loops(grid, n_items):
    """Assert that some CTA (warp) of ``grid`` takes two items or more and that the last round is uneven; return the range of
    items per CTA (warp) as text."""
    assert n_items > grid and n_items % grid != 0, f"{n_items} items on {grid}: the work loop does not wrap unevenly"
    return f"{n_items} items on {grid}: {n_items // grid}-{_cdiv(n_items, grid)} each"
