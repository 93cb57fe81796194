"""The grids of the kernels whose CTAs (or warps) loop over work items, restated from their host launch code, so that a test
can show that its shape makes the loop run more than once and end on an uneven last round; and the launch geometry of the
fused stem's backward (cv_stem_train.cu), so that a test at the edge of the training limits can show which edge it reaches.

Each work-loop function returns ``(grid, n_items)`` where ``grid`` counts the CTAs (or warps) that share the ``n_items`` items
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


STEM_WC, STEM_TH = 128, 4                                   # cv_stem_train.cu: kStWC, kStTH
STEM_MAPS_US = (8, 4, 2, 1)                                 # cv_stem_train.cu: the maps kernel's rows per step, largest first
SMEM_DEFAULT = 48 * 1024                                    # dynamic shared memory a launch gets without the opt-in


def stem_maps(b, o, df, hf, wf):
    """stem_bwd_maps_kernel<U>: (U, grid, threads, dynamic shared-memory bytes); mirrors cv_stem_bwd (cv_stem_train.cu).  U is
    the largest of 8, 4, 2, 1 that divides Df."""
    u = next(u for u in STEM_MAPS_US if df % u == 0)
    return u, (hf, o, b), _cdiv(wf + 4, 32) * 32, (2 * u + 5) * wf * 4


def stem_bwd_inputs(b, o, hf, wf):
    """stem_bwd_inputs_kernel: (grid, dynamic shared-memory bytes); grid z = 2B (batch item, side)."""
    r = 9 * o
    return (_cdiv(wf, STEM_WC), _cdiv(hf, STEM_TH), 2 * b), (max(r * STEM_WC, STEM_TH * 12 * 128) + 3 * r * 16) * 4


def stem_bwd_weight(b, o, hf):
    """stem_bwd_weight_kernel: (grid, threads): one thread per 4x4 register tile of the (9*O rounded up to 4) x 36 product."""
    rp = (9 * o + 3) // 4 * 4
    return (hf, 2 * b), _cdiv(rp // 4 * 9, 32) * 32


CC_HT, CC_DT = 8, 8                                         # conv3d_cc.cu: kCcHT, kCcDT (the forward's tile; kCcWT = CC_WT)
PW_THREADS = 128                                            # conv3d_pw.cu: kPwThreads


def cc_fwd(b, d, h, w):
    """conv3d_cc_fwd_kernel's grid (also the data gradient's); mirrors cc_launch_fwd (conv3d_cc.cu)."""
    return _cdiv(w, CC_WT), _cdiv(h, CC_HT), b * _cdiv(d, CC_DT)


def pw_fwd(b, d, h, w):
    """conv3d_pw_fwd_kernel's grid: float4 voxel groups of one batch item in x, the batch item in y (pw_launch_fwd)."""
    return _cdiv(d * h * w // 4, PW_THREADS), b


def bn3d_rows(b, o, h):
    """The grid of bn3d.cu's two row kernels (moments, backward sums): one CTA per (h, o, b) row."""
    return h, o, b


def loops(grid, n_items):
    """Assert that some CTA (warp) of ``grid`` takes two items or more and that the last round is uneven; return the range of
    items per CTA (warp) as text."""
    assert n_items > grid and n_items % grid != 0, f"{n_items} items on {grid}: the work loop does not wrap unevenly"
    return f"{n_items} items on {grid}: {n_items // grid}-{_cdiv(n_items, grid)} each"
