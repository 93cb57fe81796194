"""tests/_grids.py restates the work-loop grids of four kernels; its constants must be the ones the CUDA sources launch with,
or the work-loop tests would check shapes that no longer make the loops wrap."""
import os
import re

from tests import _grids

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rag_b200", "csrc")


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _constexpr(text, name):
    found = re.findall(r"\b" + name + r"\s*=\s*(\d+)\s*[,;]", text)
    assert len(found) == 1, f"{name}: {found}"
    return int(found[0])


def test_grid_constants_match_the_sources():
    cc = _src("conv3d_cc.cu")
    assert [_constexpr(cc, n) for n in ("kCcWgGroups", "kCcWgDT", "kCcWgHT", "kCcWT")] == \
        [_grids.CC_WG_GROUPS, _grids.CC_WG_DT, _grids.CC_WG_HT, _grids.CC_WT]
    lb = _src("last_conv_bwd.cu")
    assert [_constexpr(lb, n) for n in ("kLbGroups", "kWmDS")] == [_grids.LB_GROUPS, _grids.WM_DS]
    assert _constexpr(_src("disp_head_x3w.cuh"), "kBwJ") == _grids.BW_J
    head = _src("disp_head.cu")
    # one persistent grid per direction, both sized num_sms() * 3
    assert [int(k) for k in re.findall(r"num_sms\(\)\s*\*\s*(\d+)", head)] == [_grids.HEAD_CTAS_PER_SM] * 2
    assert _constexpr(head, "warps") == _grids.HEAD_FWD_WARPS


def test_grid_helpers_give_the_counts_of_the_shapes_they_are_used_at():
    assert _grids.cc_wgrad(3, 17, 37, 136) == (296, 513)
    assert _grids.cc_wgrad(4, 64, 96, 192) == (296, 4608)
    assert _grids.c1_bwd_weight(24, 33, 38, 132) == (1184, 2400)
    assert _grids.c1_bwd_weight(8, 64, 96, 192) == (1184, 2304)
    assert _grids.loops(296, 513) == "513 items on 296: 1-2 each"
