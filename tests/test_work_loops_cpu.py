"""tests/_grids.py restates the work-loop grids of four kernels and the launch geometry of the training kernels; its constants
must be the ones the CUDA sources launch with, or the work-loop tests would check shapes that no longer make the loops wrap,
and the training-limit tests shapes that no longer reach the edge they are written for."""
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


def test_stem_backward_geometry_matches_the_source():
    """The launch lines of cv_stem_bwd that tests/test_training_limits_gpu.py builds its cases on, as the source states them."""
    st = _src("cv_stem_train.cu")
    assert [_constexpr(st, n) for n in ("kStWC", "kStTH")] == [_grids.STEM_WC, _grids.STEM_TH]
    us = re.findall(r"const int U = Df % (\d) == 0 \? (\d) : Df % (\d) == 0 \? (\d) : Df % (\d) == 0 \? (\d) : (\d);", st)
    assert len(us) == 1 and us[0] == ("8", "8", "4", "4", "2", "2", "1"), us
    assert tuple(int(u) for u in us[0][1::2] + us[0][-1:]) == _grids.STEM_MAPS_US
    for text in ("const int nt = ((Wf + 4 + 31) / 32) * 32;",
                 "const size_t smem = ((size_t)2 * U + 5) * Wf * sizeof(float);",
                 "kern<<<dim3(Hf, O, B), nt, smem, st>>>",
                 "std::max((size_t)R * kStWC, (size_t)kStTH * 12 * 128) + (size_t)3 * R * 16) * sizeof(float)",
                 "stem_bwd_inputs_kernel<<<dim3((Wf + kStWC - 1) / kStWC, (Hf + kStTH - 1) / kStTH, 2 * B), 256, smem, st>>>",
                 "const int nt = (((Rp >> 2) * 9 + 31) / 32) * 32;",
                 "stem_bwd_weight_kernel<<<dim3(Hf, 2 * B), nt, smem, st>>>"):
        assert st.count(text) == 1, text
    # every launch of the maps kernel opts in to the shared memory it asks for
    assert st.count("cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)") == 1


def test_interior_and_bn3d_grids_match_the_sources():
    cc = _src("conv3d_cc.cu")
    assert [_constexpr(cc, n) for n in ("kCcHT", "kCcDT")] == [_grids.CC_HT, _grids.CC_DT]
    assert cc.count("k<<<dim3((W + kCcWT - 1) / kCcWT, (H + kCcHT - 1) / kCcHT, B * n_dt), kCcThreads, smem, st>>>") == 1
    assert cc.count("const int n_dt = (D + kCcDT - 1) / kCcDT;") == 1
    pw = _src("conv3d_pw.cu")
    assert _constexpr(pw, "kPwThreads") == _grids.PW_THREADS
    assert pw.count("conv3d_pw_fwd_kernel<OT><<<dim3((unsigned)((S4 + kPwThreads - 1) / kPwThreads), B), kPwThreads, smem, st>>>") == 1
    bn = _src("bn3d.cu")
    assert bn.count("<<<dim3(H, O, B), 256, 0, st>>>") == 2
    assert _grids.cc_fwd(32767, 3, 1, 8) == (1, 1, 32767) and _grids.cc_fwd(1, 3, 65535, 1016) == (16, 8192, 1)
    assert _grids.pw_fwd(32767, 3, 1, 8) == (1, 32767) and _grids.bn3d_rows(32767, 32, 65535) == (65535, 32, 32767)


def test_stem_backward_geometry_at_the_training_limits():
    """The edges the cases of tests/test_training_limits_gpu.py are written for."""
    # (Df, Wf) -> (U, maps kernel's dynamic shared memory); the last width under 48 KB and the first over it, per U
    assert _grids.stem_maps(1, 12, 64, 1, 584)[::3] == (8, 49056) and _grids.stem_maps(1, 12, 64, 1, 588)[::3] == (8, 49392)
    assert _grids.stem_maps(1, 12, 36, 1, 944)[::3] == (4, 49088) and _grids.stem_maps(1, 12, 36, 1, 948)[::3] == (4, 49296)
    assert _grids.stem_maps(1, 12, 64, 1, 1016)[3] == 85344 and _grids.stem_maps(1, 32, 64, 5, 1016)[2] == 1024
    assert [_grids.stem_maps(1, 1, df, 1, 132)[0] for df in (18, 33, 3)] == [2, 1, 1]
    assert 49056 <= _grids.SMEM_DEFAULT < 49296
    # O = 32: 672 threads in the weight kernel, about 198 KB of shared memory in the inputs kernel
    assert _grids.stem_bwd_weight(1, 32, 5) == ((5, 2), 672)
    assert _grids.stem_bwd_inputs(1, 32, 5, 1016) == ((8, 2, 2), 202752)
    # B = 32767: the inputs kernel's grid z and the weight kernel's grid y are 2B = 65534, one under the hardware's 65535
    assert _grids.stem_bwd_inputs(32767, 1, 1, 8)[0][2] == 65534 and _grids.stem_bwd_weight(32767, 1, 1)[0][1] == 65534
    assert _grids.stem_maps(1, 1, 3, 65535, 8)[1] == (65535, 1, 1)


def test_grid_helpers_give_the_counts_of_the_shapes_they_are_used_at():
    assert _grids.cc_wgrad(3, 17, 37, 136) == (296, 513)
    assert _grids.cc_wgrad(4, 64, 96, 192) == (296, 4608)
    assert _grids.c1_bwd_weight(24, 33, 38, 132) == (1184, 2400)
    assert _grids.c1_bwd_weight(8, 64, 96, 192) == (1184, 2304)
    assert _grids.loops(296, 513) == "513 items on 296: 1-2 each"
