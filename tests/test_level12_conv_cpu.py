"""CPU-side checks of the level-12 interior ConvBR_3d path (``ConvBR_3d(16, 16, 3, 1, 1)``: the rag_conv3d_cc16_* entries of
csrc/conv3d_cc.cu; ``install(..., matching_convs=True, level12_convs=True)``): argument errors and the workspace query of the
C entries without a GPU, the flag's rules and the routing predicate's exclusions."""
import pytest
import torch
import torch.nn as nn

from tests._stand_in import _stand_in


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi

    L = _cabi.lib()
    fake = 256
    fwd, bwd = L.rag_conv3d_cc16_fwd, L.rag_conv3d_cc16_bwd
    assert fwd(None, fake, None, None, 1, fake, 1, 16, 16, 4, 4, 8, None) == -1
    assert b"null" in L.rag_last_error()
    assert fwd(fake, None, None, None, 1, fake, 1, 16, 16, 4, 4, 8, None) == -1
    assert fwd(fake, fake, None, None, 1, None, 1, 16, 16, 4, 4, 8, None) == -1
    assert fwd(fake, fake, fake, None, 1, fake, 1, 16, 16, 4, 4, 8, None) == -1          # scale without shift
    assert bwd(None, fake, fake, fake, fake, fake, 1, 16, 16, 4, 4, 8, None) == -1       # gz
    assert bwd(fake, fake, None, fake, None, None, 1, 16, 16, 4, 4, 8, None) == -1       # gin without w
    assert bwd(fake, None, fake, None, fake, fake, 1, 16, 16, 4, 4, 8, None) == -1       # gw without in
    assert bwd(fake, fake, fake, None, fake, None, 1, 16, 16, 4, 4, 8, None) == -1       # gw without workspace
    # shape errors come before any pointer is touched: every other pair, W % 4, a non-positive dimension
    for c, o in ((4, 4), (8, 8), (12, 12), (16, 8), (8, 16), (15, 15), (32, 32)):
        assert fwd(fake, fake, None, None, 0, fake, 1, c, o, 4, 4, 8, None) == -2
        assert b"not compiled" in L.rag_last_error()
        assert bwd(fake, fake, fake, fake, fake, fake, 1, c, o, 4, 4, 8, None) == -2
        assert b"not compiled" in L.rag_last_error()
    assert fwd(fake, fake, None, None, 0, fake, 1, 16, 16, 4, 4, 6, None) == -2
    assert bwd(fake, fake, fake, fake, fake, fake, 1, 16, 16, 4, 4, 10, None) == -2
    for dims in ((0, 4, 4, 8), (1, 0, 4, 8), (1, 4, 0, 8), (1, 4, 4, 0), (-1, 4, 4, 8)):
        b, d, h, w = dims
        assert fwd(fake, fake, None, None, 0, fake, b, 16, 16, d, h, w, None) == -2
        assert bwd(fake, fake, fake, fake, fake, fake, b, 16, 16, d, h, w, None) == -2
    # the limits of the existing entries: 3*H*W < 2^31, B*ceil(D/8) <= 65535
    assert fwd(fake, fake, None, None, 0, fake, 1, 16, 16, 3, 2 ** 16, 2 ** 14, None) == -2
    assert fwd(fake, fake, None, None, 0, fake, 65536, 16, 16, 3, 1, 8, None) == -2
    # misaligned pointers (the shape is fine): in / out / gz / gin want 16 bytes, w / workspace 4
    assert fwd(fake + 4, fake, None, None, 0, fake, 1, 16, 16, 4, 4, 8, None) == -3
    assert fwd(fake, fake, None, None, 0, fake + 8, 1, 16, 16, 4, 4, 8, None) == -3
    assert fwd(fake, fake + 2, None, None, 0, fake, 1, 16, 16, 4, 4, 8, None) == -3
    assert bwd(fake + 4, fake, fake, fake, None, None, 1, 16, 16, 4, 4, 8, None) == -3
    assert bwd(fake, fake, fake, fake + 4, None, None, 1, 16, 16, 4, 4, 8, None) == -3
    assert bwd(fake, fake + 4, fake, None, fake, fake, 1, 16, 16, 4, 4, 8, None) == -3
    assert bwd(fake, fake, fake, None, fake, fake + 2, 1, 16, 16, 4, 4, 8, None) == -3


def test_existing_entries_still_refuse_16():
    from rag_b200 import _cabi

    L = _cabi.lib()
    fake = 256
    assert L.rag_conv3d_cc_fwd(fake, fake, None, None, 0, fake, 1, 16, 16, 4, 4, 8, None) == -2
    assert L.rag_conv3d_cc_bwd(fake, fake, fake, fake, fake, fake, 1, 16, 16, 4, 4, 8, None) == -2
    assert L.rag_conv3d_cc_bwd_workspace_bytes(4, 16, 16, 16, 24, 48) == 0
    assert L.rag_conv3d_cc_tf32_fwd(fake, fake, None, None, 0, fake, 1, 16, 16, 4, 4, 8, None) == -2
    assert L.rag_conv3d_cc_tf32_bwd_weight_workspace_bytes(4, 16, 16, 16, 24, 48) == 0


def test_workspace_query():
    """Non-zero exactly for (16,16) with positive dimensions -- [G][O][C][27] fp32 partials -- and no device needed."""
    from rag_b200 import _cabi

    L = _cabi.lib()
    q = L.rag_conv3d_cc16_bwd_workspace_bytes
    for shape in ((4, 16, 24, 48), (8, 16, 40, 80), (1, 3, 1, 8)):
        b, d, h, w = shape
        n = q(b, 16, 16, d, h, w)
        assert n > 0 and n % (16 * 16 * 27 * 4) == 0
    for c in (1, 4, 8, 12, 15, 16, 24, 32):
        for o in (4, 8, 12, 16, 32):
            assert (q(4, c, o, 16, 24, 48) > 0) == ((c, o) == (16, 16)), (c, o)
    for dims in ((0, 4, 4, 8), (1, 0, 4, 8), (1, 4, 0, 8), (1, 4, 4, 0)):
        assert q(dims[0], 16, 16, *dims[1:]) == 0


def test_cpu_tensors_raise():
    from rag_b200.matching_conv import conv3d_cc_forward

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conv3d_cc_forward(torch.zeros(1, 16, 3, 4, 8), torch.zeros(16, 16, 3, 3, 3))


def test_install_flag_rules(monkeypatch):
    from rag_b200 import fused_stem, matching_conv
    from rag_b200 import network as N

    rag_model, ops3d, _ = _stand_in()
    N.uninstall()
    try:
        with pytest.raises(ValueError, match="matching_convs=True"):
            N.install(rag_model, None, ops3d, level12_convs=True)
        assert not matching_conv._LEVEL12
        N.install(rag_model, None, ops3d, matching_convs=True, level12_convs=True)
        assert matching_conv._LEVEL12
        N.install(rag_model, None, ops3d, matching_convs=True)          # a later install() without it turns it off
        assert not matching_conv._LEVEL12
        N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32=True, matching_tf32_wgrad=True, level12_convs=True)
        assert matching_conv._LEVEL12
        N.uninstall()
        assert not matching_conv._LEVEL12
    finally:
        N.uninstall()
    # with the flag off, a 16 -> 16 layer goes to stem_forward (the fuse_stem binding), as before
    seen = []
    monkeypatch.setattr(matching_conv, "stem_forward", lambda self, x: seen.append(self) or "stem")
    monkeypatch.setattr(matching_conv, "level12_qualifies", lambda layer, x: True)    # as if on a GPU
    layer = _ConvBR(16, 16)
    assert matching_conv.matching_forward(layer, torch.zeros(1, 16, 4, 4, 8)) == "stem" and seen == [layer]
    # the TF32 switches never select 16 -> 16: there is no TF32 kernel for it
    monkeypatch.setattr(matching_conv, "_TF32", True)
    monkeypatch.setattr(matching_conv, "_TF32_WGRAD", True)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", True)
    assert not matching_conv.use_tf32(16) and not matching_conv.use_tf32_wgrad(16)
    assert matching_conv.use_tf32(12) and matching_conv.use_tf32(8) and not matching_conv.use_tf32(4)


class _ConvBR(nn.Module):
    """The reference's ConvBR_3d field layout (operations_3d.py:31-47)."""

    def __init__(self, c, o, k=3, s=1, p=1, bn=True, relu=True, bias=False, affine=True):
        super().__init__()
        self.conv = nn.Conv3d(c, o, k, stride=s, padding=p, bias=bias)
        self.use_bn = bn
        self.bn = nn.BatchNorm3d(o, affine=affine) if bn else None
        self.relu = relu


def test_level12_predicate_rejects_each_exclusion():
    """Each exclusion is rejected by the clause that names it; (16,16) with only that field changed qualifies, device aside
    (the input clauses are checked with the weight-on-CUDA clause replaced by the positive control's)."""
    from rag_b200 import matching_conv as M

    assert M._layer_is(_ConvBR(16, 16), (M.LEVEL12_PAIR,))
    assert not M.layer_qualifies(_ConvBR(16, 16))            # PAIRS is unchanged
    assert (16, 16) not in M.PAIRS
    no_stats = _ConvBR(16, 16)
    no_stats.bn = nn.BatchNorm3d(16, track_running_stats=False)
    excluded = {
        "stride 2": _ConvBR(16, 16, 3, 2, 1),
        "bias": _ConvBR(16, 16, bias=True),
        "no BatchNorm": _ConvBR(16, 16, bn=False),
        "affine-free BatchNorm": _ConvBR(16, 16, affine=False),
        "no running stats": no_stats,
        "no ReLU": _ConvBR(16, 16, relu=False),
        "fp64": _ConvBR(16, 16).double(),
        "(16,8)": _ConvBR(16, 8),
        "(12,12)": _ConvBR(12, 12),
        "1x1 kernel": _ConvBR(16, 16, 1, 1, 0),
    }
    for name, layer in excluded.items():
        assert not M._layer_is(layer, (M.LEVEL12_PAIR,)), name
        assert not M.level12_qualifies(layer, torch.zeros(1, layer.conv.in_channels, 4, 4, 8)), name
    # CPU tensors (and a CPU weight) stay off the kernels
    assert not M.level12_qualifies(_ConvBR(16, 16).eval(), torch.zeros(1, 16, 4, 4, 8))
