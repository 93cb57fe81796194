"""CPU-side checks of the interior ConvBR_3d path (csrc/conv3d_cc.cu, rag_b200/matching_conv.py): argument errors of the C
ABI without a GPU, no CPU fallback, the install()/uninstall() binding and the routing decision's exclusions."""
import pytest
import torch
import torch.nn as nn

from tests._mirror_net import reference_modules


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi
    from rag_b200.matching_conv import PAIRS

    L = _cabi.lib()
    assert L.rag_conv3d_cc_fwd(None, None, None, None, 1, None, 1, 12, 12, 4, 4, 8, None) == -1
    assert b"null" in L.rag_last_error()
    assert L.rag_bn3d_bwd_gz(None, None, None, None, 1, 12, 4, 4, 8, None) == -1
    assert L.rag_conv3d_cc_bwd(None, None, None, None, None, None, 1, 12, 12, 4, 4, 8, None) == -1
    # an unsupported (C, O) is a shape error, reported before any pointer is touched
    fake = 256
    assert L.rag_conv3d_cc_fwd(fake, fake, None, None, 0, fake, 1, 5, 5, 4, 4, 8, None) == -2
    assert b"not compiled" in L.rag_last_error()
    assert L.rag_conv3d_cc_bwd(fake, fake, fake, fake, None, None, 1, 12, 8, 4, 4, 8, None) == -2
    assert L.rag_conv3d_cc_fwd(fake, fake, None, None, 0, fake, 1, 12, 12, 4, 4, 6, None) == -2      # W % 4 != 0
    # the workspace query names the compiled set: non-zero exactly for PAIRS
    for c in (1, 2, 4, 5, 8, 12, 16, 24, 32):
        for o in (1, 4, 8, 12, 16):
            n = L.rag_conv3d_cc_bwd_workspace_bytes(2, c, o, 4, 4, 8)
            assert (n > 0) == ((c, o) in PAIRS), (c, o, n)


def test_cpu_tensors_raise():
    from rag_b200.matching_conv import conv3d_cc_forward

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conv3d_cc_forward(torch.zeros(1, 12, 3, 4, 8), torch.zeros(12, 12, 3, 3, 3))


class _ConvBR(nn.Module):
    """The reference's ConvBR_3d field layout (operations_3d.py:31-47)."""

    def __init__(self, c, o, k=3, s=1, p=1, bn=True, relu=True, bias=False, affine=True):
        super().__init__()
        self.conv = nn.Conv3d(c, o, k, stride=s, padding=p, bias=bias)
        self.use_bn = bn
        self.bn = nn.BatchNorm3d(o, affine=affine) if bn else None
        self.relu = relu


def test_qualifies_rejects_excluded_geometries():
    """Each exclusion is rejected by the clause that names it: the layer predicate is device-independent, and the same
    construction with only that one field changed qualifies (positive control)."""
    from rag_b200 import matching_conv as M

    assert M.layer_qualifies(_ConvBR(12, 12))
    for c in (4, 8, 12):
        assert M.layer_qualifies(_ConvBR(c, c))
    excluded = {
        "1x1 kernel": _ConvBR(12, 12, 1, 1, 0),
        "stride 2": _ConvBR(12, 12, 3, 2, 1),
        "bias": _ConvBR(12, 12, bias=True),
        "(5,5)": _ConvBR(5, 5),
        "(16,16)": _ConvBR(16, 16),
        "(12,8)": _ConvBR(12, 8),
        "no BatchNorm": _ConvBR(12, 12, bn=False),
        "affine-free BatchNorm": _ConvBR(12, 12, affine=False),
        "no ReLU": _ConvBR(12, 12, relu=False),
        "fp64": _ConvBR(12, 12).double(),
    }
    for name, layer in excluded.items():
        assert not M.layer_qualifies(layer), name
        assert not M.qualifies(layer, torch.zeros(1, layer.conv.in_channels, 4, 4, 8)), name
    no_stats = _ConvBR(12, 12)
    no_stats.bn = nn.BatchNorm3d(12, track_running_stats=False)
    assert not M.layer_qualifies(no_stats)
    # a qualifying layer on the CPU stays off the kernels
    assert not M.qualifies(_ConvBR(12, 12).eval(), torch.zeros(1, 12, 4, 4, 8))


def test_install_binds_convbr_and_uninstall_restores():
    from rag_b200 import network as N
    from rag_b200.matching_conv import matching_forward

    rag_model, mdenas, ops3d = reference_modules()
    orig = ops3d.ConvBR_3d.forward
    with pytest.raises(ValueError, match="operations_3d"):
        N.install(rag_model, mdenas, None, matching_convs=True)
    N.uninstall()
    try:
        done = N.install(rag_model, mdenas, ops3d, matching_convs=True)
        assert ops3d.ConvBR_3d.forward is matching_forward
        assert done["operations_3d"] == ["ConvBR_3d.forward"]
        assert N._STEM_AWARE and not N._FUSE_STEM
        N.install(rag_model, mdenas, ops3d, fuse_stem=True, upsample=True, matching_convs=True)
        assert ops3d.ConvBR_3d.forward is matching_forward and N._FUSE_STEM
    finally:
        N.uninstall()
    assert ops3d.ConvBR_3d.forward is orig
    assert not N._STEM_AWARE and not N._FUSE_STEM
    # without the flag the binding is the fused stem's, as before
    try:
        N.install(rag_model, mdenas, ops3d, fuse_stem=True)
        from rag_b200.fused_stem import stem_forward

        assert ops3d.ConvBR_3d.forward is stem_forward
    finally:
        N.uninstall()
