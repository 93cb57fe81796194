"""CPU-side checks of the pointwise ConvBR_3d path (csrc/conv3d_pw.cu, rag_b200/pointwise_conv.py): argument errors of the C
ABI without a GPU, no CPU fallback, the routing predicate's exclusions and the install()/uninstall() binding."""
import pytest
import torch
import torch.nn as nn

from tests._mirror_net import reference_modules

FAKE = 256          # a 16-byte aligned non-null "pointer": every call below must fail before touching it


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi

    L = _cabi.lib()
    # null pointers: -1 with "null" in the text
    assert L.rag_conv3d_pw_fwd(None, None, None, None, 1, None, 1, 48, 24, 4, 4, 8, None) == -1
    assert b"null" in L.rag_last_error()
    assert L.rag_conv3d_pw_fwd(FAKE, FAKE, FAKE, None, 1, FAKE, 1, 48, 24, 4, 4, 8, None) == -1      # scale without shift
    assert b"null" in L.rag_last_error()
    assert L.rag_conv3d_pw_bwd(None, None, None, None, None, None, None, None, 1, 48, 24, 4, 4, 8, None) == -1
    assert b"null" in L.rag_last_error()
    assert L.rag_conv3d_pw_bwd(FAKE, FAKE, FAKE, None, None, FAKE, None, None, 1, 48, 24, 4, 4, 8, None) == -1   # gin without w
    assert L.rag_conv3d_pw_bwd(FAKE, FAKE, FAKE, FAKE, FAKE, None, FAKE, None, 1, 48, 24, 4, 4, 8, None) == -1   # gw without workspace
    # shapes outside the limits: -2, before any pointer is touched
    for c, o, d, h, w in [(65, 24, 4, 4, 8), (48, 33, 4, 4, 8), (48, 0, 4, 4, 8), (0, 4, 4, 4, 8), (12, 4, 3, 3, 3), (12, 4, 1, 1, 6)]:
        assert L.rag_conv3d_pw_fwd(FAKE, FAKE, None, None, 0, FAKE, 1, c, o, d, h, w, None) == -2, (c, o, d, h, w)
        assert L.rag_conv3d_pw_bwd(FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 1, c, o, d, h, w, None) == -2, (c, o, d, h, w)
        assert L.rag_conv3d_pw_bwd_workspace_bytes(1, c, o, d, h, w) == 0, (c, o, d, h, w)
    assert L.rag_conv3d_pw_fwd(FAKE, FAKE, None, None, 0, FAKE, 65536, 12, 4, 4, 4, 8, None) == -2                 # B > 65535
    # misaligned tensors: -3
    assert L.rag_conv3d_pw_fwd(FAKE + 4, FAKE, None, None, 0, FAKE, 1, 12, 4, 4, 4, 8, None) == -3
    assert L.rag_conv3d_pw_bwd(FAKE, FAKE + 8, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 1, 12, 4, 4, 4, 8, None) == -3
    # the workspace query: non-zero inside the limits, one fp32 partial per weight and CTA of a grid that depends on (C, O)
    # only (148 x 1..6 CTAs), whatever the batch and volume
    for c in (1, 5, 12, 48, 64):
        for o in (1, 3, 4, 24, 32):
            n = L.rag_conv3d_pw_bwd_workspace_bytes(2, c, o, 4, 4, 8)
            assert n % (148 * o * c * 4) == 0 and 1 <= n // (148 * o * c * 4) <= 6, (c, o, n)
            assert L.rag_conv3d_pw_bwd_workspace_bytes(7, c, o, 64, 96, 192) == n, (c, o)


def test_cpu_tensors_raise():
    from rag_b200.pointwise_conv import conv3d_pw_forward

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conv3d_pw_forward(torch.zeros(1, 12, 3, 4, 8), torch.zeros(4, 12, 1, 1, 1))


class _ConvBR(nn.Module):
    """The reference's ConvBR_3d field layout (operations_3d.py:31-47); a pointwise layer by default."""

    def __init__(self, c, o, k=1, s=1, p=0, bn=True, relu=True, bias=False, affine=True, track=True):
        super().__init__()
        self.conv = nn.Conv3d(c, o, k, stride=s, padding=p, bias=bias)
        self.use_bn = bn
        self.bn = nn.BatchNorm3d(o, affine=affine, track_running_stats=track) if bn else None
        self.relu = relu


def _excluded():
    return {
        "3x3x3 kernel": _ConvBR(48, 24, 3, 1, 1),
        "stride 2": _ConvBR(48, 24, 1, 2, 0),
        "padding 1": _ConvBR(48, 24, 1, 1, 1),
        "bias": _ConvBR(48, 24, bias=True),
        "no BatchNorm": _ConvBR(48, 24, bn=False),
        "affine-free BatchNorm": _ConvBR(48, 24, affine=False),
        "track_running_stats=False": _ConvBR(48, 24, track=False),
        "no ReLU": _ConvBR(48, 24, relu=False),
        "fp64": _ConvBR(48, 24).double(),
        "O > 32": _ConvBR(48, 33),
        "C > 64": _ConvBR(65, 24),
    }


def test_layer_qualifies_positive_control_and_exclusions():
    """Each exclusion differs from a qualifying construction in one field only; the predicate is device-independent."""
    from rag_b200 import pointwise_conv as P

    for c, o in [(48, 24), (24, 12), (5, 3), (12, 4), (1, 1), (64, 32)]:
        assert P.layer_qualifies(_ConvBR(c, o)), (c, o)
    for name, layer in _excluded().items():
        assert not P.layer_qualifies(layer), name
        assert not P.qualifies(layer, torch.zeros(1, layer.conv.in_channels, 4, 4, 8)), name
    # a qualifying layer on the CPU stays off the kernels
    assert not P.qualifies(_ConvBR(48, 24).eval(), torch.zeros(1, 48, 4, 4, 8))


def test_matching_conv_answers_as_before():
    """The BatchNorm / ReLU half now lives in batchnorm.bn_relu_qualifies: matching_conv.layer_qualifies still accepts its
    3x3x3 pairs and rejects every pointwise layer and every BatchNorm / ReLU exclusion above."""
    from rag_b200 import matching_conv as M

    for c in (4, 8, 12):
        assert M.layer_qualifies(_ConvBR(c, c, 3, 1, 1))
    for c, o in [(48, 24), (24, 12), (5, 3), (12, 4), (12, 12), (4, 4)]:
        assert not M.layer_qualifies(_ConvBR(c, o))
    for name, layer in _excluded().items():
        assert not M.layer_qualifies(layer), name
    for kw in (dict(bn=False), dict(affine=False), dict(track=False), dict(relu=False), dict(bias=True)):
        assert not M.layer_qualifies(_ConvBR(12, 12, 3, 1, 1, **kw)), kw
    assert not M.layer_qualifies(_ConvBR(12, 12, 3, 1, 1).double())


def test_install_binds_pointwise_and_uninstall_restores():
    from rag_b200 import network as N
    from rag_b200.fused_stem import stem_forward
    from rag_b200.matching_conv import matching_forward
    from rag_b200.pointwise_conv import pointwise_forward, pointwise_matching_forward

    rag_model, mdenas, ops3d = reference_modules()
    orig = ops3d.ConvBR_3d.forward
    with pytest.raises(ValueError, match="operations_3d"):
        N.install(rag_model, mdenas, None, pointwise_convs=True)
    N.uninstall()
    try:
        # the flag alone: the fallthrough is the fused stem's binding
        done = N.install(rag_model, mdenas, ops3d, pointwise_convs=True)
        assert ops3d.ConvBR_3d.forward is pointwise_forward and pointwise_forward.fallthrough is stem_forward
        assert done["operations_3d"] == ["ConvBR_3d.forward"]
        assert N._STEM_AWARE and not N._FUSE_STEM
        # with matching_convs: the fallthrough is matching_forward
        N.install(rag_model, mdenas, ops3d, matching_convs=True, pointwise_convs=True)
        assert ops3d.ConvBR_3d.forward is pointwise_matching_forward and pointwise_matching_forward.fallthrough is matching_forward
        # with fuse_stem (and the rest): same rule, the stem flag is kept
        N.install(rag_model, mdenas, ops3d, fuse_stem=True, upsample=True, pointwise_convs=True)
        assert ops3d.ConvBR_3d.forward is pointwise_forward and N._FUSE_STEM
        N.install(rag_model, mdenas, ops3d, fuse_stem=True, upsample=True, matching_convs=True, pointwise_convs=True)
        assert ops3d.ConvBR_3d.forward is pointwise_matching_forward and N._FUSE_STEM
    finally:
        N.uninstall()
    assert ops3d.ConvBR_3d.forward is orig
    assert not N._STEM_AWARE and not N._FUSE_STEM
    # without the flag nothing changes
    try:
        N.install(rag_model, mdenas, ops3d, matching_convs=True)
        assert ops3d.ConvBR_3d.forward is matching_forward
        N.install(rag_model, mdenas, ops3d, fuse_stem=True)
        assert ops3d.ConvBR_3d.forward is stem_forward
    finally:
        N.uninstall()
    assert ops3d.ConvBR_3d.forward is orig
