"""CPU-side checks of the TF32 weight gradient of the interior ConvBR_3d layers (csrc/conv3d_cc_tf32.cu): argument errors and
the workspace query of its C entries without a GPU, and the ``install(..., matching_tf32_wgrad=True)`` flag's rules."""
import pytest
import torch

from tests._stand_in import _stand_in


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi

    L = _cabi.lib()
    fake = 256
    bwd = L.rag_conv3d_cc_tf32_bwd_weight
    for i in range(4):                                     # gz, in, gw, workspace: each required
        args = [fake] * 4
        args[i] = None
        assert bwd(*args, 1, 12, 12, 4, 4, 8, None) == -1
        assert b"null" in L.rag_last_error()
    # shape errors are reported before any pointer is touched: uncompiled pairs (4 -> 4 included), W % 4, a non-positive
    # dimension
    for c, o in ((4, 4), (5, 5), (16, 16), (12, 8)):
        assert bwd(fake, fake, fake, fake, 1, c, o, 4, 4, 8, None) == -2
        assert b"not compiled" in L.rag_last_error()
    assert bwd(fake, fake, fake, fake, 1, 12, 12, 4, 4, 6, None) == -2
    assert bwd(fake, fake, fake, fake, 1, 8, 8, 4, 4, 10, None) == -2
    assert bwd(fake, fake, fake, fake, 0, 8, 8, 4, 4, 8, None) == -2
    assert bwd(fake, fake, fake, fake, 1, 8, 8, 0, 4, 8, None) == -2
    # misaligned pointers (the shape is fine): gz / in want 16 bytes, gw / workspace 4
    assert bwd(fake + 4, fake, fake, fake, 1, 8, 8, 4, 4, 8, None) == -3
    assert bwd(fake, fake + 4, fake, fake, 1, 12, 12, 4, 4, 8, None) == -3
    assert bwd(fake, fake, fake + 2, fake, 1, 12, 12, 4, 4, 8, None) == -3
    assert bwd(fake, fake, fake, fake + 2, 1, 12, 12, 4, 4, 8, None) == -3


def test_workspace_query():
    """Non-zero exactly for the compiled pairs, the fp32 entry's size there; no device needed."""
    from rag_b200 import _cabi

    L = _cabi.lib()
    q = L.rag_conv3d_cc_tf32_bwd_weight_workspace_bytes
    for c, o in ((8, 8), (12, 12)):
        n = q(4, c, o, 64, 96, 192)
        assert n > 0 and n % (o * c * 27 * 4) == 0
        assert n == L.rag_conv3d_cc_bwd_workspace_bytes(4, c, o, 64, 96, 192)
        assert q(0, c, o, 64, 96, 192) == 0 and q(4, c, o, 64, 96, 0) == 0
    for c, o in ((4, 4), (16, 16), (12, 8), (5, 5), (0, 0)):
        assert q(4, c, o, 64, 96, 192) == 0


def test_install_flag_rules():
    from rag_b200 import matching_conv
    from rag_b200 import network as N

    rag_model, ops3d, _ = _stand_in()
    old = torch.backends.cudnn.allow_tf32
    N.uninstall()
    try:
        torch.backends.cudnn.allow_tf32 = True
        with pytest.raises(ValueError, match="matching_tf32=True"):
            N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32_wgrad=True)
        assert not matching_conv.use_tf32_wgrad(12)
        N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32=True)   # matching_tf32 alone: fp32 weight gradient
        assert matching_conv.use_tf32(12) and not matching_conv.use_tf32_wgrad(12)
        N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32=True, matching_tf32_wgrad=True)
        assert matching_conv.use_tf32_wgrad(12) and matching_conv.use_tf32_wgrad(8) and not matching_conv.use_tf32_wgrad(4)
        torch.backends.cudnn.allow_tf32 = False           # read at call time
        assert not matching_conv.use_tf32_wgrad(12)
        torch.backends.cudnn.allow_tf32 = True
        assert matching_conv.use_tf32_wgrad(12)
        N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32=True)   # a later install() without it turns it off
        assert matching_conv.use_tf32(12) and not matching_conv.use_tf32_wgrad(12)
        N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32=True, matching_tf32_wgrad=True)
        N.uninstall()
        assert not matching_conv.use_tf32_wgrad(12) and not matching_conv.use_tf32(12)
    finally:
        N.uninstall()
        torch.backends.cudnn.allow_tf32 = old
