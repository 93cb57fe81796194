"""CPU-side checks of the TF32 interior ConvBR_3d path (csrc/conv3d_cc_tf32.cu): argument errors of its two C entries
without a GPU, and the ``install(..., matching_tf32=True)`` flag's rules."""
import pytest
import torch

from tests._stand_in import _stand_in


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi

    L = _cabi.lib()
    fake = 256
    assert L.rag_conv3d_cc_tf32_fwd(None, None, None, None, 1, None, 1, 12, 12, 4, 4, 8, None) == -1
    assert b"null" in L.rag_last_error()
    assert L.rag_conv3d_cc_tf32_fwd(fake, fake, fake, None, 1, fake, 1, 12, 12, 4, 4, 8, None) == -1      # scale without shift
    assert L.rag_conv3d_cc_tf32_bwd_data(None, fake, fake, 1, 12, 12, 4, 4, 8, None) == -1
    assert L.rag_conv3d_cc_tf32_bwd_data(fake, None, fake, 1, 12, 12, 4, 4, 8, None) == -1
    assert L.rag_conv3d_cc_tf32_bwd_data(fake, fake, None, 1, 12, 12, 4, 4, 8, None) == -1
    # shape errors are reported before any pointer is touched: an uncompiled pair, W % 4, a non-positive dimension
    for c, o in ((5, 5), (16, 16), (12, 8)):
        assert L.rag_conv3d_cc_tf32_fwd(fake, fake, None, None, 0, fake, 1, c, o, 4, 4, 8, None) == -2
        assert b"not compiled" in L.rag_last_error()
        assert L.rag_conv3d_cc_tf32_bwd_data(fake, fake, fake, 1, c, o, 4, 4, 8, None) == -2
    assert L.rag_conv3d_cc_tf32_fwd(fake, fake, None, None, 0, fake, 1, 12, 12, 4, 4, 6, None) == -2
    assert L.rag_conv3d_cc_tf32_bwd_data(fake, fake, fake, 1, 8, 8, 4, 4, 10, None) == -2
    assert L.rag_conv3d_cc_tf32_fwd(fake, fake, None, None, 0, fake, 0, 4, 4, 4, 4, 8, None) == -2
    # a misaligned pointer (the shape is fine)
    assert L.rag_conv3d_cc_tf32_fwd(fake + 4, fake, None, None, 0, fake, 1, 4, 4, 4, 4, 8, None) == -3
    assert L.rag_conv3d_cc_tf32_bwd_data(fake, fake, fake + 4, 1, 4, 4, 4, 4, 8, None) == -3


def test_cpu_tensors_raise():
    from rag_b200.matching_conv import conv3d_cc_forward

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conv3d_cc_forward(torch.zeros(1, 12, 3, 4, 8), torch.zeros(12, 12, 3, 3, 3), tf32=True)


def test_install_flag_rules():
    from rag_b200 import matching_conv
    from rag_b200 import network as N

    rag_model, ops3d, _ = _stand_in()
    old = torch.backends.cudnn.allow_tf32
    N.uninstall()
    try:
        torch.backends.cudnn.allow_tf32 = True
        with pytest.raises(ValueError, match="matching_convs"):
            N.install(rag_model, None, ops3d, fuse_stem=True, matching_tf32=True)
        assert not matching_conv.use_tf32(12)
        N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32=True)
        assert matching_conv.use_tf32(12) and matching_conv.use_tf32(8) and not matching_conv.use_tf32(4)
        torch.backends.cudnn.allow_tf32 = False           # read at call time
        assert not matching_conv.use_tf32(12)
        torch.backends.cudnn.allow_tf32 = True
        N.uninstall()
        assert not matching_conv.use_tf32(12)
        N.install(rag_model, None, ops3d, matching_convs=True, matching_tf32=True)
        N.install(rag_model, None, ops3d, matching_convs=True)   # a later install() without the flag turns it off
        assert not matching_conv.use_tf32(12)
    finally:
        N.uninstall()
        torch.backends.cudnn.allow_tf32 = old
