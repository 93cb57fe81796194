"""CPU-side checks of the training-mode BatchNorm3d shared by the fused stem and the interior ConvBR_3d layers (csrc/bn3d.cu,
rag_b200/batchnorm.py): argument errors of the C ABI without a GPU, and the mode / running-statistics policy on real
nn.BatchNorm3d modules."""
import copy

import pytest
import torch
import torch.nn as nn


def test_exports_answer_errors_without_gpu():
    from rag_b200 import _cabi

    L = _cabi.lib()
    fake = 256                                    # 16-byte aligned, never dereferenced: every call below fails its checks first
    # null pointers
    assert L.rag_bn3d_moments(None, None, None, 1, 4, 4, 4, 8, None) == -1
    assert L.rag_bn3d_finalize(None, None, None, None, None, None, 4, 64.0, 1e-5, 0.1, 1, 1, None) == -1
    assert L.rag_bn3d_relu(None, None, 1, 4, 4, 4, 8, None) == -1
    assert L.rag_bn3d_bwd_sums(None, None, None, None, None, 1, 4, 4, 4, 8, None) == -1
    assert L.rag_bn3d_bwd_consts(None, None, None, None, 4, 64.0, 1, None) == -1
    assert L.rag_bn3d_bwd_gz(None, None, None, None, 1, 4, 4, 4, 8, None) == -1
    # eval mode reads the running statistics: they are required then, the batch sums are not
    assert L.rag_bn3d_finalize(None, fake, fake, None, None, fake, 4, 64.0, 1e-5, 0.1, 0, 0, None) == -1
    # shapes outside the limits, for a 4-channel layer: the message names the bn3d function and no feature-channel count
    shape_errors = {
        "bn3d_moments": lambda: L.rag_bn3d_moments(fake, fake, fake, 1, 4, 4, 4, 6, None),               # W % 4 != 0
        "bn3d_relu": lambda: L.rag_bn3d_relu(fake, fake, 1, 4, 2, 4, 8, None),                          # D < 3
        "bn3d_bwd_sums": lambda: L.rag_bn3d_bwd_sums(fake, fake, fake, fake, fake, 1, 33, 4, 4, 8, None),  # O > 32
        "bn3d_bwd_gz": lambda: L.rag_bn3d_bwd_gz(fake, fake, fake, fake, 1, 4, 4, 4, 1020, None),       # W > 1016
        "bn3d_finalize": lambda: L.rag_bn3d_finalize(fake, fake, fake, fake, fake, fake, 0, 64.0, 1e-5, 0.1, 1, 1, None),
        "bn3d_bwd_consts": lambda: L.rag_bn3d_bwd_consts(fake, fake, fake, fake, 4, 0.5, 1, None),     # n < 1
    }
    for name, call in shape_errors.items():
        assert call() == -2, name
        msg = L.rag_last_error().decode()
        assert msg.startswith(name + ":") and "C == 12" not in msg, msg
    assert L.rag_bn3d_bwd_gz(fake, fake, fake, fake, 40000, 4, 4, 4, 8, None) == -2                  # B > 32767
    assert L.rag_bn3d_moments(fake, fake, fake, 1, 4, 4, 70000, 8, None) == -2                        # H > 65535


def _stem_copy(bn):
    """The fused stem's decision before it moved to rag_b200.batchnorm (stem_train_forward)."""
    use_batch = bn.training or not bn.track_running_stats
    update = use_batch and bn.training and bn.track_running_stats
    f = 0.0
    if update:
        if bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
        f = (1.0 / float(bn.num_batches_tracked)) if bn.momentum is None else float(bn.momentum)
    return use_batch, update, f


def _convbr_copy(bn):
    """The interior layers' decision before it moved (convbr_forward; their layers always track running statistics)."""
    f = 0.0
    if bn.training:
        if bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
        f = (1.0 / float(bn.num_batches_tracked)) if bn.momentum is None else float(bn.momentum)
    return bn.training, bn.training, f


def _modules():
    return {
        "train": nn.BatchNorm3d(4).train(),
        "train momentum=0.3": nn.BatchNorm3d(4, momentum=0.3).train(),
        "train cumulative average": nn.BatchNorm3d(4, momentum=None).train(),
        "eval": nn.BatchNorm3d(4).eval(),
        "eval cumulative average": nn.BatchNorm3d(4, momentum=None).eval(),
        "no running stats, train": nn.BatchNorm3d(4, track_running_stats=False).train(),
        "no running stats, eval": nn.BatchNorm3d(4, track_running_stats=False).eval(),
    }


@pytest.mark.parametrize("name", list(_modules()))
def test_mode_matches_both_former_copies(name):
    from rag_b200.batchnorm import mode

    bn = _modules()[name]
    copies = [_stem_copy] + ([_convbr_copy] if bn.track_running_stats else [])
    for copy_fn in copies:
        ours, theirs = copy.deepcopy(bn), copy.deepcopy(bn)
        for _ in range(3):                        # the cumulative average changes from call to call
            assert mode(ours) == copy_fn(theirs), (name, copy_fn.__name__)
            assert (ours.num_batches_tracked is None) == (theirs.num_batches_tracked is None)
            if ours.num_batches_tracked is not None:
                assert int(ours.num_batches_tracked) == int(theirs.num_batches_tracked)
    expect = {"train": (True, True, 0.1), "eval": (False, False, 0.0), "no running stats, train": (True, False, 0.0),
              "no running stats, eval": (True, False, 0.0)}
    if name in expect:
        assert mode(copy.deepcopy(bn)) == expect[name]
    if name == "train cumulative average":
        b2 = copy.deepcopy(bn)
        assert [mode(b2)[2] for _ in range(3)] == [1.0, 0.5, 1.0 / 3.0] and int(b2.num_batches_tracked) == 3


def test_apply_bumps_running_buffer_versions_only_when_they_move():
    from rag_b200 import batchnorm

    class Recorder:
        @staticmethod
        def apply(*args):
            Recorder.args = args
            return "out"

    for bn, moves in ((nn.BatchNorm3d(4).train(), True), (nn.BatchNorm3d(4).eval(), False)):
        v0 = (bn.running_mean._version, bn.running_var._version)
        assert batchnorm.apply(Recorder, bn, "x", "w") == "out"
        a = Recorder.args
        assert a[:2] == ("x", "w") and a[2] is bn.weight and a[3] is bn.bias and a[4] is bn.running_mean and a[5] is bn.running_var
        assert a[6:] == (bn.training, moves, 0.1 if moves else 0.0, bn.eps)
        grew = (bn.running_mean._version > v0[0], bn.running_var._version > v0[1])
        assert grew == (moves, moves)


def test_eval_fold():
    from rag_b200.batchnorm import eval_fold

    g = torch.Generator().manual_seed(3)
    for affine in (True, False):
        bn = nn.BatchNorm3d(5, affine=affine).eval()
        with torch.no_grad():
            bn.running_mean.copy_(torch.randn(5, generator=g))
            bn.running_var.copy_(0.5 + torch.rand(5, generator=g))
            if affine:
                bn.weight.copy_(torch.randn(5, generator=g))
                bn.bias.copy_(torch.randn(5, generator=g))
        x = torch.randn(2, 5, 3, 4, 4, generator=g)
        scale, shift = eval_fold(bn)
        with torch.no_grad():
            torch.testing.assert_close(x * scale.view(1, 5, 1, 1, 1) + shift.view(1, 5, 1, 1, 1), bn(x), rtol=1e-5, atol=1e-6)
