"""The BatchNorm3d + ReLU of a ``ConvBR_3d`` (operations_3d.py:31-47) with autograd, on csrc/bn3d.cu: batch or running
statistics, how the running estimates move, and the launches of its forward and backward, for the fused stem
(``fused_stem.FusedStemFn``), the interior layers (``matching_conv.ConvBR3dFn``) and the pointwise layers
(``pointwise_conv.PointwiseBR3dFn``)."""
from __future__ import annotations

import torch
import torch.nn as nn
from torch.autograd.graph import increment_version

from . import _cabi
from .functional import _stream


def _ptr(t):
    return t.data_ptr() if t is not None else None


def bn_relu_qualifies(layer: nn.Module, out_channels: int) -> bool:
    """The BatchNorm / ReLU half of a ConvBR_3d routing predicate (``matching_conv`` and ``pointwise_conv``): ``layer.bn`` is
    an affine fp32 BatchNorm3d over ``out_channels`` that tracks running statistics and is in use, followed by a ReLU."""
    bn = getattr(layer, "bn", None)
    return bool(getattr(layer, "use_bn", False) and isinstance(bn, nn.BatchNorm3d) and bn.affine and bn.track_running_stats
                and bn.num_features == out_channels and bn.weight.dtype == torch.float32 and bn.running_mean.dtype == torch.float32
                and bool(getattr(layer, "relu", False)))


def mode(bn: nn.BatchNorm3d) -> tuple[bool, bool, float]:
    """(use batch statistics, update the running estimates, update factor) for one call of ``bn``, as nn.BatchNorm3d decides
    them; counts the batch in ``num_batches_tracked`` when the estimates move (factor 1/num_batches_tracked if momentum=None)."""
    use_batch = bn.training or not bn.track_running_stats
    update = bn.training and bn.track_running_stats
    f = 0.0
    if update:
        if bn.num_batches_tracked is not None:
            bn.num_batches_tracked.add_(1)
        f = (1.0 / float(bn.num_batches_tracked)) if bn.momentum is None else float(bn.momentum)
    return use_batch, update, f


def apply(fn, bn: nn.BatchNorm3d, *args):
    """``fn.apply(*args, gamma, beta, running_mean, running_var, use_batch, update, factor, eps)`` with ``mode(bn)``.  The
    finaliser writes the running estimates in place: their version counters are bumped afterwards, as F.batch_norm does."""
    use_batch, update, f = mode(bn)
    out = fn.apply(*args, bn.weight, bn.bias, bn.running_mean, bn.running_var, use_batch, update, f, bn.eps)
    if update:
        increment_version(bn.running_mean)
        increment_version(bn.running_var)
    return out


def eval_fold(bn: nn.BatchNorm3d) -> tuple[torch.Tensor, torch.Tensor]:
    """(scale, shift) folding eval-mode ``bn`` into a convolution's store; gamma = 1, beta = 0 without affine parameters."""
    scale = (bn.weight if bn.weight is not None else torch.ones_like(bn.running_var)) * torch.rsqrt(bn.running_var + bn.eps)
    shift = (bn.bias if bn.bias is not None else torch.zeros_like(bn.running_mean)) - bn.running_mean * scale
    return scale, shift


def forward(z, out, gamma, beta, running_mean, running_var, use_batch, update, momentum, eps) -> torch.Tensor:
    """out <- relu(batchnorm(out)) with the statistics of the convolution output z [B,O,D,H,W] (``out`` is z itself or a copy)
    when ``use_batch``, else the running ones; the running estimates move in place when ``update``.  Returns the [O,4] table
    (scale, shift, mean, rstd) that ``backward`` takes."""
    b, o, d, h, w = z.shape
    dev = z.device
    L = _cabi.lib()
    gamma, beta = gamma.contiguous(), beta.contiguous()
    with torch.cuda.device(dev):
        st = _stream(z)
        sums = None
        if use_batch:
            sums = torch.empty((o, 2), dtype=torch.float64, device=dev)
            rows = torch.empty((b * h * o * 2,), dtype=torch.float64, device=dev)
            _cabi.check(L.rag_bn3d_moments(z.data_ptr(), sums.data_ptr(), rows.data_ptr(), b, o, d, h, w, st), "rag_bn3d_moments")
        bn = torch.empty((o, 4), dtype=torch.float32, device=dev)
        _cabi.check(L.rag_bn3d_finalize(_ptr(sums), gamma.data_ptr(), beta.data_ptr(), _ptr(running_mean), _ptr(running_var), bn.data_ptr(),
                                        o, float(b * d * h * w), float(eps), float(momentum), int(bool(use_batch)), int(bool(update)), st),
                    "rag_bn3d_finalize")
        _cabi.check(L.rag_bn3d_relu(out.data_ptr(), bn.data_ptr(), b, o, d, h, w, st), "rag_bn3d_relu")
    return bn


def backward(g, z, bn, use_batch, want_gz):
    """From the contiguous upstream gradient g of the layer output: (consts [O,7], dgamma, dbeta, gz).  consts are what a kernel
    needs to form the gradient gz at the convolution output on the fly; gz itself is formed only when ``want_gz``."""
    b, o, d, h, w = z.shape
    dev = z.device
    n = float(b * d * h * w)
    L = _cabi.lib()
    with torch.cuda.device(dev):
        st = _stream(z)
        sums = torch.empty((o, 2), dtype=torch.float64, device=dev)
        rows = torch.empty((b * h * o * 2,), dtype=torch.float64, device=dev)
        _cabi.check(L.rag_bn3d_bwd_sums(g.data_ptr(), z.data_ptr(), bn.data_ptr(), sums.data_ptr(), rows.data_ptr(), b, o, d, h, w, st),
                    "rag_bn3d_bwd_sums")
        consts = torch.empty((o, 7), dtype=torch.float32, device=dev)
        gparam = torch.empty((2, o), dtype=torch.float32, device=dev)
        _cabi.check(L.rag_bn3d_bwd_consts(sums.data_ptr(), bn.data_ptr(), consts.data_ptr(), gparam.data_ptr(), o, n, int(bool(use_batch)), st),
                    "rag_bn3d_bwd_consts")
        gz = None
        if want_gz:
            gz = torch.empty_like(z)
            _cabi.check(L.rag_bn3d_bwd_gz(g.data_ptr(), z.data_ptr(), consts.data_ptr(), gz.data_ptr(), b, o, d, h, w, st), "rag_bn3d_bwd_gz")
    return consts, gparam[0], gparam[1], gz
