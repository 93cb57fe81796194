"""The Matching Net's interior 3x3x3 layers on the hand-written kernels, inference and training.

``ConvBR_3d(C, O, 3, 1, 1)`` (operations_3d.py:31-47) is a bias-free Conv3d C -> O (3x3x3, stride 1, zero padding 1)
followed by BatchNorm3d and ReLU.  In the growable ``Network`` it is ``stem3d1`` (12 -> 12 at the volume's resolution) and
every ``conv_3x3`` op of the ``Cell_3d``s.  cuDNN is poor at these small-channel 3-D convolutions; ``csrc/conv3d_cc.cu``
runs them in fp32 for (C, O) in ``PAIRS``:

* inference (BatchNorm in eval(), no gradient): one pass, the BatchNorm folded into the store with the ReLU;
* with batch statistics or a gradient: ``ConvBR3dFn`` -- the raw convolution output z, then the BatchNorm + ReLU of
  ``batchnorm`` (csrc/bn3d.cu) into a copy of z (z survives for the backward).  The backward forms the gradient at the
  convolution output once (``batchnorm.backward``), runs the forward kernel on it with the weights transposed and flipped for
  the data gradient, and reduces the weight gradient in a fixed order (bitwise repeatable).

``qualifies(layer, x)`` is the only routing decision; ``matching_forward`` -- bound onto ``ConvBR_3d.forward`` by
``rag_b200.network.install(..., matching_convs=True)`` -- sends qualifying plain-tensor calls here and everything else to
``fused_stem.stem_forward`` unchanged.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _cabi, batchnorm
from .functional import _require, _stream
from .fused_stem import stem_forward

PAIRS = ((4, 4), (8, 8), (12, 12))     # the (C, O) instantiations of csrc/conv3d_cc.cu (16 -> 16 lost to cuDNN: DESIGN.md 5.10)


def conv3d_cc_forward(x: torch.Tensor, weight: torch.Tensor, scale=None, shift=None, relu: bool = False) -> torch.Tensor:
    """out = relu?(fma(conv3d(x, weight, padding=1), scale, shift)) for weight [O,C,3,3,3]; x [B,C,D,H,W] CUDA fp32.
    scale / shift [O] (both or neither) fold an eval-mode BatchNorm into the store."""
    _require(x, "x"), _require(weight, "weight")
    if x.dim() != 5:
        raise RuntimeError(f"rag_b200: conv3d_cc wants a [B,C,D,H,W] input, got {tuple(x.shape)}")
    b, c, d, h, w = x.shape
    o = weight.shape[0]
    if tuple(weight.shape) != (o, c, 3, 3, 3):
        raise RuntimeError(f"rag_b200: conv3d_cc wants a [O,{c},3,3,3] weight, got {tuple(weight.shape)}")
    if (scale is None) != (shift is None):
        raise RuntimeError("rag_b200: conv3d_cc takes scale and shift together")
    x, weight = x.contiguous(), weight.contiguous()
    out = torch.empty((b, o, d, h, w), dtype=torch.float32, device=x.device)
    if out.numel() == 0:
        return out
    if scale is not None:
        scale, shift = scale.contiguous(), shift.contiguous()
    L = _cabi.lib()
    with torch.cuda.device(x.device):
        rc = L.rag_conv3d_cc_fwd(x.data_ptr(), weight.data_ptr(), scale.data_ptr() if scale is not None else None,
                                 shift.data_ptr() if shift is not None else None, int(bool(relu)), out.data_ptr(),
                                 b, c, o, d, h, w, _stream(x))
    _cabi.check(rc, "rag_conv3d_cc_fwd")
    return out


class ConvBR3dFn(torch.autograd.Function):
    """out = relu(batchnorm(conv3d(x, weight))) with gradients w.r.t. x, weight, gamma and beta, each only when wanted.

    BatchNorm with batch statistics (``batch_stats``; the running estimates updated in place when ``update_running``) or with
    the running statistics (eval-mode BatchNorm behind trainable layers).  Saved for the backward: x, the convolution output z
    and the [O,4] table (scale, shift, mean, rstd) -- the reference's own layer keeps its conv output too, so no fourth
    convolution pass is spent on recomputing z.  The backward re-evaluates the forward's own ``fma(z, scale, shift) > 0`` for
    the ReLU decision (bit-identical)."""

    @staticmethod
    def forward(ctx, x, weight, gamma, beta, running_mean, running_var, batch_stats, update_running, momentum, eps):
        z = conv3d_cc_forward(x, weight)
        out = z.clone()
        bn = batchnorm.forward(z, out, gamma, beta, running_mean, running_var, batch_stats, update_running, momentum, eps)
        ctx.save_for_backward(x, weight, z, bn)
        ctx.batch_stats = bool(batch_stats)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        x, weight, z, bn = ctx.saved_tensors
        b, c, d, h, w = x.shape
        o = weight.shape[0]
        need_x, need_w, need_gamma, need_beta = ctx.needs_input_grad[:4]
        _, ggamma, gbeta, gz = batchnorm.backward(g.contiguous(), z, bn, ctx.batch_stats, want_gz=need_x or need_w)
        gx = gw = None
        if need_x or need_w:
            L = _cabi.lib()
            with torch.cuda.device(x.device):
                gx = torch.empty_like(x) if need_x else None
                gw = torch.empty_like(weight) if need_w else None
                ws = torch.empty(int(L.rag_conv3d_cc_bwd_workspace_bytes(b, c, o, d, h, w)) // 4, dtype=torch.float32, device=x.device) if need_w else None
                rc = L.rag_conv3d_cc_bwd(gz.data_ptr(), x.data_ptr(), weight.data_ptr(), gx.data_ptr() if gx is not None else None,
                                         gw.data_ptr() if gw is not None else None, ws.data_ptr() if ws is not None else None,
                                         b, c, o, d, h, w, _stream(x))
            _cabi.check(rc, "rag_conv3d_cc_bwd")
        return gx, gw, ggamma if need_gamma else None, gbeta if need_beta else None, None, None, None, None, None, None


def _wants_grad(layer: nn.Module, x: torch.Tensor) -> bool:
    return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in layer.parameters()))


def layer_qualifies(layer: nn.Module) -> bool:
    """The layer half of ``qualifies``, independent of devices: ``layer`` (a ConvBR_3d: .conv, .bn, .use_bn, .relu) is a
    Conv3d 3x3x3 / stride 1 / padding 1 / dilation 1 / groups 1, bias-free (the kernels have no bias term), zero padding,
    fp32, with (C, O) in PAIRS, followed by an affine fp32 BatchNorm3d that tracks running statistics and a ReLU."""
    conv = getattr(layer, "conv", None)
    if not (isinstance(conv, nn.Conv3d) and conv.bias is None and conv.kernel_size == (3, 3, 3) and conv.stride == (1, 1, 1)
            and conv.padding == (1, 1, 1) and conv.dilation == (1, 1, 1) and conv.groups == 1 and conv.padding_mode == "zeros"
            and conv.weight.dtype == torch.float32 and (conv.in_channels, conv.out_channels) in PAIRS):
        return False
    return batchnorm.bn_relu_qualifies(layer, conv.out_channels)


def qualifies(layer: nn.Module, x) -> bool:
    """True when ``layer(x)`` is the layer csrc/conv3d_cc.cu implements: ``layer_qualifies(layer)`` with the weight on CUDA,
    and x a CUDA fp32 [B,C,D,H,W] tensor on the weight's device with W % 4 == 0 and within the kernels' limits.  Whenever
    batch statistics are used or a gradient is wanted, also the limits of the BatchNorm kernels (csrc/bn3d.cu):
    O <= 32, D >= 3, 8 <= W <= 1016."""
    if not layer_qualifies(layer) or not layer.conv.weight.is_cuda:
        return False
    conv, bn = layer.conv, layer.bn
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.device == conv.weight.device
            and x.shape[1] == conv.in_channels and x.numel() > 0):
        return False
    b, _, d, h, w = x.shape
    if w % 4 or 3 * h * w + 68 >= 2 ** 31 or b * ((d + 7) // 8) > 65535 or (h + 1) // 2 > 65535:
        return False
    if x.is_contiguous() and x.data_ptr() % 16:
        return False
    if bn.training or _wants_grad(layer, x):
        if not (d >= 3 and 8 <= w <= 1016 and b <= 32767 and h <= 65535):
            return False
    return True


def convbr_forward(layer: nn.Module, x: torch.Tensor) -> torch.Tensor:
    """A qualifying ConvBR_3d call on the kernels.  Updates the running statistics exactly like nn.BatchNorm3d does in
    train() (momentum or cumulative average, unbiased variance, batch count)."""
    if not layer.bn.training and not _wants_grad(layer, x):
        return conv3d_cc_forward(x, layer.conv.weight, *batchnorm.eval_fold(layer.bn), relu=True)
    return batchnorm.apply(ConvBR3dFn, layer.bn, x.contiguous(), layer.conv.weight)


def matching_forward(self, x):
    """Replacement for ConvBR_3d.forward (operations_3d.py:41-47) under ``install(..., matching_convs=True)``."""
    if isinstance(x, torch.Tensor) and qualifies(self, x):
        return convbr_forward(self, x)
    return stem_forward(self, x)
