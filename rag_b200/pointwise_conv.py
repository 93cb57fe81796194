"""The Matching Net's pointwise layers on the hand-written kernels, inference and training.

``ConvBR_3d(C, O, 1, 1, 0)`` (operations_3d.py:31-47) is a bias-free 1x1x1 Conv3d C -> O followed by BatchNorm3d and ReLU:
``last_12_3d`` (48 -> 24), ``last_6_3d`` (24 -> 12) and, inferred from those, the cells' own 1x1x1 layers.  They do almost
no arithmetic per byte, so what they cost is passes over HBM; ``csrc/conv3d_pw.cu`` runs them in fp32 for any
1 <= C <= 64, 1 <= O <= 32:

* inference (BatchNorm in eval(), no gradient): one pass, the BatchNorm folded into the store with the ReLU;
* with batch statistics or a gradient: ``PointwiseBR3dFn`` -- the raw convolution output z, then the BatchNorm + ReLU of
  ``batchnorm`` (csrc/bn3d.cu) into a copy of z.  The backward takes the BatchNorm constants from ``batchnorm.backward`` and
  runs one fused kernel that forms the gradient at the convolution output in registers and produces the data gradient and
  the per-CTA weight-gradient partials from it (bitwise repeatable).

``qualifies(layer, x)`` is the only routing decision; ``pointwise_forward`` -- bound onto ``ConvBR_3d.forward`` by
``rag_b200.network.install(..., pointwise_convs=True)`` -- sends qualifying plain-tensor calls here and everything else to
the binding ``install()`` makes without the flag (``fallthrough``).
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _cabi, batchnorm
from .functional import _require, _stream
from .fused_stem import stem_forward
from .matching_conv import _wants_grad, matching_forward

MAX_C, MAX_O = 64, 32       # the limits of csrc/conv3d_pw.cu (O: also the BatchNorm kernels' limit)
# Smaller inputs (B*D*H*W voxels) stay on cuDNN, a conservative rule: at the level-12 shape of B=4 288x576 (73,728 voxels)
# cuDNN TF32 beat these kernels for 48 -> 24 and was only 7 % slower (training) for 48 -> 16; at 409,600 voxels and up
# they win 2.4x or more.  Nothing between the two sizes was measured: 2^17 lies between them (DESIGN.md 5.11,
# profiles/r4_pointwise_conv_times.jsonl)
MIN_VOXELS = 2 ** 17


def conv3d_pw_forward(x: torch.Tensor, weight: torch.Tensor, scale=None, shift=None, relu: bool = False) -> torch.Tensor:
    """out = relu?(fma(conv3d(x, weight), scale, shift)) for weight [O,C,1,1,1]; x [B,C,D,H,W] CUDA fp32 with D*H*W % 4 == 0.
    scale / shift [O] (both or neither) fold an eval-mode BatchNorm into the store."""
    _require(x, "x"), _require(weight, "weight")
    if x.dim() != 5:
        raise RuntimeError(f"rag_b200: conv3d_pw wants a [B,C,D,H,W] input, got {tuple(x.shape)}")
    b, c, d, h, w = x.shape
    o = weight.shape[0]
    if tuple(weight.shape) != (o, c, 1, 1, 1):
        raise RuntimeError(f"rag_b200: conv3d_pw wants a [O,{c},1,1,1] weight, got {tuple(weight.shape)}")
    if (scale is None) != (shift is None):
        raise RuntimeError("rag_b200: conv3d_pw takes scale and shift together")
    x, weight = x.contiguous(), weight.contiguous()
    out = torch.empty((b, o, d, h, w), dtype=torch.float32, device=x.device)
    if out.numel() == 0:
        return out
    if scale is not None:
        scale, shift = scale.contiguous(), shift.contiguous()
    L = _cabi.lib()
    with torch.cuda.device(x.device):
        rc = L.rag_conv3d_pw_fwd(x.data_ptr(), weight.data_ptr(), scale.data_ptr() if scale is not None else None,
                                 shift.data_ptr() if shift is not None else None, int(bool(relu)), out.data_ptr(),
                                 b, c, o, d, h, w, _stream(x))
    _cabi.check(rc, "rag_conv3d_pw_fwd")
    return out


class PointwiseBR3dFn(torch.autograd.Function):
    """out = relu(batchnorm(conv3d_1x1x1(x, weight))) with gradients w.r.t. x, weight, gamma and beta, each only when wanted.

    Same BatchNorm handling as ``matching_conv.ConvBR3dFn`` (batch or running statistics, running estimates updated in place
    by ``batchnorm``).  Saved for the backward: x, the convolution output z and the [O,4] table.  The backward never writes
    the gradient at the convolution output: the fused kernel forms it from g, z and the BatchNorm constants in registers."""

    @staticmethod
    def forward(ctx, x, weight, gamma, beta, running_mean, running_var, batch_stats, update_running, momentum, eps):
        z = conv3d_pw_forward(x, weight)
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
        g = g.contiguous()
        consts, ggamma, gbeta, _ = batchnorm.backward(g, z, bn, ctx.batch_stats, want_gz=False)
        gx = gw = None
        if need_x or need_w:
            L = _cabi.lib()
            weight = weight.contiguous()
            with torch.cuda.device(x.device):
                gx = torch.empty_like(x) if need_x else None
                gw = torch.empty_like(weight) if need_w else None
                ws = torch.empty(int(L.rag_conv3d_pw_bwd_workspace_bytes(b, c, o, d, h, w)) // 4, dtype=torch.float32, device=x.device) if need_w else None
                rc = L.rag_conv3d_pw_bwd(g.data_ptr(), z.data_ptr(), consts.data_ptr(), x.data_ptr(), weight.data_ptr(),
                                         gx.data_ptr() if gx is not None else None, gw.data_ptr() if gw is not None else None,
                                         ws.data_ptr() if ws is not None else None, b, c, o, d, h, w, _stream(x))
            _cabi.check(rc, "rag_conv3d_pw_bwd")
        return gx, gw, ggamma if need_gamma else None, gbeta if need_beta else None, None, None, None, None, None, None


def layer_qualifies(layer: nn.Module) -> bool:
    """The layer half of ``qualifies``, independent of devices: ``layer`` (a ConvBR_3d: .conv, .bn, .use_bn, .relu) is a
    Conv3d 1x1x1 / stride 1 / padding 0 / dilation 1 / groups 1, bias-free, fp32, with 1 <= C <= MAX_C and 1 <= O <= MAX_O,
    followed by an affine fp32 BatchNorm3d that tracks running statistics and a ReLU (``batchnorm.bn_relu_qualifies``)."""
    conv = getattr(layer, "conv", None)
    if not (isinstance(conv, nn.Conv3d) and conv.bias is None and conv.kernel_size == (1, 1, 1) and conv.stride == (1, 1, 1)
            and conv.padding == (0, 0, 0) and conv.dilation == (1, 1, 1) and conv.groups == 1
            and conv.weight.dtype == torch.float32 and 1 <= conv.in_channels <= MAX_C and 1 <= conv.out_channels <= MAX_O):
        return False
    return batchnorm.bn_relu_qualifies(layer, conv.out_channels)


def qualifies(layer: nn.Module, x) -> bool:
    """True when ``layer(x)`` is the layer csrc/conv3d_pw.cu implements: ``layer_qualifies(layer)`` with the weight on CUDA,
    and x a CUDA fp32 [B,C,D,H,W] tensor on the weight's device with D*H*W % 4 == 0, B <= 65535 and at least MIN_VOXELS
    voxels in all (a conservative floor: the smallest measured shape, under it, had cuDNN faster for one layer and barely
    slower for another; see MIN_VOXELS).  Whenever batch statistics are used or a gradient is wanted, also the limits of the
    BatchNorm kernels (csrc/bn3d.cu): D >= 3, 8 <= W <= 1016, W % 4 == 0, B <= 32767, H <= 65535."""
    if not layer_qualifies(layer) or not layer.conv.weight.is_cuda:
        return False
    conv, bn = layer.conv, layer.bn
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and x.device == conv.weight.device
            and x.shape[1] == conv.in_channels and x.numel() > 0):
        return False
    b, _, d, h, w = x.shape
    if (d * h * w) % 4 or b > 65535 or (d * h * w + 255) // 256 >= 2 ** 31 or b * d * h * w < MIN_VOXELS:
        return False
    if x.is_contiguous() and x.data_ptr() % 16:
        return False
    if bn.training or _wants_grad(layer, x):
        if not (d >= 3 and 8 <= w <= 1016 and w % 4 == 0 and b <= 32767 and h <= 65535
                and b * conv.out_channels * d * h * w < 2 ** 40):
            return False
    return True


def convbr_forward(layer: nn.Module, x: torch.Tensor) -> torch.Tensor:
    """A qualifying pointwise ConvBR_3d call on the kernels.  Updates the running statistics exactly like nn.BatchNorm3d does
    in train() (momentum or cumulative average, unbiased variance, batch count)."""
    if not layer.bn.training and not _wants_grad(layer, x):
        return conv3d_pw_forward(x, layer.conv.weight, *batchnorm.eval_fold(layer.bn), relu=True)
    return batchnorm.apply(PointwiseBR3dFn, layer.bn, x.contiguous(), layer.conv.weight)


def _make_forward(fallthrough):
    def pointwise_forward(self, x):
        """Replacement for ConvBR_3d.forward (operations_3d.py:41-47) under ``install(..., pointwise_convs=True)``."""
        if isinstance(x, torch.Tensor) and qualifies(self, x):
            return convbr_forward(self, x)
        return fallthrough(self, x)

    pointwise_forward.fallthrough = fallthrough
    return pointwise_forward


# the two bindings install(..., pointwise_convs=True) makes: non-qualifying calls go where install() sends them without the flag
pointwise_forward = _make_forward(stem_forward)
pointwise_matching_forward = _make_forward(matching_forward)
