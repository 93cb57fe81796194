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

With ``install(..., matching_convs=True, matching_tf32=True)`` the convolutions of a qualifying call run on the tensor cores
in TF32 (csrc/conv3d_cc_tf32.cu: the forward, and the data gradient) while ``torch.backends.cudnn.allow_tf32`` is on, read
at call time -- the switch that makes the reference's own cuDNN convolutions TF32.  The BatchNorm and the weight gradient
stay fp32, and so does 4 -> 4 (``use_tf32``).  With ``matching_tf32_wgrad=True`` as well, the weight gradient of such a call
runs in TF32 too (``use_tf32_wgrad``; csrc/conv3d_cc_tf32.cu's weight-gradient kernel), so all three convolutions of a
training step run at the precision cuDNN gives the reference.

The level-12 cells' ``conv_3x3`` op, ``ConvBR_3d(16, 16, 3, 1, 1)``, runs on entries of its own (``rag_conv3d_cc16_*``: the
same kernels on a geometry for small volumes) under ``install(..., matching_convs=True, level12_convs=True)``
(``level12_qualifies``); it stays fp32 under the TF32 flags, which have no 16 -> 16 kernels.

``qualifies(layer, x)`` -- and, with ``level12_convs``, ``level12_qualifies(layer, x)`` -- is the only routing decision;
``matching_forward`` -- bound onto ``ConvBR_3d.forward`` by ``rag_b200.network.install(..., matching_convs=True)`` -- sends
qualifying plain-tensor calls here and everything else to ``fused_stem.stem_forward`` unchanged.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _cabi, batchnorm
from .functional import _require, _stream
from .fused_stem import stem_forward

PAIRS = ((4, 4), (8, 8), (12, 12))     # the (C, O) instantiations of csrc/conv3d_cc.cu (16 -> 16 lost to cuDNN: DESIGN.md 5.10)
LEVEL12_PAIR = (16, 16)                 # the level-12 op: its own entries, rag_conv3d_cc16_* (DESIGN.md 5.10.3)
LEVEL12_MIN_VOXELS = 2 ** 17            # B*D*H*W from which the level-12 op trains faster than on cuDNN TF32 (DESIGN.md 5.10.3)
_TF32 = False                           # set by network.install(matching_tf32=...), cleared by network.uninstall()
_TF32_WGRAD = False                     # likewise, by network.install(matching_tf32_wgrad=...)
_LEVEL12 = False                        # likewise, by network.install(level12_convs=...)


def set_tf32(on: bool) -> None:
    global _TF32
    _TF32 = bool(on)


def set_tf32_wgrad(on: bool) -> None:
    global _TF32_WGRAD
    _TF32_WGRAD = bool(on)


def set_level12(on: bool) -> None:
    global _LEVEL12
    _LEVEL12 = bool(on)


def use_tf32(c: int) -> bool:
    """True when a qualifying call with C input channels runs its convolutions in TF32: ``install(..., matching_tf32=True)``
    and torch's cuDNN TF32 switch (``torch.backends.cudnn.allow_tf32``) both on, and C > 4.  At C = 4 the TF32 kernel is no
    faster than the fp32 one on the measured shapes (DESIGN.md 5.10), so 4 -> 4 stays fp32; 16 -> 16 has no TF32 kernel."""
    return _TF32 and torch.backends.cudnn.allow_tf32 and c > 4 and c != LEVEL12_PAIR[0]


def use_tf32_wgrad(c: int) -> bool:
    """True when a qualifying training call with C input channels also takes its weight gradient from the TF32 kernel:
    ``install(..., matching_tf32_wgrad=True)`` and ``use_tf32(c)``, both read at call time."""
    return _TF32_WGRAD and use_tf32(c)


def conv3d_cc_forward(x: torch.Tensor, weight: torch.Tensor, scale=None, shift=None, relu: bool = False,
                      tf32: bool = False) -> torch.Tensor:
    """out = relu?(fma(conv3d(x, weight, padding=1), scale, shift)) for weight [O,C,3,3,3]; x [B,C,D,H,W] CUDA fp32.
    scale / shift [O] (both or neither) fold an eval-mode BatchNorm into the store.  ``tf32`` runs the convolution on the
    tensor cores (``rag_conv3d_cc_tf32_fwd``), else in fp32 (``rag_conv3d_cc_fwd``; ``rag_conv3d_cc16_fwd`` for 16 -> 16)."""
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
    name = "rag_conv3d_cc_tf32_fwd" if tf32 else "rag_conv3d_cc16_fwd" if (c, o) == LEVEL12_PAIR else "rag_conv3d_cc_fwd"
    with torch.cuda.device(x.device):
        rc = getattr(L, name)(x.data_ptr(), weight.data_ptr(), scale.data_ptr() if scale is not None else None,
                              shift.data_ptr() if shift is not None else None, int(bool(relu)), out.data_ptr(),
                              b, c, o, d, h, w, _stream(x))
    _cabi.check(rc, name)
    return out


class ConvBR3dFn(torch.autograd.Function):
    """out = relu(batchnorm(conv3d(x, weight))) with gradients w.r.t. x, weight, gamma and beta, each only when wanted.

    BatchNorm with batch statistics (``batch_stats``; the running estimates updated in place when ``update_running``) or with
    the running statistics (eval-mode BatchNorm behind trainable layers).  Saved for the backward: x, the convolution output z
    and the [O,4] table (scale, shift, mean, rstd) -- the reference's own layer keeps its conv output too, so no fourth
    convolution pass is spent on recomputing z.  The backward re-evaluates the forward's own ``fma(z, scale, shift) > 0`` for
    the ReLU decision (bit-identical).  ``use_tf32``, read once in the forward, puts z and the data gradient on the TF32
    kernels; ``use_tf32_wgrad``, read with it, puts the weight gradient there too, else it is the fp32 kernel's.  16 -> 16 runs
    on the fp32 ``rag_conv3d_cc16_*`` entries."""

    @staticmethod
    def forward(ctx, x, weight, gamma, beta, running_mean, running_var, batch_stats, update_running, momentum, eps):
        ctx.tf32 = use_tf32(x.shape[1])
        ctx.tf32_wgrad = use_tf32_wgrad(x.shape[1])
        z = conv3d_cc_forward(x, weight, tf32=ctx.tf32)
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
                bwd = "rag_conv3d_cc16_bwd" if (c, o) == LEVEL12_PAIR else "rag_conv3d_cc_bwd"
                ws_bytes = L.rag_conv3d_cc_tf32_bwd_weight_workspace_bytes if ctx.tf32_wgrad else getattr(L, bwd + "_workspace_bytes")
                ws = torch.empty(int(ws_bytes(b, c, o, d, h, w)) // 4, dtype=torch.float32, device=x.device) if need_w else None
                if ctx.tf32 and gx is not None:      # TF32 data gradient; the fp32 call below then takes the weight gradient only
                    _cabi.check(L.rag_conv3d_cc_tf32_bwd_data(gz.data_ptr(), weight.data_ptr(), gx.data_ptr(), b, c, o, d, h, w, _stream(x)),
                                "rag_conv3d_cc_tf32_bwd_data")
                if ctx.tf32_wgrad and gw is not None:   # TF32 weight gradient: no fp32 call below
                    _cabi.check(L.rag_conv3d_cc_tf32_bwd_weight(gz.data_ptr(), x.data_ptr(), gw.data_ptr(), ws.data_ptr(),
                                                                b, c, o, d, h, w, _stream(x)), "rag_conv3d_cc_tf32_bwd_weight")
                gin = None if ctx.tf32 or gx is None else gx.data_ptr()
                gwp = None if ctx.tf32_wgrad or gw is None else gw.data_ptr()
                if gin is not None or gwp is not None:
                    _cabi.check(getattr(L, bwd)(gz.data_ptr(), x.data_ptr(), weight.data_ptr(), gin, gwp,
                                                ws.data_ptr() if gwp is not None else None, b, c, o, d, h, w, _stream(x)), bwd)
        return gx, gw, ggamma if need_gamma else None, gbeta if need_beta else None, None, None, None, None, None, None


def _wants_grad(layer: nn.Module, x: torch.Tensor) -> bool:
    return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in layer.parameters()))


def _layer_is(layer: nn.Module, pairs) -> bool:
    conv = getattr(layer, "conv", None)
    if not (isinstance(conv, nn.Conv3d) and conv.bias is None and conv.kernel_size == (3, 3, 3) and conv.stride == (1, 1, 1)
            and conv.padding == (1, 1, 1) and conv.dilation == (1, 1, 1) and conv.groups == 1 and conv.padding_mode == "zeros"
            and conv.weight.dtype == torch.float32 and (conv.in_channels, conv.out_channels) in pairs):
        return False
    return batchnorm.bn_relu_qualifies(layer, conv.out_channels)


def layer_qualifies(layer: nn.Module) -> bool:
    """The layer half of ``qualifies``, independent of devices: ``layer`` (a ConvBR_3d: .conv, .bn, .use_bn, .relu) is a
    Conv3d 3x3x3 / stride 1 / padding 1 / dilation 1 / groups 1, bias-free (the kernels have no bias term), zero padding,
    fp32, with (C, O) in PAIRS, followed by an affine fp32 BatchNorm3d that tracks running statistics and a ReLU."""
    return _layer_is(layer, PAIRS)


def qualifies(layer: nn.Module, x) -> bool:
    """True when ``layer(x)`` is the layer csrc/conv3d_cc.cu implements: ``layer_qualifies(layer)`` with the weight on CUDA,
    and x a CUDA fp32 [B,C,D,H,W] tensor on the weight's device with W % 4 == 0 and within the kernels' limits.  Whenever
    batch statistics are used or a gradient is wanted, also the limits of the BatchNorm kernels (csrc/bn3d.cu):
    O <= 32, D >= 3, 8 <= W <= 1016."""
    return layer_qualifies(layer) and _input_qualifies(layer, x)


def level12_qualifies(layer: nn.Module, x) -> bool:
    """``qualifies`` for the level-12 op: the same layer, BatchNorm / ReLU and input clauses and limits, with (C, O) =
    LEVEL12_PAIR -- the layer the ``rag_conv3d_cc16_*`` entries implement -- for training calls (batch statistics or a
    gradient) of at least LEVEL12_MIN_VOXELS voxels.  The eval forward, and training below that size, are faster on cuDNN
    TF32 at the measured shapes (DESIGN.md 5.10.3), so they stay there."""
    if not (_layer_is(layer, (LEVEL12_PAIR,)) and _input_qualifies(layer, x)):
        return False
    b, _, d, h, w = x.shape
    return (layer.bn.training or _wants_grad(layer, x)) and b * d * h * w >= LEVEL12_MIN_VOXELS


def _input_qualifies(layer: nn.Module, x) -> bool:
    if not layer.conv.weight.is_cuda:
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
        return conv3d_cc_forward(x, layer.conv.weight, *batchnorm.eval_fold(layer.bn), relu=True, tf32=use_tf32(x.shape[1]))
    return batchnorm.apply(ConvBR3dFn, layer.bn, x.contiguous(), layer.conv.weight)


def matching_forward(self, x):
    """Replacement for ConvBR_3d.forward (operations_3d.py:41-47) under ``install(..., matching_convs=True)``."""
    if isinstance(x, torch.Tensor) and (qualifies(self, x) or _LEVEL12 and level12_qualifies(self, x)):
        return convbr_forward(self, x)
    return stem_forward(self, x)
