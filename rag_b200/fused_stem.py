"""Fused cost volume + first Matching-Net layer (SURVEY.md section 8f rank 1), inference AND training.

The reference builds the [B,2C,Df,Hf,Wf] volume (rag_model.py:375-383) and immediately feeds it to
``self.stem3d0[i]`` = ConvBR_3d(2C->C, 3x3x3) (rag_model.py:341, operations_3d.py:31-47).  Because the
volume is a masked/shifted broadcast of two 2-D feature maps, that 3-D convolution collapses to two 2-D
maps broadcast-added along the disparity axis (csrc/cv_stem.cu): the 2.5 GB volume is never written and
the layer's 51 GFLOP/pair become ~10 FMA per output.

Drop-in mechanism: ``cost_volume_lazy`` returns a ``VirtualCostVolume`` (just the two feature tensors);
``stem_forward`` -- bound onto ``ConvBR_3d.forward`` by ``rag_b200.network.install`` -- recognises it and
runs the fused kernel (conv + folded BatchNorm + ReLU).  With autograd the layer runs as ``FusedStemFn``: batch
statistics from the collapsed row maps, the forward kernel, and a backward that rebuilds the gradient at the
convolution output on the fly and reduces it along the disparity axis (csrc/cv_stem_train.cu) -- neither the
volume, nor its gradient, nor the convolution output are ever held.  Whenever the fusion does not apply (a
different conv geometry, no BatchNorm / ReLU, affine-free BatchNorm) the volume is materialised with the
cost-volume kernel and the layer runs as in the reference.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi, batchnorm
from .functional import _require, _stream, cost_volume
from .last_conv import conv_forward


class VirtualCostVolume:
    """The concatenation volume of (x, y), not yet materialised."""

    def __init__(self, x: torch.Tensor, y: torch.Tensor, maxdisp: int):
        self.x, self.y, self.maxdisp = x, y, maxdisp

    @property
    def shape(self):
        b, c, hf, wf = self.x.shape
        return (b, 2 * c, int(self.maxdisp / 3), hf, wf)

    def size(self):
        return torch.Size(self.shape)

    def materialize(self) -> torch.Tensor:
        return cost_volume(self.x, self.y, self.maxdisp)


def _stem_workspace(L, c, o, device):
    """Caller-owned buffer for the regrouped weights (rag_cv_stem_workspace_bytes): fresh per launch from the caching
    allocator, so it is stream-ordered and never shared between launches."""
    n = int(L.rag_cv_stem_workspace_bytes(c, o))
    return torch.empty(n // 4, dtype=torch.float32, device=device) if n else None


def cv_stem_forward(x, y, weight, scale=None, shift=None, relu=False, maxdisp=192, variant=None) -> torch.Tensor:
    """out = relu?(scale * conv3d(cost_volume(x, y), weight, padding=1) + shift), fp32, volume never built."""
    _require(x, "x"), _require(y, "y"), _require(weight, "weight")
    if x.dim() != 4 or x.shape != y.shape:
        raise RuntimeError("rag_b200: fused stem wants x,y of identical [B,C,Hf,Wf] shape")
    b, c, hf, wf = x.shape
    o = weight.shape[0]
    if tuple(weight.shape) != (o, 2 * c, 3, 3, 3):
        raise RuntimeError(f"rag_b200: fused stem wants a [O,{2 * c},3,3,3] weight, got {tuple(weight.shape)}")
    df = int(maxdisp / 3)
    x, y, weight = x.contiguous(), y.contiguous(), weight.contiguous()
    out = torch.empty((b, o, df, hf, wf), dtype=torch.float32, device=x.device)
    if out.numel() == 0:
        return out
    scale = scale.contiguous() if scale is not None else None
    shift = shift.contiguous() if shift is not None else None
    sp = scale.data_ptr() if scale is not None else None
    hp = shift.data_ptr() if shift is not None else None
    L = _cabi.lib()
    with torch.cuda.device(x.device):
        ws = _stem_workspace(L, c, o, x.device)
        wp = ws.data_ptr() if ws is not None else None
        if variant is None:
            rc = L.rag_cv_stem_fwd(x.data_ptr(), y.data_ptr(), weight.data_ptr(), sp, hp, int(relu), out.data_ptr(), b, c, o, df, hf, wf, wp, _stream(x))
        else:
            rc = L.rag_cv_stem_fwd_v(x.data_ptr(), y.data_ptr(), weight.data_ptr(), sp, hp, int(relu), out.data_ptr(), b, c, o, df, hf, wf, wp, variant, _stream(x))
    _cabi.check(rc, "rag_cv_stem_fwd")
    return out


def cv_stem_batch_stats(x, y, weight, maxdisp=192):
    """Per-channel batch (mean, biased variance, count) of conv3d(cost_volume(x, y), weight, padding=1) -- what a
    training-mode BatchNorm3d after the stem normalises with -- computed from the collapsed row maps: neither the
    volume nor the convolution output is formed (csrc/cv_stem.cu, MOMENTS; DESIGN.md section 10)."""
    _require(x, "x"), _require(y, "y"), _require(weight, "weight")
    if x.dim() != 4 or x.shape != y.shape:
        raise RuntimeError("rag_b200: fused stem wants x,y of identical [B,C,Hf,Wf] shape")
    b, c, hf, wf = x.shape
    o = weight.shape[0]
    if tuple(weight.shape) != (o, 2 * c, 3, 3, 3):
        raise RuntimeError(f"rag_b200: fused stem wants a [O,{2 * c},3,3,3] weight, got {tuple(weight.shape)}")
    df = int(maxdisp / 3)
    x, y, weight = x.contiguous(), y.contiguous(), weight.contiguous()
    rows = torch.empty((b, hf, o, 2), dtype=torch.float64, device=x.device)
    L = _cabi.lib()
    with torch.cuda.device(x.device):
        ws = _stem_workspace(L, c, o, x.device)
        rc = L.rag_cv_stem_moments(x.data_ptr(), y.data_ptr(), weight.data_ptr(), rows.data_ptr(), b, c, o, df, hf, wf,
                                   ws.data_ptr() if ws is not None else None, _stream(x))
    _cabi.check(rc, "rag_cv_stem_moments")
    s = rows.sum(dim=(0, 1))                      # fixed-order fp64 reduction of B*Hf row pairs per channel
    n = b * df * hf * wf
    mean = s[:, 0] / n
    return mean, s[:, 1] / n - mean * mean, n


class FusedStemFn(torch.autograd.Function):
    """out = relu(batchnorm(conv3d(cost_volume(x, y), weight))) with gradients w.r.t. x, y, weight, gamma, beta.

    Forward: the convolution output z from the fused kernel (the volume is never built), then the BatchNorm + ReLU of
    ``batchnorm.forward`` IN PLACE.  Saved for the backward: the two feature maps, the weight and the [O,4] table -- no
    [B,*,Df,Hf,Wf] tensor: z is RECOMPUTED by the forward kernel inside ``backward`` into a temporary, and the backward kernels
    re-evaluate the forward's own expression ``fma(z, scale, shift) > 0`` for the ReLU decision (bit-identical)."""

    @staticmethod
    def forward(ctx, x, y, weight, maxdisp, gamma, beta, running_mean, running_var, batch_stats, update_running, momentum, eps):
        z = cv_stem_forward(x, y, weight, None, None, False, maxdisp)
        bn = batchnorm.forward(z, z, gamma, beta, running_mean, running_var, batch_stats, update_running, momentum, eps)
        ctx.save_for_backward(x, y, weight, bn)
        ctx.batch_stats, ctx.maxdisp = bool(batch_stats), maxdisp
        return z                                      # z now holds the layer output

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        x, y, weight, bn = ctx.saved_tensors
        g = g.contiguous()
        b, c, hf, wf = x.shape
        o, df = weight.shape[0], g.shape[2]
        L = _cabi.lib()
        need_in = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        need_w = ctx.needs_input_grad[2]
        with torch.cuda.device(x.device):
            z = cv_stem_forward(x, y, weight, None, None, False, ctx.maxdisp)           # temporary: the convolution output again
            consts, ggamma, gbeta, _ = batchnorm.backward(g, z, bn, ctx.batch_stats, want_gz=False)
            gx = gy = gw = None
            if need_in or need_w:
                ws = torch.empty(int(L.rag_cv_stem_bwd_workspace_bytes(b, c, o, hf, wf)) // 4, dtype=torch.float32, device=x.device)
                if need_in:
                    gx, gy = torch.empty_like(x), torch.empty_like(y)
                gw = torch.empty_like(weight) if need_w else None
                rc = L.rag_cv_stem_bwd(g.data_ptr(), z.data_ptr(), consts.data_ptr(), x.data_ptr(), y.data_ptr(), weight.data_ptr(),
                                       gx.data_ptr() if gx is not None else None, gy.data_ptr() if gy is not None else None,
                                       gw.data_ptr() if gw is not None else None, ws.data_ptr(), b, c, o, df, hf, wf, _stream(x))
                _cabi.check(rc, "rag_cv_stem_bwd")
        return (gx if ctx.needs_input_grad[0] else None, gy if ctx.needs_input_grad[1] else None, gw, None,
                ggamma if ctx.needs_input_grad[4] else None, gbeta if ctx.needs_input_grad[5] else None,
                None, None, None, None, None, None)


def _train_fusable(self, vol: VirtualCostVolume) -> bool:
    """The layer csrc/cv_stem_train.cu (the convolution) and csrc/bn3d.cu (its BatchNorm) differentiate: Conv3d(2*12 -> O <= 32,
    3x3x3) + affine BatchNorm3d + ReLU on a volume with Wf % 4 == 0, 8 <= Wf <= 1016 and Df >= 3."""
    bn = self.bn
    b, c, hf, wf = vol.x.shape
    return (self.use_bn and bool(self.relu) and isinstance(bn, nn.BatchNorm3d) and bn.affine and bn.weight.dtype == torch.float32
            and (bn.training or bn.track_running_stats) and c == 12 and self.conv.out_channels <= 32
            and wf % 4 == 0 and 8 <= wf <= 1016 and int(vol.maxdisp / 3) >= 3 and hf <= 65535 and b <= 32767)


def stem_train_forward(self, vol: VirtualCostVolume) -> torch.Tensor:
    """ConvBR_3d.forward on a VirtualCostVolume with autograd (train() or eval() BatchNorm), fused.  Updates the running
    statistics exactly like nn.BatchNorm3d does in train() (momentum / cumulative average, unbiased variance)."""
    return batchnorm.apply(FusedStemFn, self.bn, vol.x.contiguous(), vol.y.contiguous(), self.conv.weight, vol.maxdisp)


def _fusable(conv: nn.Conv3d, vol: VirtualCostVolume) -> bool:
    return (isinstance(conv, nn.Conv3d) and conv.bias is None and conv.kernel_size == (3, 3, 3) and conv.stride == (1, 1, 1)
            and conv.padding == (1, 1, 1) and conv.dilation == (1, 1, 1) and conv.groups == 1
            and conv.in_channels == 2 * vol.x.shape[1] and conv.weight.dtype == torch.float32)


def stem_forward(self, x):
    """Replacement for ConvBR_3d.forward (operations_3d.py:41-47).  ``self`` has .conv, .bn, .use_bn, .relu."""
    if not isinstance(x, VirtualCostVolume):
        x = conv_forward(self.conv, x)     # last_3_3d (C -> 1, inference) takes the hand-written kernel, the rest cuDNN
        if self.use_bn:
            x = self.bn(x)
        if self.relu:
            x = F.relu(x, inplace=True)
        return x
    needs_grad = torch.is_grad_enabled() and (x.x.requires_grad or x.y.requires_grad
                                              or any(p.requires_grad for p in self.parameters()))
    bn_batch_stats = self.use_bn and (self.bn.training or not self.bn.track_running_stats)
    if not _fusable(self.conv, x):
        return stem_forward(self, x.materialize())          # the reference's path on the materialised volume
    if needs_grad:
        if _train_fusable(self, x):
            return stem_train_forward(self, x)               # fused forward + volume-free backward (csrc/cv_stem_train.cu)
        return stem_forward(self, x.materialize())
    if bn_batch_stats:                                       # conv fused, BatchNorm with batch statistics by torch
        out = cv_stem_forward(x.x, x.y, self.conv.weight, maxdisp=x.maxdisp)
        out = self.bn(out)
        return F.relu(out, inplace=True) if self.relu else out
    scale, shift = batchnorm.eval_fold(self.bn) if self.use_bn else (None, None)
    return cv_stem_forward(x.x, x.y, self.conv.weight, scale, shift, bool(self.relu), x.maxdisp)


def cost_volume_lazy(x: torch.Tensor, y: torch.Tensor, maxdisp: int = 192):
    """What the patched forwards hand to ``matching``: a VirtualCostVolume when the first layer has been made
    fusion-aware (``install(..., fuse_stem=True)``), else the materialised volume."""
    return VirtualCostVolume(x, y, maxdisp)
