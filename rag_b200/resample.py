"""A drop-in ``torch.nn.functional.interpolate`` whose linear modes run on the hand-written kernels: the resampling inside the
growable network's cells (``Cell_2d`` / ``Cell_3d``, which move between levels 3, 6 and 12 with ``F.interpolate``).

``interpolate`` has ``F.interpolate``'s signature, defaults and output shape.  A call goes to ``csrc/trilinear.cu`` when

* the input is a contiguous (NCHW / NCDHW, not channels_last) CUDA fp32 tensor and not empty,
* it is 5-D ``trilinear`` (``rag_trilinear_resize_fwd/bwd``) or 4-D ``bilinear`` (``rag_bilinear_resize_fwd/bwd``), without
  ``antialias``, and its sizes are within the kernels' limits,
* the source-index scale ATen would use is the one the kernels compute: in/out (or (in-1)/(out-1) with
  ``align_corners=True``).  That holds for an explicit ``size``, for ``align_corners=True`` and for
  ``recompute_scale_factor=True``; a ``scale_factor`` with ``align_corners=False`` makes ATen use 1/scale_factor instead.

Every other call is ``F.interpolate`` itself, unchanged.  The kernels use PyTorch's fp32 index arithmetic; their backward
gathers in a fixed order, so it is bitwise repeatable and needs neither atomics nor ``torch.use_deterministic_algorithms``.
Under that mode torch itself sends CUDA linear-mode calls to a decomposition whose backward is a sorted ``index_put_``;
these kernels replace it.

``install(..., resample=True)`` (rag_b200.network) binds ``FProxy()`` as ``F`` in the reference's modules, the analogue of
``upsample.NNProxy`` for ``nn``.
"""
import math
from typing import Optional

import torch
import torch.nn.functional as F

from .upsample import TrilinearResizeFn, _resize
from .functional import _require

_VOXELS = 1 << 31        # check_tri: each volume has fewer than 2^31 voxels
_TABLES = 160 * 1024     # check_tri: per-axis tables of the backward within 160 KB of shared memory


def _within_limits(bc: int, si, so) -> bool:
    """csrc/trilinear.cu check_tri's shape limits (a 2-D resize is a 3-D one with Di = Do = 1)."""
    if len(si) == 2:
        si, so = (1,) + tuple(si), (1,) + tuple(so)
    if bc <= 0 or bc >= _VOXELS or min(si) <= 0 or min(so) <= 0:
        return False
    if math.prod(si) >= _VOXELS or math.prod(so) >= _VOXELS:
        return False
    return sum(so) * 8 + (sum(si) + 3) * 4 <= _TABLES


def _is_int(v) -> bool:
    return isinstance(v, int) and not isinstance(v, bool)


def output_size(input: torch.Tensor, size=None, scale_factor=None, recompute_scale_factor=None):
    """The spatial output size ``F.interpolate`` produces for these arguments, or None where it would raise or where this
    module does not follow it (non-integer sizes, non-numeric scale factors)."""
    n = input.dim() - 2
    if n < 1 or (size is None) == (scale_factor is None):
        return None
    if size is not None:
        if recompute_scale_factor:
            return None
        out = tuple(size) if isinstance(size, (list, tuple)) else (size,) * n
        return out if len(out) == n and all(_is_int(s) for s in out) else None
    sf = tuple(scale_factor) if isinstance(scale_factor, (list, tuple)) else (scale_factor,) * n
    if len(sf) != n or not all(isinstance(f, (int, float)) and not isinstance(f, bool) for f in sf):
        return None
    return tuple(int(math.floor(float(s) * float(f))) for s, f in zip(input.shape[2:], sf))


def plan(input, size=None, scale_factor=None, mode="nearest", align_corners=None, recompute_scale_factor=None,
         antialias=False):
    """The routing decision: (output size, align_corners) when the call goes to the kernels, else None."""
    if not isinstance(input, torch.Tensor) or antialias:
        return None
    if not ((input.dim() == 5 and mode == "trilinear") or (input.dim() == 4 and mode == "bilinear")):
        return None
    if not (input.is_cuda and input.dtype == torch.float32 and input.is_contiguous()) or input.numel() == 0:
        return None
    ac = bool(align_corners) if align_corners is not None else False
    if scale_factor is not None and not ac and not recompute_scale_factor:
        return None                  # ATen's source-index scale would be 1/scale_factor, not in/out
    out = output_size(input, size, scale_factor, recompute_scale_factor)
    if out is None or not _within_limits(input.shape[0] * input.shape[1], tuple(input.shape[2:]), out):
        return None
    return out, ac


class BilinearResizeFn(torch.autograd.Function):
    """The 2-D counterpart of ``upsample.TrilinearResizeFn``: [B,C,H,W] -> [B,C,Ho,Wo]."""

    @staticmethod
    def forward(ctx, x, size, align_corners):
        _require(x, "x")
        if x.dim() != 4:
            raise RuntimeError(f"rag_b200: bilinear resize wants a [B,C,H,W] tensor, got {tuple(x.shape)}")
        x = x.contiguous()
        size = tuple(int(s) for s in size)
        ctx.in_size, ctx.out_size, ctx.align = tuple(x.shape[2:]), size, bool(align_corners)
        ctx.bc = tuple(x.shape[:2])
        return _resize("rag_bilinear_resize_fwd", x, ctx.bc + size, ctx.in_size, size, align_corners)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g):
        g = g.contiguous()
        gin = _resize("rag_bilinear_resize_bwd", g, ctx.bc + ctx.in_size, ctx.in_size, ctx.out_size, ctx.align)
        return gin, None, None


def bilinear_resize(x: torch.Tensor, size, align_corners: bool = True) -> torch.Tensor:
    """F.interpolate(x, size, mode='bilinear', align_corners=...) for CUDA fp32 [B,C,H,W]."""
    return BilinearResizeFn.apply(x, size, align_corners)


def interpolate(input: torch.Tensor, size: Optional[int] = None, scale_factor: Optional[list[float]] = None,
                mode: str = "nearest", align_corners: Optional[bool] = None, recompute_scale_factor: Optional[bool] = None,
                antialias: bool = False) -> torch.Tensor:
    """``torch.nn.functional.interpolate``; see the module docstring for the calls that take the kernels."""
    p = plan(input, size, scale_factor, mode, align_corners, recompute_scale_factor, antialias)
    if p is None:
        return F.interpolate(input, size, scale_factor, mode, align_corners, recompute_scale_factor, antialias)
    out, ac = p
    fn = TrilinearResizeFn if input.dim() == 5 else BilinearResizeFn
    return fn.apply(input, out, ac)


class FProxy:
    """What ``install(resample=True)`` binds as ``F`` in the reference's modules: ``torch.nn.functional`` with
    ``interpolate`` replaced."""

    interpolate = staticmethod(interpolate)

    def __getattr__(self, name):
        return getattr(F, name)
