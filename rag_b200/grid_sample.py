"""A drop-in ``torch.nn.functional.grid_sample`` whose 4-D bilinear calls run on the hand-written kernels: the warp with which a
self-supervised stereo loss synthesises the left view from the right image and the predicted disparity (the reference's
``src_self/models/loss.py``; that its warp is ``F.grid_sample`` is inferred, the loss itself is unread).

``grid_sample`` has ``F.grid_sample``'s signature and defaults.  A call goes to ``csrc/grid_sample.cu`` when ``routes`` says so:

* ``mode='bilinear'``, ``padding_mode`` ``'zeros'`` or ``'border'``;
* ``input`` [N,C,Hi,Wi] and ``grid`` [N,Ho,Wo,2], both contiguous (NCHW, not channels_last) CUDA fp32 on one device, not empty;
* the sizes are within the kernels' limits (every flat index and 4*N*Ho*Wo below 2^31).

Every other call is ``F.grid_sample`` itself, unchanged: nearest, bicubic, reflection padding, 5-D, fp64, channels_last,
empty tensors, out-of-limit sizes.  ``align_corners=None`` warns as ``F.grid_sample`` does and means False.

The forward and the grid gradient restate ATen's fp32 arithmetic.  The input gradient sums in a fixed order (ascending sample,
then corner nw, ne, sw, se) instead of ATen's atomicAdd arrival order, so it is bitwise repeatable and runs under
``torch.use_deterministic_algorithms(True)``, where ATen's backward raises.  (For zeros padding with ``align_corners=True``
torch itself sends CUDA calls to cuDNN's sampler rather than ATen's kernel; the drop-in follows ATen's kernel.  On finite grids the two
agree within rounding; for a NaN grid value cuDNN's sampler returns NaN where ATen's kernel and the drop-in return 0.)

``install(..., grid_sample=True, grid_sample_modules=(...))`` (rag_b200.network) binds ``GridSampleProxy(module.F)`` as ``F`` in
each listed module.
"""
import warnings
from typing import Optional

import torch
import torch.nn.functional as F

from . import _cabi
from .functional import _require, _stream

_LIMIT = 1 << 31
_PADDING = {"zeros": 0, "border": 1}


def _within_limits(n: int, c: int, hi: int, wi: int, ho: int, wo: int) -> bool:
    """csrc/grid_sample.cu gs_check_shape."""
    if min(n, c, hi, wi, ho, wo) <= 0:
        return False
    s, p = n * ho * wo, n * hi * wi
    return 4 * s < _LIMIT and p < _LIMIT and c * p < _LIMIT and c * s < _LIMIT


def routes(input, grid, mode: str = "bilinear", padding_mode: str = "zeros", align_corners: Optional[bool] = None) -> bool:
    """The routing decision: True when the call goes to the kernels."""
    if not isinstance(input, torch.Tensor) or not isinstance(grid, torch.Tensor):
        return False
    if mode != "bilinear" or padding_mode not in _PADDING or input.dim() != 4 or grid.dim() != 4:
        return False
    for t in (input, grid):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            return False
    if input.device != grid.device:
        return False
    n, c, hi, wi = input.shape
    gn, ho, wo, two = grid.shape
    return gn == n and two == 2 and _within_limits(n, c, hi, wi, ho, wo)


class GridSampleFn(torch.autograd.Function):
    """F.grid_sample(input, grid, 'bilinear', padding_mode, align_corners) on routed arguments."""

    @staticmethod
    def forward(ctx, input, grid, padding_mode, align_corners):
        _require(input, "input"), _require(grid, "grid")
        n, c, hi, wi = input.shape
        _, ho, wo, _ = grid.shape
        ctx.args = (n, c, hi, wi, ho, wo, _PADDING[padding_mode], int(bool(align_corners)))
        out = torch.empty((n, c, ho, wo), dtype=torch.float32, device=input.device)
        with torch.cuda.device(input.device):
            rc = _cabi.lib().rag_grid_sample_fwd(input.data_ptr(), grid.data_ptr(), out.data_ptr(), *ctx.args, _stream(input))
        _cabi.check(rc, "rag_grid_sample_fwd")
        ctx.save_for_backward(input, grid)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        input, grid = ctx.saved_tensors
        want_in, want_grid = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (want_in or want_grid):
            return None, None, None, None
        gout = gout.contiguous()
        n, c, hi, wi, ho, wo = ctx.args[:6]
        L = _cabi.lib()
        gin = torch.empty_like(input) if want_in else None
        ggrid = torch.empty_like(grid) if want_grid else None
        ws, nbytes = None, 0
        if want_in:
            nbytes = L.rag_grid_sample_bwd_workspace_bytes(n, c, hi, wi, ho, wo)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=input.device)
        with torch.cuda.device(input.device):
            rc = L.rag_grid_sample_bwd(gout.data_ptr(), input.data_ptr(), grid.data_ptr(),
                                       gin.data_ptr() if want_in else None, ggrid.data_ptr() if want_grid else None,
                                       ws.data_ptr() if want_in else None, nbytes, *ctx.args, _stream(gout))
        _cabi.check(rc, "rag_grid_sample_bwd")
        return gin, ggrid, None, None


def grid_sample(input: torch.Tensor, grid: torch.Tensor, mode: str = "bilinear", padding_mode: str = "zeros",
                align_corners: Optional[bool] = None) -> torch.Tensor:
    """``torch.nn.functional.grid_sample``; see the module docstring for the calls that take the kernels."""
    if not routes(input, grid, mode, padding_mode, align_corners):
        return F.grid_sample(input, grid, mode, padding_mode, align_corners)
    if align_corners is None:
        warnings.warn(
            "Default grid_sample and affine_grid behavior has changed "
            "to align_corners=False since 1.3.0. Please specify "
            "align_corners=True if the old behavior is desired. "
            "See the documentation of grid_sample for details.",
            stacklevel=2,
        )
        align_corners = False
    return GridSampleFn.apply(input, grid, padding_mode, align_corners)


class GridSampleProxy:
    """What ``install(grid_sample=True)`` binds as ``F`` in a module: ``base`` (the module's ``F`` before, which may itself be
    ``resample.FProxy``) with ``grid_sample`` replaced."""

    grid_sample = staticmethod(grid_sample)

    def __init__(self, base):
        self.base = base

    def __getattr__(self, name):
        return getattr(self.base, name)
