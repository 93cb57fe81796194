"""A stand-in for the self-supervised variant's loss (the reference's ``src_self/models/loss.py``, unread: SURVEY.md row 13
records it as "warp + SSIM/L1 + smoothness, consumes ``disp_est``").  Like the reference's modules it is a module object with
its own ``F``, so ``install(grid_sample=True, grid_sample_modules=(loss,))`` can bind into it.

``loss.photometric(left, right, disp)``: the right image warped to the left view by the predicted disparity (``F.grid_sample``,
bilinear, zeros padding, align_corners=True; x shifted left by ``disp``, y the row), then 0.85 * SSIM (3x3, unpadded
``avg_pool2d``) + 0.15 * L1 between the warp and the left image, plus 0.1 * an edge-aware smoothness of the disparity.
"""
import types

_LOSS = '''
import torch
import torch.nn.functional as F


def warp(right, disp):
    """right [B,C,H,W] sampled at (x - disp, y): the left view synthesised from the right image."""
    b, _, h, w = right.shape
    xs = torch.arange(w, device=disp.device, dtype=disp.dtype).view(1, 1, w)
    ys = torch.arange(h, device=disp.device, dtype=disp.dtype).view(1, h, 1)
    gx = 2 * (xs - disp) / (w - 1) - 1
    gy = (2 * ys / (h - 1) - 1).expand(b, h, w)
    return F.grid_sample(right, torch.stack([gx, gy], -1), mode="bilinear", padding_mode="zeros", align_corners=True)


def ssim(x, y):
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    mx, my = F.avg_pool2d(x, 3, 1), F.avg_pool2d(y, 3, 1)
    sx = F.avg_pool2d(x * x, 3, 1) - mx * mx
    sy = F.avg_pool2d(y * y, 3, 1) - my * my
    sxy = F.avg_pool2d(x * y, 3, 1) - mx * my
    return ((2 * mx * my + c1) * (2 * sxy + c2)) / ((mx * mx + my * my + c1) * (sx + sy + c2))


def smoothness(disp, img):
    d = disp.unsqueeze(1)
    ddx, ddy = d[:, :, :, 1:] - d[:, :, :, :-1], d[:, :, 1:, :] - d[:, :, :-1, :]
    idx = (img[:, :, :, 1:] - img[:, :, :, :-1]).abs().mean(1, keepdim=True)
    idy = (img[:, :, 1:, :] - img[:, :, :-1, :]).abs().mean(1, keepdim=True)
    return (ddx.abs() * torch.exp(-idx)).mean() + (ddy.abs() * torch.exp(-idy)).mean()


def photometric(left, right, disp):
    est = warp(right, disp)
    return (0.85 * ((1 - ssim(est, left)) / 2).mean() + 0.15 * (est - left).abs().mean()
            + 0.1 * smoothness(disp, left))
'''


def loss_module():
    """A fresh ``models.loss`` module object (``import torch.nn.functional as F`` at its top, as the reference's modules)."""
    m = types.ModuleType("models.loss")
    exec(compile(_LOSS, "<stand-in models.loss>", "exec"), m.__dict__)
    return m
