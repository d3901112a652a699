"""Photometric training loss: SSIM and L1 on fused sm_100a kernels (include/bsplat.h: bsplat_ssim_fwd / _bwd).

``ssim(img, target)`` is 3DGS's ``ssim`` (11x11 Gaussian window with sigma 1.5, per channel, zero padding 5,
C1 = 0.01^2, C2 = 0.03^2, mean over every value) for one (H, W, C) image, C in 1..4 -- the layout
``render_gaussians[_diff]`` returns.  ``l1_dssim_loss(img, target, lambda_dssim=0.2)`` is the 3DGS training loss
``(1 - lambda) L1 + lambda (1 - SSIM)``.  Both come from one forward and one backward launch chain that computes the
two means together; gradients flow to ``img`` only (a ``target`` that requires grad is rejected).
"""
from __future__ import annotations

import torch

from . import _lib


def _check_pair(img: torch.Tensor, target: torch.Tensor):
    if not isinstance(img, torch.Tensor) or not isinstance(target, torch.Tensor):
        raise TypeError("img and target must be torch.Tensors")
    if target.requires_grad:
        raise ValueError("target must not require grad: the loss gives no gradient to the target")
    if img.dim() != 3 or img.shape != target.shape:
        raise ValueError(f"img and target must both be (H, W, C); got {tuple(img.shape)} and {tuple(target.shape)}")
    H, W, C = img.shape
    if not 1 <= C <= 4 or H < 1 or W < 1:
        raise ValueError(f"expected H, W >= 1 and 1 <= C <= 4, got {(H, W, C)}")
    if img.device != target.device:
        raise ValueError(f"img and target are on different devices ({img.device}, {target.device})")
    return H, W, C


class _SsimL1Fn(torch.autograd.Function):
    """(mean SSIM, mean |img - target|) with a backward pass to img (bsplat_ssim_fwd / bsplat_ssim_bwd)."""

    @staticmethod
    def forward(ctx, img, target):
        H, W, C = _check_pair(img, target)
        dev = img.device
        L = _lib.require_device(dev)
        x = _lib.as_f32(img, "img")
        y = _lib.as_f32(target, "target")
        out2 = torch.empty((2,), dtype=torch.float32, device=dev)
        maps = torch.empty((3, H, W, C), dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        ws = _lib.workspace.get(dev, "ssim", L.bsplat_ssim_workspace_bytes(H, W, C))
        with torch.cuda.device(dev):
            rc = L.bsplat_ssim_fwd(H, W, C, _lib.ptr(x), _lib.ptr(y), _lib.ptr(out2), _lib.ptr(maps), _lib.ptr(ws),
                                   ws.numel(), None, _lib.stream_ptr(dev))
        _lib.check(rc, "bsplat_ssim_fwd")
        if maps is not None:
            ctx.save_for_backward(x, y, maps)
        return out2[0], out2[1]

    @staticmethod
    def backward(ctx, g_ssim, g_l1):
        x, y, maps = ctx.saved_tensors
        dev = x.device
        L = _lib.require_device(dev)
        H, W, C = x.shape
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        v_out2 = torch.stack([zero if g_ssim is None else g_ssim.to(torch.float32).reshape(()),
                              zero if g_l1 is None else g_l1.to(torch.float32).reshape(())])
        v_img = torch.empty_like(x)
        with torch.cuda.device(dev):
            rc = L.bsplat_ssim_bwd(H, W, C, _lib.ptr(x), _lib.ptr(y), _lib.ptr(maps), _lib.ptr(v_out2),
                                   _lib.ptr(v_img), _lib.stream_ptr(dev))
        _lib.check(rc, "bsplat_ssim_bwd")
        return v_img, None


def ssim_l1(img: torch.Tensor, target: torch.Tensor):
    """(mean SSIM, mean L1) of one image pair as two 0-d tensors, both differentiable with respect to ``img``."""
    return _SsimL1Fn.apply(img, target)


def ssim(img: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """Mean SSIM of two (H, W, C) images (3DGS's definition) as a 0-d tensor, differentiable with respect to img."""
    return ssim_l1(img, target)[0]


def l1_dssim_loss(img: torch.Tensor, target: torch.Tensor, lambda_dssim: float = 0.2) -> torch.Tensor:
    """3DGS's training loss ``(1 - lambda_dssim) * mean|img - target| + lambda_dssim * (1 - SSIM(img, target))``."""
    s, l1 = ssim_l1(img, target)
    return (1.0 - lambda_dssim) * l1 + lambda_dssim * (1.0 - s)
