"""Spherical-harmonics colours (additive: the reference has a placeholder, render.py:82-87).

``eval_sh(sh_degree, sh_coeffs[N, K, 3], means3d, camera) -> colors[N, 3]`` with the standard 3DGS convention
(view direction = normalize(mean - camera position), +0.5 offset, clamp at 0); include/bsplat.h: bsplat_sh_eval.
``eval_sh_diff`` is the same with a backward pass (bsplat_sh_bwd).
"""
from __future__ import annotations

from ctypes import byref, c_float

import torch

from . import _lib
from .utils import Camera


def camera_position(camera: Camera) -> torch.Tensor:
    """World-space camera centre -R^T T of a world->camera pose (CPU tensor, 3 floats)."""
    R = camera.R.detach().to("cpu", torch.float64)
    T = camera.T.detach().to("cpu", torch.float64)
    return (-(R.t() @ T)).to(torch.float32)


def eval_sh(sh_degree: int, sh_coeffs: torch.Tensor, means3d: torch.Tensor, camera: Camera) -> torch.Tensor:
    if sh_coeffs.dim() != 3 or sh_coeffs.shape[-1] != 3:
        raise ValueError("sh_coeffs must be (N, K, 3)")
    N, K, _ = sh_coeffs.shape
    if not 0 <= int(sh_degree) <= 3 or K < (int(sh_degree) + 1) ** 2:
        raise ValueError(f"sh_degree {sh_degree} needs at least {(int(sh_degree) + 1) ** 2} coefficients, got {K}")
    dev = sh_coeffs.device
    L = _lib.require_device(dev)
    coeffs = _lib.as_f32(sh_coeffs, "sh_coeffs")
    means3d = _lib.as_f32(means3d, "means3d")
    if means3d.shape != (N, 3):
        raise ValueError("means3d must be (N, 3)")
    colors = torch.empty((N, 3), dtype=torch.float32, device=dev)
    pos = camera_position(camera)
    cpos = (c_float * 3)(float(pos[0]), float(pos[1]), float(pos[2]))
    with torch.cuda.device(dev):
        rc = L.bsplat_sh_eval(N, int(sh_degree), K, _lib.ptr(coeffs), _lib.ptr(means3d), byref(cpos), _lib.ptr(colors),
                              _lib.stream_ptr(dev))
    _lib.check(rc, "bsplat_sh_eval")
    return colors


class _ShFn(torch.autograd.Function):
    """SH colours with a backward pass (bsplat_sh_eval / bsplat_sh_bwd)."""

    @staticmethod
    def forward(ctx, sh_degree, sh_coeffs, means3d, camera):
        colors = eval_sh(sh_degree, sh_coeffs, means3d, camera)
        ctx.save_for_backward(_lib.as_f32(sh_coeffs, "sh_coeffs"), _lib.as_f32(means3d, "means3d"))
        ctx.sh_degree, ctx.camera = int(sh_degree), camera
        return colors

    @staticmethod
    def backward(ctx, v_colors):
        coeffs, means3d = ctx.saved_tensors
        dev = coeffs.device
        L = _lib.require_device(dev)
        N, K, _ = coeffs.shape
        v_colors = _lib.as_f32(v_colors, "v_colors")
        v_coeffs = torch.empty_like(coeffs)
        v_means3d = torch.empty((N, 3), dtype=torch.float32, device=dev) if ctx.needs_input_grad[2] else None
        pos = camera_position(ctx.camera)
        cpos = (c_float * 3)(float(pos[0]), float(pos[1]), float(pos[2]))
        with torch.cuda.device(dev):
            rc = L.bsplat_sh_bwd(N, ctx.sh_degree, K, _lib.ptr(coeffs), _lib.ptr(means3d), byref(cpos),
                                 _lib.ptr(v_colors), _lib.ptr(v_coeffs), _lib.ptr(v_means3d), _lib.stream_ptr(dev))
        _lib.check(rc, "bsplat_sh_bwd")
        return None, v_coeffs, v_means3d, None


def eval_sh_diff(sh_degree: int, sh_coeffs: torch.Tensor, means3d: torch.Tensor, camera: Camera) -> torch.Tensor:
    """Differentiable ``eval_sh`` (same values): gradients flow to ``sh_coeffs`` and, for degree >= 1, to ``means3d``
    through the view direction.  The camera gets none."""
    return _ShFn.apply(int(sh_degree), sh_coeffs, means3d, camera)
