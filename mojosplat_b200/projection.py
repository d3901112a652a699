"""Stage 1 -- projection dispatcher (mirrors the reference's mojosplat/projection.py:15-48).

``project_gaussians(means3d, scales, quats, opacity_features, camera, backend)`` keeps the
reference's positional order, return arity, shapes and dtypes:
``(means2d[N,2] f32, conics[N,3] f32, depths[N] f32, radii[N,2] i32)``.
New backend strings: ``"cuda"`` (alias ``"b200"``; the reference torch backend's rules,
projection.py:199-283) and ``"cuda_gsplat"`` (the gsplat / Mojo rules, projection.mojo:59-257).
``project_gaussians_diff`` is the differentiable form (additive: the reference is forward-only).
"""
from __future__ import annotations

from ctypes import byref

import torch

from . import _lib
from .utils import Camera  # noqa: F401  (re-exported like projection.py:10 of the reference)

CUDA_BACKENDS = {"cuda": _lib.SEM_TORCH, "b200": _lib.SEM_TORCH, "cuda_gsplat": _lib.SEM_GSPLAT}


def _reference_module(name: str):
    """Other backends live in the reference package; use it when it is installed."""
    try:
        import importlib
        return importlib.import_module(f"mojosplat.{name}")
    except Exception as e:  # pragma: no cover - depends on the environment
        raise RuntimeError(
            f"backend needs the reference package `mojosplat` ({name}), which is not importable "
            f"here ({type(e).__name__}: {e}); this package only ships the CUDA backends") from e


def project_gaussians(
    means3d: torch.Tensor,  # (N, 3)
    scales: torch.Tensor,  # (N, 3) log-scales
    quats: torch.Tensor,  # (N, 4) w,x,y,z
    opacity_features: torch.Tensor,  # (N, 1) or (N,)
    camera: Camera,
    backend: str = "cuda",
) -> tuple:
    """Projects 3D Gaussians to the image plane (reference: projection.py:15-48)."""
    if backend in CUDA_BACKENDS:
        return project_gaussians_cuda(means3d, scales, quats, opacity_features, camera,
                                      semantics=CUDA_BACKENDS[backend])
    if backend in ("torch", "gsplat", "mojo"):
        return _reference_module("projection").project_gaussians(
            means3d, scales, quats, opacity_features, camera, backend=backend)
    raise ValueError(f"Invalid backend: {backend}")


def project_gaussians_cuda(means3d, scales, quats, opacities, camera, semantics=_lib.SEM_TORCH,
                           out=None, allow_fma=False, fast_math=False):
    """sm_100a kernel behind the C ABI (include/bsplat.h: bsplat_project_fwd).
    ``allow_fma``: the A/B build with FMA contraction allowed (BSPLAT_PROJ_ALLOW_FMA)."""
    L = _lib.require_device(means3d.device)
    dev = means3d.device
    means3d = _lib.as_f32(means3d, "means3d")
    scales = _lib.as_f32(scales, "scales")
    quats = _lib.as_f32(quats, "quats")
    N = means3d.shape[0]
    if means3d.shape != (N, 3) or scales.shape != (N, 3) or quats.shape != (N, 4):
        raise ValueError("expected means3d (N,3), scales (N,3), quats (N,4)")
    op = None
    if opacities is not None:
        op = _lib.as_f32(opacities, "opacity_features").reshape(-1)
        if op.shape[0] != N:
            raise ValueError("opacity_features must have N entries")
    if out is None:
        means2d = torch.empty((N, 2), dtype=torch.float32, device=dev)
        conics = torch.empty((N, 3), dtype=torch.float32, device=dev)
        depths = torch.empty((N,), dtype=torch.float32, device=dev)
        radii = torch.empty((N, 2), dtype=torch.int32, device=dev)
    else:
        means2d, conics, depths, radii = out
    cam = _lib.camera_struct(camera)
    with torch.cuda.device(dev):
        rc = L.bsplat_project_fwd(N, _lib.ptr(means3d), _lib.ptr(scales), _lib.ptr(quats), _lib.ptr(op),
                                  byref(cam), 1, 0.3, semantics | (_lib.PROJ_ALLOW_FMA if allow_fma else 0) | (_lib.PROJ_FAST_MATH if fast_math else 0),
                                  _lib.ptr(means2d), _lib.ptr(conics),
                                  _lib.ptr(depths), _lib.ptr(radii), _lib.stream_ptr(dev))
    _lib.check(rc, "bsplat_project_fwd")
    return means2d, conics, depths, radii


class _ProjectFn(torch.autograd.Function):
    """Projection with a backward pass (bsplat_project_fwd / bsplat_project_bwd)."""

    @staticmethod
    def forward(ctx, means3d, scales, quats, opacities, camera, semantics):
        means2d, conics, depths, radii = project_gaussians_cuda(means3d, scales, quats, opacities, camera,
                                                                semantics=semantics)
        ctx.save_for_backward(_lib.as_f32(means3d, "means3d"), _lib.as_f32(scales, "scales"),
                              _lib.as_f32(quats, "quats"), radii)
        ctx.camera, ctx.semantics = camera, semantics
        ctx.mark_non_differentiable(radii)
        return means2d, conics, depths, radii

    @staticmethod
    def backward(ctx, v_means2d, v_conics, v_depths, _v_radii):
        means3d, scales, quats, radii = ctx.saved_tensors
        dev = means3d.device
        L = _lib.require_device(dev)
        N = means3d.shape[0]
        v_means2d = _lib.as_f32(v_means2d, "v_means2d")
        v_conics = _lib.as_f32(v_conics, "v_conics")
        v_depths = _lib.as_f32(v_depths, "v_depths")
        v_means3d = torch.empty((N, 3), dtype=torch.float32, device=dev)
        v_scales = torch.empty((N, 3), dtype=torch.float32, device=dev)
        v_quats = torch.empty((N, 4), dtype=torch.float32, device=dev)
        cam = _lib.camera_struct(ctx.camera)
        with torch.cuda.device(dev):
            rc = L.bsplat_project_bwd(N, _lib.ptr(means3d), _lib.ptr(scales), _lib.ptr(quats), byref(cam), 0.3,
                                      ctx.semantics, _lib.ptr(radii), _lib.ptr(v_means2d), _lib.ptr(v_conics),
                                      _lib.ptr(v_depths), _lib.ptr(v_means3d), _lib.ptr(v_scales), _lib.ptr(v_quats),
                                      _lib.stream_ptr(dev))
        _lib.check(rc, "bsplat_project_bwd")
        return v_means3d, v_scales, v_quats, None, None, None


def project_gaussians_diff(means3d, scales, quats, opacities, camera, backend="cuda"):
    """Differentiable ``project_gaussians`` -> ``(means2d, conics, depths, radii)``.  The forward is the exact stage
    kernel (values bit-identical to ``project_gaussians``); gradients flow to ``means3d``, the log-``scales`` and the
    raw (unnormalised) ``quats``.  ``radii`` is not differentiable, and neither is the opacity (it only decides the
    cull of the ``"cuda_gsplat"`` rules).  Culled rows (radii == 0) get zero gradients."""
    if backend not in CUDA_BACKENDS:
        raise ValueError(f"Invalid backend: {backend}")
    return _ProjectFn.apply(means3d, scales, quats, opacities, camera, CUDA_BACKENDS[backend])
