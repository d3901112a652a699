"""Stage 3 -- rasterization dispatcher (mirrors the reference's mojosplat/rasterization.py:13-57).

``rasterize_gaussians(means2d, conics, colors, opacities, background_color, tile_ranges,
sorted_gaussian_indices, camera, tile_size=16, backend)`` -> ``image[H, W, C]`` float32.
Opacities are used raw (no sigmoid), tile_ranges may be int64 (cast like rasterization.py:163).
``rasterize_gaussians_diff`` is the differentiable counterpart; with ``means2d_absgrad`` its backward also adds
AbsGS's absolute screen-space gradients (gsplat's ``absgrad``) into that tensor.
"""
from __future__ import annotations

import torch

from . import _lib
from .projection import CUDA_BACKENDS, _reference_module
from .utils import Camera

RASTER_MODES = {"fast": _lib.RASTER_FAST, "faithful": _lib.RASTER_FAITHFUL, "fast_nocull": _lib.RASTER_FAST_NOCULL}


def rasterize_gaussians(
    means2d: torch.Tensor,  # (N, 2)
    conics: torch.Tensor,  # (N, 3)
    colors: torch.Tensor,  # (N, C)
    opacities: torch.Tensor,  # (N,) or (N, 1)
    background_color: torch.Tensor,  # (C,)
    tile_ranges: torch.Tensor,  # (tile_height, tile_width, 2)
    sorted_gaussian_indices: torch.Tensor,  # (M,)
    camera: Camera,
    tile_size: int = 16,
    backend: str = "cuda",
) -> torch.Tensor:
    """Rasterizes 2D Gaussians to pixels (reference: rasterization.py:13-57)."""
    if backend in CUDA_BACKENDS:
        return rasterize_gaussians_cuda(means2d, conics, colors, opacities, background_color, tile_ranges,
                                        sorted_gaussian_indices, camera, tile_size)
    if backend in ("torch", "gsplat", "mojo"):
        return _reference_module("rasterization").rasterize_gaussians(
            means2d, conics, colors, opacities, background_color, tile_ranges, sorted_gaussian_indices,
            camera, tile_size=tile_size, backend=backend)
    raise ValueError(f"Invalid backend: {backend}")


def _prep(means2d, conics, colors, opacities, background_color, tile_ranges, sorted_ids):
    dev = means2d.device
    means2d = _lib.as_f32(means2d, "means2d")
    conics = _lib.as_f32(conics, "conics")
    colors = _lib.as_f32(colors, "colors")
    opacities = _lib.as_f32(opacities, "opacities").reshape(-1)
    background = _lib.as_f32(background_color, "background_color").reshape(-1).to(dev)
    tile_ranges = tile_ranges.to(torch.int32).contiguous()
    sorted_ids = sorted_ids.reshape(-1).to(torch.int32).contiguous()
    N, C = colors.shape
    if means2d.shape != (N, 2) or conics.shape != (N, 3) or opacities.shape != (N,):
        raise ValueError("expected means2d (N,2), conics (N,3), colors (N,C), opacities (N,)")
    if background.shape[0] != C:
        raise ValueError(f"Background color channels ({background.shape[0]}) must match gaussian color channels ({C})")
    return dev, means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, N, C


def rasterize_gaussians_cuda(means2d, conics, colors, opacities, background_color, tile_ranges,
                             sorted_gaussian_indices, camera, tile_size=16, mode="fast", tile_rows=None,
                             out=None):
    """sm_100a tile rasterizer behind the C ABI (include/bsplat.h: bsplat_rasterize_fwd).

    ``tile_rows=(begin, end)`` rasterizes only that band of tile rows into ``out`` (the other rows of
    the image are left untouched): the per-rank step of the row-band multi-GPU split."""
    L = _lib.require_device(means2d.device)
    dev, means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, N, C = _prep(
        means2d, conics, colors, opacities, background_color, tile_ranges, sorted_gaussian_indices)
    H, W = int(camera.H), int(camera.W)
    image = torch.empty((H, W, C), dtype=torch.float32, device=dev) if out is None else out
    th, tw = tile_ranges.shape[0], tile_ranges.shape[1]
    r0, r1 = (0, th) if tile_rows is None else (int(tile_rows[0]), int(tile_rows[1]))
    with torch.cuda.device(dev):
        order = None
        if mode != "faithful" and int(tile_size) == 16 and C == 3 and r1 > r0:
            # heavy tiles first: a scheduling hint only, results do not depend on it
            order = torch.empty(((r1 - r0) * tw,), dtype=torch.int32, device=dev)
            _lib.check(L.bsplat_tile_order(r0 * tw, order.numel(), _lib.ptr(tile_ranges), _lib.ptr(order),
                                           _lib.stream_ptr(dev)), "bsplat_tile_order")
        ws = None
        if order is not None and mode in ("fast", "fast_nocull"):
            ws = _lib.workspace.get(dev, "raster_rec", L.bsplat_rasterize_workspace_bytes(N))
        rc = L.bsplat_rasterize_fwd(N, C, _lib.ptr(means2d), _lib.ptr(conics), _lib.ptr(colors),
                                    _lib.ptr(opacities), _lib.ptr(background), _lib.ptr(tile_ranges),
                                    _lib.ptr(order), _lib.ptr(sorted_ids), sorted_ids.numel(), W, H, int(tile_size),
                                    r0, r1, RASTER_MODES[mode], _lib.ptr(image), _lib.ptr(ws),
                                    0 if ws is None else ws.numel(), _lib.stream_ptr(dev))
    _lib.check(rc, "bsplat_rasterize_fwd")
    return image


def rasterize_gaussians_stats(means2d, conics, colors, opacities, background_color, tile_ranges,
                              sorted_gaussian_indices, camera, tile_size=16):
    """Faithful kernel + work counters: returns (image, E_all, E_pass) -- the evaluated and the
    contributing (pixel, Gaussian) pairs of the reference algorithm (SURVEY.md 8d)."""
    L = _lib.require_device(means2d.device)
    dev, means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, N, C = _prep(
        means2d, conics, colors, opacities, background_color, tile_ranges, sorted_gaussian_indices)
    H, W = int(camera.H), int(camera.W)
    image = torch.empty((H, W, C), dtype=torch.float32, device=dev)
    stats = torch.zeros((2,), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        rc = L.bsplat_rasterize_stats(N, C, _lib.ptr(means2d), _lib.ptr(conics), _lib.ptr(colors),
                                      _lib.ptr(opacities), _lib.ptr(background), _lib.ptr(tile_ranges),
                                      _lib.ptr(sorted_ids), sorted_ids.numel(), W, H, int(tile_size),
                                      _lib.ptr(image), _lib.ptr(stats), _lib.stream_ptr(dev))
    _lib.check(rc, "bsplat_rasterize_stats")
    e_all, e_pass = stats.tolist()
    return image, int(e_all), int(e_pass)


class _RasterizeFn(torch.autograd.Function):
    """Differentiable compositing (bsplat_rasterize_fwd_train / bsplat_rasterize_bwd)."""

    @staticmethod
    def forward(ctx, means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, H, W, tile_size,
                mode="fast", means2d_absgrad=None):
        L = _lib.require_device(means2d.device)
        dev, means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, N, C = _prep(
            means2d, conics, colors, opacities, background, tile_ranges, sorted_ids)
        if not 1 <= C <= 4:
            raise ValueError("the differentiable rasterizer supports 1..4 colour channels")
        image = torch.empty((H, W, C), dtype=torch.float32, device=dev)
        final_T = torch.empty((H, W), dtype=torch.float32, device=dev)
        last_idx = torch.empty((H, W), dtype=torch.int32, device=dev)
        # the fast forward kernel serves the default shape (16x16 tiles, RGB); everything else, and mode="faithful",
        # goes through the kernel with the reference's operation order
        fast = (mode == "fast" and int(tile_size) == 16 and C == 3 and means2d.data_ptr() % 8 == 0 and H > 0 and W > 0)
        with torch.cuda.device(dev):
            if fast:
                th, tw = tile_ranges.shape[0], tile_ranges.shape[1]
                order = torch.empty((th * tw,), dtype=torch.int32, device=dev)
                _lib.check(L.bsplat_tile_order(0, order.numel(), _lib.ptr(tile_ranges), _lib.ptr(order),
                                               _lib.stream_ptr(dev)), "bsplat_tile_order")
                ws = _lib.workspace.get(dev, "raster_rec", L.bsplat_rasterize_workspace_bytes(N))
                rc = L.bsplat_rasterize_fwd_train_fast(N, _lib.ptr(means2d), _lib.ptr(conics), _lib.ptr(colors),
                                                       _lib.ptr(opacities), _lib.ptr(background),
                                                       _lib.ptr(tile_ranges), _lib.ptr(order), _lib.ptr(sorted_ids),
                                                       sorted_ids.numel(), W, H, _lib.ptr(image), _lib.ptr(final_T),
                                                       _lib.ptr(last_idx), _lib.ptr(ws), ws.numel(),
                                                       _lib.stream_ptr(dev))
            else:
                rc = L.bsplat_rasterize_fwd_train(N, C, _lib.ptr(means2d), _lib.ptr(conics), _lib.ptr(colors),
                                                  _lib.ptr(opacities), _lib.ptr(background), _lib.ptr(tile_ranges),
                                                  _lib.ptr(sorted_ids), sorted_ids.numel(), W, H, int(tile_size),
                                                  _lib.ptr(image), _lib.ptr(final_T), _lib.ptr(last_idx),
                                                  _lib.stream_ptr(dev))
        _lib.check(rc, "bsplat_rasterize_fwd_train_fast" if fast else "bsplat_rasterize_fwd_train")
        ctx.save_for_backward(means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, final_T,
                              last_idx)
        ctx.dims = (H, W, int(tile_size))
        ctx.fast = fast
        ctx.order = order if fast else None  # heavy tiles first: reused by the backward pass
        ctx.absgrad = means2d_absgrad  # an output of the backward, not an input: added into, never saved
        return image

    @staticmethod
    def backward(ctx, grad_image):
        means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, final_T, last_idx = ctx.saved_tensors
        H, W, ts = ctx.dims
        dev = means2d.device
        L = _lib.require_device(dev)
        N, C = colors.shape
        grad_image = grad_image.to(torch.float32).contiguous()
        g_m = torch.zeros_like(means2d); g_k = torch.zeros_like(conics)
        g_c = torch.zeros_like(colors); g_o = torch.zeros_like(opacities)
        absgrad = ctx.absgrad
        name = "bsplat_rasterize_bwd_fast" if ctx.fast else "bsplat_rasterize_bwd"
        name += "" if absgrad is None else "_abs"
        # the _abs entry points take the absolute-gradient array right after grad_means2d
        g_means = [_lib.ptr(g_m)] if absgrad is None else [_lib.ptr(g_m), _lib.ptr(absgrad)]
        with torch.cuda.device(dev):
            if ctx.fast:
                order = ctx.order
                ws = _lib.workspace.get(dev, "raster_rec", L.bsplat_rasterize_workspace_bytes(N))
                rc = getattr(L, name)(N, _lib.ptr(means2d), _lib.ptr(conics), _lib.ptr(colors),
                                      _lib.ptr(opacities), _lib.ptr(background), _lib.ptr(tile_ranges),
                                      _lib.ptr(order), _lib.ptr(sorted_ids), sorted_ids.numel(), W, H,
                                      _lib.ptr(final_T), _lib.ptr(last_idx), _lib.ptr(grad_image), *g_means,
                                      _lib.ptr(g_k), _lib.ptr(g_c), _lib.ptr(g_o), _lib.ptr(ws), ws.numel(),
                                      _lib.stream_ptr(dev))
            else:
                rc = getattr(L, name)(N, C, _lib.ptr(means2d), _lib.ptr(conics), _lib.ptr(colors),
                                      _lib.ptr(opacities), _lib.ptr(background), _lib.ptr(tile_ranges),
                                      _lib.ptr(sorted_ids), sorted_ids.numel(), W, H, ts, _lib.ptr(final_T),
                                      _lib.ptr(last_idx), _lib.ptr(grad_image), *g_means, _lib.ptr(g_k),
                                      _lib.ptr(g_c), _lib.ptr(g_o), _lib.stream_ptr(dev))
        _lib.check(rc, name)
        g_bg = (final_T.unsqueeze(-1) * grad_image).sum(dim=(0, 1))
        return g_m, g_k, g_c, g_o, g_bg, None, None, None, None, None, None, None


def rasterize_gaussians_diff(means2d, conics, colors, opacities, background_color, tile_ranges,
                             sorted_gaussian_indices, camera, tile_size=16, mode="fast", means2d_absgrad=None):
    """Differentiable ``rasterize_gaussians`` (additive: the reference is forward-only, render.py:11).
    Gradients flow to means2d, conics, colors, opacities and background_color; the tile lists are
    treated as constants. Forward values: ``mode="fast"`` (16x16 tiles, RGB) = the default inference kernel's, bit for
    bit; ``mode="faithful"`` (and every other shape) = the faithful kernel's.

    ``means2d_absgrad``: an optional (N, 2) float32 contiguous tensor on means2d's device.  Every backward pass through
    this image ADDS to it, per Gaussian, the sum over the pixels it was composited at of |d loss_p / d means2d| (x and
    y separately, the absolute value taken per pixel): AbsGS's densification statistic, gsplat's ``absgrad``.  Unlike
    the signed gradient it does not cancel when pixels on opposite sides pull the mean in opposite directions."""
    if mode not in ("fast", "faithful"):
        raise ValueError(f"Invalid mode: {mode}")
    if means2d_absgrad is not None:
        N = means2d.shape[0]
        if not isinstance(means2d_absgrad, torch.Tensor) or means2d_absgrad.shape != (N, 2):
            raise ValueError(f"means2d_absgrad must be a ({N}, 2) tensor, got "
                             f"{tuple(getattr(means2d_absgrad, 'shape', ()))}")
        if means2d_absgrad.dtype != torch.float32 or not means2d_absgrad.is_contiguous():
            raise ValueError(f"means2d_absgrad must be contiguous float32, got {means2d_absgrad.dtype}")
        if means2d_absgrad.device != means2d.device:
            raise ValueError(f"means2d_absgrad is on {means2d_absgrad.device}, means2d on {means2d.device}")
    opac = opacities.reshape(-1)
    return _RasterizeFn.apply(means2d, conics, colors, opac, background_color, tile_ranges,
                              sorted_gaussian_indices, int(camera.H), int(camera.W), int(tile_size), mode,
                              means2d_absgrad)
