"""Forward render orchestration (mirrors the reference's mojosplat/render.py:11-103).

``render_gaussians`` keeps the reference signature and behaviour (CUDA-tensor check :44-46,
background handling :48-58, ``opacities.shape == (N,)`` :60, all-zero image when nothing
intersects :73-76, ``sh_degree`` accepted but only truncating features :82-87).  With a CUDA
backend the three stages run inside ONE C call (bsplat_render_fwd): projection -> count+scan ->
one 32-byte read-back (M, depth-key range) -> emit -> onesweep sort -> tile ranges -> raster, all
on the caller's current stream, workspace reused across frames.
``render_gaussians_diff`` is the differentiable counterpart (stage by stage, with autograd); with ``absgrad=True``
it also collects AbsGS's absolute screen-space gradients for densification.
"""
from __future__ import annotations

import warnings
from ctypes import byref, c_size_t

import torch

from . import _lib
from .binning import bin_gaussians_to_tiles, bin_gaussians_to_tiles_cuda
from .projection import CUDA_BACKENDS, Camera, project_gaussians, project_gaussians_diff
from .rasterization import RASTER_MODES, rasterize_gaussians, rasterize_gaussians_diff
from .sh import eval_sh_diff

TILE_SIZE = 16


def _background_tensor(background_color, num_channels, device, dtype):
    if background_color is None:
        return torch.zeros(num_channels, device=device, dtype=dtype)
    if not isinstance(background_color, torch.Tensor):
        return torch.tensor(background_color, device=device, dtype=dtype)
    return background_color.to(device=device, dtype=dtype)


@torch.no_grad()
def render_gaussians(
    means3d: torch.Tensor,  # (N, 3) world coordinates
    scales: torch.Tensor,  # (N, 3) log-scales
    quats: torch.Tensor,  # (N, 4) w,x,y,z
    opacities: torch.Tensor,  # (N,) used as given (no activation)
    features: torch.Tensor,  # (N, C) colours
    camera: Camera,
    sh_degree: int | None = None,
    background_color: torch.Tensor | None = None,
    tile_size: int = TILE_SIZE,
    backend: str = "cuda",
) -> torch.Tensor:
    """Main function to render 3D Gaussians -> image (H, W, C). Reference: render.py:12-103."""
    required = [means3d, scales, quats, opacities, features]
    if not all(isinstance(t, torch.Tensor) and t.is_cuda for t in required):
        raise ValueError("All input gaussian tensors must be CUDA tensors.")
    if sh_degree is not None and features.dim() == 3:
        # real SH coefficients (N, K, 3): evaluate them along the view direction (additive; the reference
        # only has the placeholder below, render.py:82-87)
        from .sh import eval_sh
        features = eval_sh(int(sh_degree), features, means3d, camera).to(features.dtype)
        sh_degree = None
    num_channels = features.shape[-1]
    bg = _background_tensor(background_color, num_channels, means3d.device, features.dtype)
    if bg.shape[0] != num_channels:
        raise ValueError(f"Background color channels ({bg.shape[0]}) must match gaussian color "
                         f"channels ({num_channels})")
    assert opacities.shape == (means3d.shape[0],)

    colors = features
    if sh_degree is not None:
        # SH evaluation is a placeholder in the reference too (render.py:82-87)
        warnings.warn("SH evaluation not implemented; using the first 3 feature channels")
        if features.shape[-1] > 3:
            colors = features[..., :3]
            bg = bg[:3]

    if backend in CUDA_BACKENDS:
        image = render_fused(means3d, scales, quats, opacities, colors, camera, bg, tile_size,
                             semantics=CUDA_BACKENDS[backend])
        return image.to(features.dtype)

    # other backends: the reference's stage-by-stage flow (render.py:63-101)
    means2d, conics, depths, radii = project_gaussians(means3d, scales, quats, opacities, camera, backend=backend)
    sorted_ids, tile_ranges = bin_gaussians_to_tiles(means2d, radii, depths, camera.H, camera.W, tile_size,
                                                     backend=backend)
    if sorted_ids.numel() == 0:
        warnings.warn("No Gaussian overlaps found")
        return torch.zeros(camera.H, camera.W, colors.shape[-1], device=means3d.device, dtype=features.dtype)
    return rasterize_gaussians(means2d, conics, colors, opacities, bg, tile_ranges, sorted_ids, camera,
                               tile_size=tile_size, backend=backend)


def render_gaussians_diff(
    means3d: torch.Tensor,  # (N, 3) world coordinates
    scales: torch.Tensor,  # (N, 3) log-scales
    quats: torch.Tensor,  # (N, 4) w,x,y,z, need not be normalised
    opacities: torch.Tensor,  # (N,) used as given (no activation)
    features: torch.Tensor,  # (N, C) colours, or (N, K, 3) SH coefficients with sh_degree
    camera: Camera,
    sh_degree: int | None = None,
    background_color: torch.Tensor | None = None,
    tile_size: int = TILE_SIZE,
    backend: str = "cuda",
    return_aux: bool = False,
    absgrad: bool = False,
):
    """Differentiable ``render_gaussians``: image (H, W, C) with gradients for means3d, the log-scales, the raw quats,
    opacities, features (colours or SH coefficients) and a background_color tensor.  Arguments, checks and the
    features / SH / background rules are those of ``render_gaussians``; the camera gets no gradient.

    Stages: [eval_sh_diff] -> project_gaussians_diff -> binning (the tile lists are constants) ->
    rasterize_gaussians_diff.  Forward values equal ``render_gaussians``'s for 16x16 tiles and 3 channels; other tile
    sizes and channel counts (1..4) go through the rasterizer with the reference's operation order.  When no
    Gaussian overlaps a tile the image is the background (still differentiable with respect to it), where
    ``render_gaussians`` returns zeros.

    ``return_aux=True`` also returns ``dict(means2d, radii, depths, conics, tile_ranges, sorted_ids)``; ``means2d`` is
    the tensor of the graph (``retain_grad()`` it for screen-space statistics) and ``radii > 0`` marks the visible
    Gaussians.

    ``absgrad=True`` (needs ``return_aux=True``) adds ``aux["means2d_absgrad"]``, a zero (N, 2) float32 tensor that
    every backward pass through the image adds to: per Gaussian, the sum over the pixels it was composited at of
    |d loss_p / d means2d| (AbsGS; gsplat's ``info["means2d"].absgrad``).  It stays zero when no Gaussian overlaps a
    tile.  Densify on it with ``DensifyStats.accumulate(aux["means2d_absgrad"], aux["radii"], W, H)``."""
    if absgrad and not return_aux:
        raise ValueError("absgrad=True returns its statistic in aux: pass return_aux=True")
    required = [means3d, scales, quats, opacities, features]
    if not all(isinstance(t, torch.Tensor) and t.is_cuda for t in required):
        raise ValueError("All input gaussian tensors must be CUDA tensors.")
    if backend not in CUDA_BACKENDS:
        raise ValueError(f"Invalid backend: {backend}")
    if sh_degree is not None and features.dim() == 3:
        features = eval_sh_diff(int(sh_degree), features, means3d, camera).to(features.dtype)
        sh_degree = None
    num_channels = features.shape[-1]
    bg = _background_tensor(background_color, num_channels, means3d.device, features.dtype)
    if bg.shape[0] != num_channels:
        raise ValueError(f"Background color channels ({bg.shape[0]}) must match gaussian color "
                         f"channels ({num_channels})")
    assert opacities.shape == (means3d.shape[0],)
    colors = features
    if sh_degree is not None:
        warnings.warn("SH evaluation not implemented; using the first 3 feature channels")
        if features.shape[-1] > 3:
            colors = features[..., :3]
            bg = bg[:3]

    H, W = int(camera.H), int(camera.W)
    means2d, conics, depths, radii = project_gaussians_diff(means3d, scales, quats, opacities, camera, backend)
    sorted_ids, tile_ranges = bin_gaussians_to_tiles_cuda(means2d.detach(), radii, depths.detach(), H, W,
                                                          tile_size, semantics=CUDA_BACKENDS[backend])
    extra = {}
    if absgrad:
        extra["means2d_absgrad"] = torch.zeros((means2d.shape[0], 2), dtype=torch.float32, device=means2d.device)
    if sorted_ids.numel() == 0:
        warnings.warn("No Gaussian overlaps found; returning the background")
        image = bg.to(torch.float32).expand(H, W, bg.shape[0]).clone()
    else:
        image = rasterize_gaussians_diff(means2d, conics, colors, opacities, bg, tile_ranges, sorted_ids, camera,
                                         tile_size, means2d_absgrad=extra.get("means2d_absgrad"))
    image = image.to(features.dtype)
    if return_aux:
        return image, dict(means2d=means2d, radii=radii, depths=depths, conics=conics, tile_ranges=tile_ranges,
                           sorted_ids=sorted_ids, **extra)
    return image


def _workspace_for(L, dev, N, W, H, tile_size, hint_M=None):
    guess = hint_M if hint_M is not None else 8 * N + 4096
    need = L.bsplat_render_workspace_bytes(N, guess, W, H, tile_size)
    return _lib.workspace.get(dev, "render", need)


_last_M: dict = {}


def render_fused(means3d, scales, quats, opacities, colors, camera, background, tile_size=TILE_SIZE,
                 semantics=_lib.SEM_TORCH, raster_mode="fast", return_aux=False, timing=False, packed=False):
    """One C call per frame (include/bsplat.h: bsplat_render_fwd). Device tensors in, image out.
    ``packed``: gsplat's packed layout -- Gaussians that own no tile are compacted away right after projection
    (same image and lists; only pays under the gsplat rule set, where culled Gaussians own no tile)."""
    dev = means3d.device
    L = _lib.require_device(dev)
    means3d = _lib.as_f32(means3d, "means3d"); scales = _lib.as_f32(scales, "scales")
    quats = _lib.as_f32(quats, "quats"); opacities = _lib.as_f32(opacities, "opacities").reshape(-1)
    colors = _lib.as_f32(colors, "features"); background = _lib.as_f32(background, "background").to(dev)
    N, C = colors.shape
    H, W, ts = int(camera.H), int(camera.W), int(tile_size)
    cam = _lib.camera_struct(camera)
    image = torch.empty((H, W, C), dtype=torch.float32, device=dev)
    key = (dev.index, N, W, H, ts)
    ws = _workspace_for(L, dev, N, W, H, ts, _last_M.get(key))
    aux = _lib.BsplatRenderAux()
    aux.timing = 1 if timing else 0
    outs = None
    if return_aux:
        th, tw = (H + ts - 1) // ts, (W + ts - 1) // ts
        outs = dict(means2d=torch.empty((N, 2), dtype=torch.float32, device=dev),
                    conics=torch.empty((N, 3), dtype=torch.float32, device=dev),
                    depths=torch.empty((N,), dtype=torch.float32, device=dev),
                    radii=torch.empty((N, 2), dtype=torch.int32, device=dev),
                    tile_ranges=torch.zeros((th, tw, 2), dtype=torch.int32, device=dev))
        aux.means2d, aux.conics = outs["means2d"].data_ptr(), outs["conics"].data_ptr()
        aux.depths, aux.radii = outs["depths"].data_ptr(), outs["radii"].data_ptr()
        aux.tile_ranges = outs["tile_ranges"].data_ptr()
        cap = _last_M.get(key, 0)
        cap = int(cap * 1.3) + 4096 if cap else 0
        if cap:
            outs["sorted_ids"] = torch.empty((cap,), dtype=torch.int32, device=dev)
            aux.sorted_ids, aux.sorted_ids_capacity = outs["sorted_ids"].data_ptr(), cap
    needed = c_size_t(0)
    flags = RASTER_MODES[raster_mode] | (_lib.FLAG_PACKED if packed else 0)
    with torch.cuda.device(dev):
        for _attempt in range(3):
            rc = L.bsplat_render_fwd(N, _lib.ptr(means3d), _lib.ptr(scales), _lib.ptr(quats),
                                     _lib.ptr(opacities), _lib.ptr(colors), C, byref(cam),
                                     _lib.ptr(background), ts, semantics, flags,
                                     _lib.ptr(image), _lib.ptr(ws), ws.numel(), byref(needed), byref(aux),
                                     _lib.stream_ptr(dev))
            if rc == _lib.E_WORKSPACE:
                ws = _lib.workspace.get(dev, "render", int(needed.value))
                continue
            break
    _lib.check(rc, "bsplat_render_fwd")
    M = int(aux.n_isect)
    _last_M[key] = max(M, 1)
    if M == 0:
        warnings.warn("No Gaussian overlaps found; returning a black image (render.py:73-76)")
    if return_aux or timing:
        outs = outs if outs is not None else {}
        outs["n_isect"] = M
        outs["n_launches"] = int(aux.n_launches)
        outs["sort_passes"] = int(aux.sort_passes)
        outs["key_bits"] = int(aux.key_bits)
        if "sorted_ids" in outs:
            outs["sorted_ids"] = outs["sorted_ids"][:M] if outs["sorted_ids"].numel() >= M else None
        if timing:
            # [0] projection (+ fused epilogue), [1] depth sort + count/scan + the M read-back, [2] emit + tile sort +
            # ranges, [3] rasterizer (+ long-list pre-pass); the stage outputs are only stored with return_aux
            outs["stage_ms"] = [float(v) for v in aux.stage_ms]
        return image, outs
    return image


def render_gaussians_host(means3d, scales, quats, opacities, features, camera, background_color=None,
                          tile_size=TILE_SIZE, backend="cuda", out=None, device=None):
    """End-to-end call with HOST tensors (ideally pinned): H2D copies, render, D2H of the image, sync.
    Returns a host tensor (H, W, C).  This is the path bench.py's `e2e` figure times."""
    if backend not in CUDA_BACKENDS:
        raise ValueError(f"Invalid backend: {backend}")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    L = _lib.require_device(dev)
    for t in (means3d, scales, quats, opacities, features):
        if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError("render_gaussians_host expects contiguous float32 CPU tensors")
    N, C = features.shape
    assert opacities.shape == (N,)
    H, W, ts = int(camera.H), int(camera.W), int(tile_size)
    bg = _background_tensor(background_color, C, "cpu", torch.float32).contiguous()
    if out is None:
        out = torch.empty((H, W, C), dtype=torch.float32, pin_memory=True)
    cam = _lib.camera_struct(camera)
    key = (dev.index, N, W, H, ts)
    ws = _workspace_for(L, dev, N, W, H, ts, _last_M.get(key))
    scratch_bytes = L.bsplat_render_host_scratch_bytes(N, C, W, H)
    scratch = _lib.workspace.get(dev, "host_scratch", scratch_bytes)
    aux = _lib.BsplatRenderAux()
    needed = c_size_t(0)
    with torch.cuda.device(dev):
        for _attempt in range(3):
            rc = L.bsplat_render_fwd_host(N, means3d.data_ptr(), scales.data_ptr(), quats.data_ptr(),
                                          opacities.data_ptr(), features.data_ptr(), C, byref(cam),
                                          bg.data_ptr(), ts, CUDA_BACKENDS[backend], _lib.RASTER_FAST,
                                          out.data_ptr(), _lib.ptr(scratch), scratch.numel(), _lib.ptr(ws),
                                          ws.numel(), byref(needed), byref(aux), _lib.stream_ptr(dev))
            if rc == _lib.E_WORKSPACE:
                ws = _lib.workspace.get(dev, "render", int(needed.value))
                continue
            break
    _lib.check(rc, "bsplat_render_fwd_host")
    _last_M[key] = max(int(aux.n_isect), 1)
    return out
