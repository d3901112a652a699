"""Stage 2 -- binning dispatcher (mirrors the reference's mojosplat/binning.py:8-37).

``bin_gaussians_to_tiles(means2d, radii, depths, img_height, img_width, tile_size, backend)``
returns ``(sorted_gaussian_indices[M] int32, tile_ranges[th, tw, 2] int32)`` exactly like the
reference torch backend (binning.py:108-262); the CUDA backend is bit-exact against it, with the
stable tie order (tile, depth, gaussian index) where the reference's unstable argsort is free.
"""
from __future__ import annotations

import math
from ctypes import byref, c_int32

import numpy as np
import torch

from . import _lib
from .projection import CUDA_BACKENDS, _reference_module


def bin_gaussians_to_tiles(
    means2d: torch.Tensor,  # [N, 2]
    radii: torch.Tensor,  # [N, 2] int32 (from projection) or float
    depths: torch.Tensor,  # [N]
    img_height: int,
    img_width: int,
    tile_size: int,
    backend: str = "cuda",
) -> tuple:
    """Bin Gaussians to tiles (reference: binning.py:8-37)."""
    if backend in CUDA_BACKENDS:
        return bin_gaussians_to_tiles_cuda(means2d, radii, depths, img_height, img_width, tile_size,
                                           semantics=CUDA_BACKENDS[backend])
    if backend in ("torch", "gsplat", "mojo"):
        return _reference_module("binning").bin_gaussians_to_tiles(
            means2d, radii, depths, img_height, img_width, tile_size, backend=backend)
    raise ValueError(f"Invalid backend: {backend}")


def read_bin_info(info_dev: torch.Tensor) -> _lib.BsplatBinInfo:
    """A bin info (32 bytes: M, the depth-key range, the overflow flag) from a device tensor -- the single device->host
    read-back of the stage -- or from a host block (no copy)."""
    host = info_dev.cpu().numpy().tobytes()
    return _lib.BsplatBinInfo.from_buffer_copy(host)


def bin_gaussians_to_tiles_cuda(means2d, radii, depths, img_height, img_width, tile_size,
                                semantics=_lib.SEM_TORCH, tile_rows=None, return_keys=False,
                                algo="two_level", packed=False):
    """Binning on the GPU, two algorithms with bit-identical results:

    ``algo="two_level"`` (default): depth-sort the N Gaussians, count+scan and emit in depth order,
    stable-sort the M pairs by tile id only (bsplat_bin2_prepare / bsplat_bin2_finish).
    ``algo="single"``: count+scan -> emit packed (tile << depth_bits | depth) keys -> one onesweep
    sort over the live key bits -> tile ranges (needed for ``return_keys``).

    ``tile_rows=(begin, end)`` restricts emission to a band of tile rows (row-band multi-GPU split);
    per-tile lists inside the band are identical to the full-frame ones.
    ``packed`` (two-level only): Gaussians without a tile are compacted away before the depth sort (same lists).
    """
    if algo == "two_level" and not return_keys:
        return _bin_two_level(means2d, radii, depths, img_height, img_width, tile_size,
                              semantics | (_lib.BIN_PACKED if packed else 0), tile_rows)
    dev = means2d.device
    L = _lib.require_device(dev)
    means2d = _lib.as_f32(means2d, "means2d")
    depths = _lib.as_f32(depths, "depths").reshape(-1)
    N = means2d.shape[0]
    if radii.dtype == torch.int32:
        radii_c, radii_is_float = radii.contiguous(), 0
    else:
        radii_c, radii_is_float = radii.to(torch.float32).contiguous(), 1
    if means2d.shape != (N, 2) or radii_c.shape != (N, 2) or depths.shape != (N,):
        raise ValueError("expected means2d (N,2), radii (N,2), depths (N,)")
    H, W, ts = int(img_height), int(img_width), int(tile_size)
    th, tw = math.ceil(H / ts), math.ceil(W / ts)
    r0, r1 = (0, th) if tile_rows is None else (int(tile_rows[0]), int(tile_rows[1]))
    stream = _lib.stream_ptr(dev)

    offsets = torch.empty((N + 1,), dtype=torch.int32, device=dev)
    info = torch.empty((32,), dtype=torch.uint8, device=dev)
    scan_bytes = L.bsplat_bin_scan_workspace_bytes(N)
    scan_ws = _lib.workspace.get(dev, "scan", scan_bytes)
    tile_ranges = torch.empty((th, tw, 2), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.bsplat_bin_count_scan(N, _lib.ptr(means2d), _lib.ptr(radii_c), radii_is_float,
                                           _lib.ptr(depths), W, H, ts, r0, r1, semantics, _lib.ptr(offsets),
                                           _lib.ptr(info), _lib.ptr(scan_ws), scan_bytes, stream),
                   "bsplat_bin_count_scan")
        info_h = read_bin_info(info)
        M = int(info_h.n_isect)
        if M >= (1 << 30):
            raise _lib.BsplatError(_lib.E_OVERFLOW, "bin_gaussians_to_tiles")
        layout = L.bsplat_make_key_layout(byref(info_h), W, H, ts)
        keys = torch.empty((M,), dtype=torch.int64, device=dev)
        keys_alt = torch.empty((M,), dtype=torch.int64, device=dev)
        ids = torch.empty((M,), dtype=torch.int32, device=dev)
        ids_alt = torch.empty((M,), dtype=torch.int32, device=dev)
        end_bit = layout.depth_bits + layout.tile_bits
        _lib.check(L.bsplat_bin_emit(N, _lib.ptr(means2d), _lib.ptr(radii_c), radii_is_float, _lib.ptr(depths),
                                     W, H, ts, r0, r1, semantics, _lib.ptr(offsets), layout, _lib.ptr(keys),
                                     _lib.ptr(ids), stream), "bsplat_bin_emit")
        sort_bytes = L.bsplat_radix_sort_workspace_bytes(M, 0, end_bit)
        sort_ws = _lib.workspace.get(dev, "sort", sort_bytes)
        in_alt = c_int32(0)
        _lib.check(L.bsplat_radix_sort_pairs(M, _lib.ptr(keys), _lib.ptr(keys_alt), _lib.ptr(ids),
                                             _lib.ptr(ids_alt), 0, end_bit, _lib.ptr(sort_ws), sort_bytes,
                                             byref(in_alt), stream), "bsplat_radix_sort_pairs")
        sorted_keys, sorted_ids = (keys_alt, ids_alt) if in_alt.value else (keys, ids)
        _lib.check(L.bsplat_tile_ranges(M, _lib.ptr(sorted_keys), layout.depth_bits, th * tw,
                                        _lib.ptr(tile_ranges), stream), "bsplat_tile_ranges")
    if return_keys:
        return sorted_ids, tile_ranges, sorted_keys, layout
    return sorted_ids, tile_ranges


def _bin_two_level(means2d, radii, depths, img_height, img_width, tile_size, semantics, tile_rows):
    dev = means2d.device
    L = _lib.require_device(dev)
    means2d = _lib.as_f32(means2d, "means2d")
    depths = _lib.as_f32(depths, "depths").reshape(-1)
    N = means2d.shape[0]
    if radii.dtype == torch.int32:
        radii_c, radii_is_float = radii.contiguous(), 0
    else:
        radii_c, radii_is_float = radii.to(torch.float32).contiguous(), 1
    if means2d.shape != (N, 2) or radii_c.shape != (N, 2) or depths.shape != (N,):
        raise ValueError("expected means2d (N,2), radii (N,2), depths (N,)")
    H, W, ts = int(img_height), int(img_width), int(tile_size)
    th, tw = math.ceil(H / ts), math.ceil(W / ts)
    r0, r1 = (0, th) if tile_rows is None else (int(tile_rows[0]), int(tile_rows[1]))
    stream = _lib.stream_ptr(dev)
    info = torch.empty((32,), dtype=torch.uint8, device=dev)
    tile_ranges = torch.empty((th, tw, 2), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        ws = _lib.workspace.get(dev, "bin2", L.bsplat_bin2_workspace_bytes(N, 4 * N + 1024, th * tw))
        _lib.check(L.bsplat_bin2_prepare(N, _lib.ptr(means2d), _lib.ptr(radii_c), radii_is_float, _lib.ptr(depths),
                                         W, H, ts, r0, r1, semantics, _lib.ptr(ws), ws.numel(), _lib.ptr(info),
                                         stream), "bsplat_bin2_prepare")
        M = int(read_bin_info(info).n_isect)
        if M >= (1 << 30):
            raise _lib.BsplatError(_lib.E_OVERFLOW, "bin_gaussians_to_tiles")
        need = L.bsplat_bin2_workspace_bytes(N, M, th * tw)
        if ws.numel() < need:
            # grow, keeping the N-part (perm, offsets) that prepare just produced
            old = ws
            ws = torch.empty(int(need * 1.25), dtype=torch.uint8, device=dev)
            n_part = L.bsplat_bin2_workspace_bytes(N, 0, 0)
            ws[:n_part].copy_(old[:n_part])
            _lib.workspace.put(dev, "bin2", ws)
        sorted_ids = torch.empty((M,), dtype=torch.int32, device=dev)
        _lib.check(L.bsplat_bin2_finish(N, M, _lib.ptr(means2d), _lib.ptr(radii_c), radii_is_float, W, H, ts, r0, r1,
                                        semantics, _lib.ptr(ws), ws.numel(), _lib.ptr(sorted_ids),
                                        _lib.ptr(tile_ranges), None, stream), "bsplat_bin2_finish")
    return sorted_ids, tile_ranges
