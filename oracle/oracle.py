"""ctypes front-end of the CPU oracle (oracle/oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module; the product package ``mojosplat_b200`` never does.

All functions take and return numpy arrays (fp32 / int32), single camera, in the layouts
of the reference API (mojosplat/projection.py:15-48, binning.py:8-37, rasterization.py:13-57).
"""
from __future__ import annotations

import ctypes
import math
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB_PATH = _HERE / "_build" / "liboracle.so"
_lib = None

SEM_TORCH = 0
SEM_GSPLAT = 1


def build(force: bool = False) -> Path:
    """Compile oracle.c with gcc (seconds). Idempotent."""
    src = _HERE / "oracle.c"
    if force or not _LIB_PATH.exists() or _LIB_PATH.stat().st_mtime < src.stat().st_mtime:
        subprocess.check_call(["sh", str(_HERE / "build.sh")])
    return _LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(str(_LIB_PATH))
        L.oracle_num_threads.restype = ctypes.c_int
        L.oracle_set_num_threads.argtypes = [ctypes.c_int]
        L.oracle_bin_count.restype = ctypes.c_int64
        L.oracle_bin.restype = ctypes.c_int64
        _lib = L
    return _lib


def num_threads() -> int:
    return int(lib().oracle_num_threads())


def set_num_threads(n: int) -> None:
    lib().oracle_set_num_threads(int(n))


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(ctypes.c_void_p)


def project(means3d, log_scales, quats, opacities, viewmat, fx, fy, cx, cy, W, H,
            near=0.1, far=100.0, eps2d=0.3, semantics=SEM_TORCH):
    """-> (means2d[N,2] f32, conics[N,3] f32, depths[N] f32, radii[N,2] i32)."""
    means3d, log_scales, quats = _f32(means3d), _f32(log_scales), _f32(quats)
    viewmat = _f32(viewmat).reshape(16)
    N = means3d.shape[0]
    op = None if opacities is None else _f32(opacities).reshape(-1)
    means2d = np.zeros((N, 2), np.float32)
    conics = np.zeros((N, 3), np.float32)
    depths = np.zeros((N,), np.float32)
    radii = np.zeros((N, 2), np.int32)
    f = ctypes.c_float
    lib().oracle_project(
        ctypes.c_int64(N), _ptr(means3d), _ptr(log_scales), _ptr(quats),
        _ptr(op) if op is not None else ctypes.c_void_p(0), _ptr(viewmat),
        f(fx), f(fy), f(cx), f(cy), ctypes.c_int(W), ctypes.c_int(H),
        f(near), f(far), f(eps2d), ctypes.c_int(semantics),
        _ptr(means2d), _ptr(conics), _ptr(depths), _ptr(radii))
    return means2d, conics, depths, radii


def bin_count(means2d, radii, W, H, tile_size, semantics=SEM_TORCH):
    means2d, radii_f = _f32(means2d), _f32(radii)
    N = means2d.shape[0]
    counts = np.zeros((N,), np.int32)
    M = lib().oracle_bin_count(ctypes.c_int64(N), _ptr(means2d), _ptr(radii_f),
                               ctypes.c_int(W), ctypes.c_int(H), ctypes.c_int(tile_size),
                               ctypes.c_int(semantics), _ptr(counts))
    return int(M), counts


def bin_tiles(means2d, radii, depths, H, W, tile_size, semantics=SEM_TORCH, return_keys=False):
    """-> (sorted_ids[M] i32, tile_ranges[th,tw,2] i32[, isect_keys[M] u64])."""
    means2d, radii_f, depths = _f32(means2d), _f32(radii), _f32(depths)
    N = means2d.shape[0]
    th, tw = math.ceil(H / tile_size), math.ceil(W / tile_size)
    M, _ = bin_count(means2d, radii_f, W, H, tile_size, semantics)
    ids = np.zeros((max(M, 1),), np.int32)
    keys = np.zeros((max(M, 1),), np.uint64)
    ranges = np.zeros((th, tw, 2), np.int32)
    m = lib().oracle_bin(ctypes.c_int64(N), _ptr(means2d), _ptr(radii_f), _ptr(depths),
                         ctypes.c_int(W), ctypes.c_int(H), ctypes.c_int(tile_size),
                         ctypes.c_int(semantics), ctypes.c_int64(M), _ptr(ids), _ptr(keys),
                         _ptr(ranges))
    assert m == M, (m, M)
    if return_keys:
        return ids[:M], ranges, keys[:M]
    return ids[:M], ranges


def rasterize(means2d, conics, colors, opacities, background, tile_ranges, sorted_ids,
              W, H, tile_size=16, return_stats=False):
    """-> image[H,W,C] f32 (and (E_all, E_pass) evaluation counts)."""
    means2d, conics, colors = _f32(means2d), _f32(conics), _f32(colors)
    opacities = _f32(opacities).reshape(-1)
    background = _f32(background).reshape(-1)
    N, C = colors.shape
    ranges = np.ascontiguousarray(np.asarray(tile_ranges, dtype=np.int32))
    ids = np.ascontiguousarray(np.asarray(sorted_ids, dtype=np.int32))
    image = np.zeros((H, W, C), np.float32)
    stats = np.zeros((2,), np.int64)
    lib().oracle_rasterize(ctypes.c_int64(N), ctypes.c_int(C), _ptr(means2d), _ptr(conics),
                           _ptr(colors), _ptr(opacities), _ptr(background), _ptr(ranges),
                           _ptr(ids), ctypes.c_int(W), ctypes.c_int(H), ctypes.c_int(tile_size),
                           _ptr(image), _ptr(stats))
    if return_stats:
        return image, (int(stats[0]), int(stats[1]))
    return image


def project_f64(means3d, log_scales, quats, viewmat, fx, fy, cx, cy, W, H, near=0.1, far=100.0, eps2d=0.3):
    """Torch-rule projection evaluated in double precision from the fp32 inputs (error-budget yardstick).
    -> (means2d[N,2], conics[N,3], depths[N], radii_real[N,2]) float64; radii_real = 3.33 sqrt(c) before ceil."""
    means3d, log_scales, quats = _f32(means3d), _f32(log_scales), _f32(quats)
    viewmat = _f32(viewmat).reshape(16)
    N = means3d.shape[0]
    means2d = np.zeros((N, 2), np.float64)
    conics = np.zeros((N, 3), np.float64)
    depths = np.zeros((N,), np.float64)
    radii = np.zeros((N, 2), np.float64)
    d = ctypes.c_double
    lib().oracle_project_f64(ctypes.c_int64(N), _ptr(means3d), _ptr(log_scales), _ptr(quats), _ptr(viewmat),
                             d(fx), d(fy), d(cx), d(cy), ctypes.c_int(W), ctypes.c_int(H), d(near), d(far), d(eps2d),
                             _ptr(means2d), _ptr(conics), _ptr(depths), _ptr(radii))
    return means2d, conics, depths, radii


def rasterize_f64(means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, W, H, tile_size=16):
    """The rasterizer in double precision on the fp32 inputs -> image[H,W,C] float64."""
    means2d, conics, colors = _f32(means2d), _f32(conics), _f32(colors)
    opacities = _f32(opacities).reshape(-1)
    background = _f32(background).reshape(-1)
    N, C = colors.shape
    ranges = np.ascontiguousarray(np.asarray(tile_ranges, dtype=np.int32))
    ids = np.ascontiguousarray(np.asarray(sorted_ids, dtype=np.int32))
    image = np.zeros((H, W, C), np.float64)
    lib().oracle_rasterize_f64(ctypes.c_int64(N), ctypes.c_int(C), _ptr(means2d), _ptr(conics), _ptr(colors),
                               _ptr(opacities), _ptr(background), _ptr(ranges), _ptr(ids), ctypes.c_int(W),
                               ctypes.c_int(H), ctypes.c_int(tile_size), _ptr(image))
    return image


def raster_bwd_f64(means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, W, H, tile_size,
                   grad_image, mask_borderline=False):
    """Compositing backward in double precision on the fp32 inputs (see oracle.c: oracle_raster_bwd_f64), for the
    upstream gradient grad_image [H, W, C].  Returns a dict of numpy arrays:
      grad_means2d [N,2], grad_conics [N,3], grad_colors [N,C], grad_opacities [N], grad_background [C];
      mag_* (sums of absolute values of the same terms) and wmag_* (the same, each pixel's term weighted by the
      rounding-error weight of oracle.c, in units of 2^-22), same shapes;
      count [N] (pixels that composited each Gaussian); final_T, kappa, weight [H,W] float64; last_idx [H,W] int32
      (last composited list index, -1 if none); borderline [H,W] bool.
    mask_borderline=True differentiates with grad_image zeroed on the borderline pixels."""
    means2d, conics, colors = _f32(means2d), _f32(conics), _f32(colors)
    opacities = _f32(opacities).reshape(-1)
    background = _f32(background).reshape(-1)
    N, C = colors.shape
    assert 1 <= C <= 16
    ranges = np.ascontiguousarray(np.asarray(tile_ranges, dtype=np.int32))
    ids = np.ascontiguousarray(np.asarray(sorted_ids, dtype=np.int32))
    gimg = _f32(grad_image).reshape(H, W, C)
    V = 6 + C
    grad, mag, wmag = (np.empty((N, V), np.float64) for _ in range(3))
    count = np.empty((N,), np.int64)
    bg = np.empty((3, C), np.float64)
    final_T, kappa, weight = (np.empty((H, W), np.float64) for _ in range(3))
    last_idx = np.empty((H, W), np.int32)
    border = np.empty((H, W), np.uint8)
    lib().oracle_raster_bwd_f64(ctypes.c_int64(N), ctypes.c_int(C), _ptr(means2d), _ptr(conics), _ptr(colors),
                                _ptr(opacities), _ptr(background), _ptr(ranges), _ptr(ids), ctypes.c_int(W),
                                ctypes.c_int(H), ctypes.c_int(tile_size), _ptr(gimg),
                                ctypes.c_int(int(mask_borderline)), _ptr(grad), _ptr(mag), _ptr(wmag), _ptr(count), _ptr(bg), _ptr(final_T),
                                _ptr(last_idx), _ptr(kappa), _ptr(weight), _ptr(border))
    out = dict(count=count, final_T=final_T, last_idx=last_idx, kappa=kappa, weight=weight,
               borderline=border.astype(bool))
    for pre, arr, b in (("grad", grad, bg[0]), ("mag", mag, bg[1]), ("wmag", wmag, bg[2])):
        out[f"{pre}_means2d"] = arr[:, 0:2].copy()
        out[f"{pre}_conics"] = arr[:, 2:5].copy()
        out[f"{pre}_colors"] = arr[:, 5:5 + C].copy()
        out[f"{pre}_opacities"] = arr[:, 5 + C].copy()
        out[f"{pre}_background"] = b.copy()
    return out


def raster_audit(means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, W, H, tile_size,
                 pixels, observed, atol=1e-4, rtol=1e-4, rel_window=1e-4):
    """SURVEY H4 audit of out-of-tolerance pixels (see oracle.c: oracle_raster_audit).
    pixels [n,2] (row, col), observed [n,C] -> (explained[n] in {0: no, 1: one flip, 2: two flips, 3: already
    within tolerance}, n_borderline[n])."""
    means2d, conics, colors = _f32(means2d), _f32(conics), _f32(colors)
    opacities = _f32(opacities).reshape(-1)
    background = _f32(background).reshape(-1)
    N, C = colors.shape
    ranges = np.ascontiguousarray(np.asarray(tile_ranges, dtype=np.int32))
    ids = np.ascontiguousarray(np.asarray(sorted_ids, dtype=np.int32))
    pixels = np.ascontiguousarray(np.asarray(pixels, dtype=np.int32)).reshape(-1, 2)
    observed = _f32(observed).reshape(-1, C)
    n = pixels.shape[0]
    explained = np.zeros((n,), np.int32)
    nb = np.zeros((n,), np.int32)
    f = ctypes.c_float
    lib().oracle_raster_audit(ctypes.c_int64(N), ctypes.c_int(C), _ptr(means2d), _ptr(conics), _ptr(colors),
                              _ptr(opacities), _ptr(background), _ptr(ranges), _ptr(ids), ctypes.c_int(W),
                              ctypes.c_int(H), ctypes.c_int(tile_size), ctypes.c_int64(n), _ptr(pixels),
                              _ptr(observed), f(atol), f(rtol), f(rel_window), _ptr(explained), _ptr(nb))
    return explained, nb


def render(means3d, log_scales, quats, opacities, colors, viewmat, fx, fy, cx, cy, W, H,
           near=0.1, far=100.0, background=None, tile_size=16, semantics=SEM_TORCH,
           return_all=False):
    """Whole forward path on the CPU (render.py:63-101 order). Matches render.py:73-76:
    returns zeros (not background) when there is no intersection at all."""
    C = np.asarray(colors).shape[-1]
    bg = np.zeros((C,), np.float32) if background is None else _f32(background)
    m2, con, dep, rad = project(means3d, log_scales, quats, opacities, viewmat, fx, fy, cx, cy,
                                W, H, near, far, 0.3, semantics)
    ids, ranges = bin_tiles(m2, rad, dep, H, W, tile_size, semantics)
    if ids.size == 0:
        img, st = np.zeros((H, W, C), np.float32), (0, 0)
    else:
        img, st = rasterize(m2, con, colors, opacities, bg, ranges, ids, W, H, tile_size, True)
    if return_all:
        return dict(means2d=m2, conics=con, depths=dep, radii=rad, sorted_ids=ids,
                    tile_ranges=ranges, image=img, stats=st)
    return img
