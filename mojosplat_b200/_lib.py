"""ctypes binding of csrc/libbsplat.so (the C ABI declared in include/bsplat.h).

torch is plumbing here: it owns device memory and streams; every compute call goes through
the C entry points with raw pointers.  There is NO fallback: if the library is missing or the
device is not an sm_100 part, the call raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from ctypes import (POINTER, Structure, byref, c_char_p, c_float, c_int32, c_int64, c_size_t,
                    c_uint32, c_uint64, c_void_p)
from pathlib import Path

import torch

CSRC = Path(__file__).resolve().parent / "csrc"
# (BSPLAT_LIB: another build of the same library, for A/B measurements of kernel variants)
LIB_PATH = Path(os.environ["BSPLAT_LIB"]) if os.environ.get("BSPLAT_LIB") else CSRC / "libbsplat.so"

OK = 0
E_ARG, E_WORKSPACE, E_OVERFLOW, E_NODEVICE = -1, -2, -3, -4
SEM_TORCH, SEM_GSPLAT = 0, 1
RASTER_FAST, RASTER_FAITHFUL, RASTER_FAST_NOCULL = 0, 1, 2
FLAG_CAMERA_INDIRECT = 0x200
FLAG_PACKED = 0x400
FLAG_NO_BAND_PRETEST = 0x1000
PROJ_ALLOW_FMA = 0x100  # or-ed into `semantics` of bsplat_project_fwd
PROJ_FAST_MATH = 0x200  # ditto: the "within 1e-4" build (radii may be one off at integer boundaries)
BIN_PACKED = 0x100      # or-ed into `semantics` of bsplat_bin2_prepare / bsplat_bin2_finish

# every symbol include/bsplat.h declares (checked by tests/test_capi_symbols.py)
SYMBOLS = [
    "bsplat_version", "bsplat_error_string", "bsplat_check_device", "bsplat_project_fwd",
    "bsplat_bin_scan_workspace_bytes", "bsplat_bin_count_scan", "bsplat_make_key_layout",
    "bsplat_bin_emit", "bsplat_radix_sort_workspace_bytes", "bsplat_radix_sort_pairs",
    "bsplat_tile_ranges", "bsplat_rasterize_fwd", "bsplat_rasterize_stats",
    "bsplat_render_workspace_bytes", "bsplat_render_fwd", "bsplat_render_host_scratch_bytes",
    "bsplat_render_fwd_host", "bsplat_microbench", "bsplat_bin2_workspace_bytes", "bsplat_bin2_prepare",
    "bsplat_bin2_finish", "bsplat_tile_order", "bsplat_render_begin", "bsplat_render_end",
    "bsplat_render_enqueue", "bsplat_rasterize_workspace_bytes", "bsplat_rasterize_fwd_train",
    "bsplat_rasterize_fwd_train_fast", "bsplat_rasterize_bwd", "bsplat_rasterize_bwd_fast", "bsplat_render_enqueue_band", "bsplat_render_enqueue_band_p2p", "bsplat_sh_eval",
    "bsplat_project_bwd", "bsplat_sh_bwd", "bsplat_ssim_workspace_bytes", "bsplat_ssim_fwd", "bsplat_ssim_bwd",
    "bsplat_densify_workspace_bytes", "bsplat_densify_stats", "bsplat_densify_plan", "bsplat_densify_apply",
]


class BsplatCamera(Structure):
    _fields_ = [("viewmat", c_float * 16), ("fx", c_float), ("fy", c_float), ("cx", c_float),
                ("cy", c_float), ("width", c_int32), ("height", c_int32), ("near_plane", c_float),
                ("far_plane", c_float)]


class BsplatBinInfo(Structure):
    _fields_ = [("n_isect", c_uint64), ("min_depth_key", c_uint32), ("max_depth_key", c_uint32),
                ("reserved", c_uint32 * 4)]


class BsplatKeyLayout(Structure):
    _fields_ = [("depth_bias", c_uint32), ("depth_bits", c_int32), ("tile_bits", c_int32)]


class BsplatRenderAux(Structure):
    _fields_ = [("means2d", c_void_p), ("conics", c_void_p), ("depths", c_void_p), ("radii", c_void_p),
                ("tile_ranges", c_void_p), ("sorted_ids", c_void_p), ("sorted_ids_capacity", c_int64),
                ("n_isect", c_int64), ("timing", c_int32), ("n_launches", c_int32), ("sort_passes", c_int32),
                ("key_bits", c_int32), ("stage_ms", c_float * 4)]


class BsplatDensifyParams(Structure):
    _fields_ = [("grad_threshold", c_float), ("log_clone_max_scale", c_float), ("min_opacity", c_float),
                ("log_max_world_scale", c_float), ("max_screen_radius", c_int32), ("reserved", c_int32)]


class BsplatDensifyTensor(Structure):
    _fields_ = [("src", c_void_p), ("dst", c_void_p), ("width", c_int32), ("role", c_int32)]


class BsplatDensifyCounts(Structure):
    _fields_ = [("n_out", c_int64), ("n_clone", c_int64), ("n_split", c_int64), ("n_pruned", c_int64)]


DENSIFY_COPY, DENSIFY_MEANS, DENSIFY_LOG_SCALES, DENSIFY_STATE = 0, 1, 2, 3


class BsplatError(RuntimeError):
    def __init__(self, code: int, where: str):
        self.code = code
        msg = _lib.bsplat_error_string(code).decode() if _lib is not None else str(code)
        super().__init__(f"{where}: {msg} (code {code})")


_lib = None
_lock = threading.Lock()


def build(verbose: bool = False) -> Path:
    """Compile libbsplat.so in-tree with nvcc for sm_100a (no GPU needed)."""
    out = subprocess.run(["make", "-C", str(CSRC), "-j8"], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise RuntimeError("building libbsplat.so failed")
    return LIB_PATH


def load() -> ctypes.CDLL:
    """Load the library (never builds implicitly on a box without the .so: fails loudly)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make -C {CSRC}` (or __graft_entry__.build()); "
                "the CUDA backend has no CPU fallback")
        L = ctypes.CDLL(str(LIB_PATH))
        L.bsplat_version.restype = ctypes.c_int
        L.bsplat_error_string.restype = c_char_p
        L.bsplat_error_string.argtypes = [ctypes.c_int]
        L.bsplat_check_device.argtypes = [ctypes.c_int]
        L.bsplat_project_fwd.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                         POINTER(BsplatCamera), c_int32, c_float, c_int32, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p]
        L.bsplat_bin_scan_workspace_bytes.restype = c_size_t
        L.bsplat_bin_scan_workspace_bytes.argtypes = [c_int64]
        L.bsplat_bin_count_scan.argtypes = [c_int64, c_void_p, c_void_p, c_int32, c_void_p, c_int32,
                                            c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                            c_void_p, c_void_p, c_size_t, c_void_p]
        L.bsplat_make_key_layout.restype = BsplatKeyLayout
        L.bsplat_make_key_layout.argtypes = [POINTER(BsplatBinInfo), c_int32, c_int32, c_int32]
        L.bsplat_bin_emit.argtypes = [c_int64, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32,
                                      c_int32, c_int32, c_int32, c_int32, c_void_p, BsplatKeyLayout,
                                      c_void_p, c_void_p, c_void_p]
        L.bsplat_radix_sort_workspace_bytes.restype = c_size_t
        L.bsplat_radix_sort_workspace_bytes.argtypes = [c_int64, c_int32, c_int32]
        L.bsplat_radix_sort_pairs.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                              c_int32, c_void_p, c_size_t, POINTER(c_int32), c_void_p]
        L.bsplat_tile_ranges.argtypes = [c_int64, c_void_p, c_int32, c_int32, c_void_p, c_void_p]
        L.bsplat_rasterize_fwd.argtypes = [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32,
                                           c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_size_t,
                                           c_void_p]
        L.bsplat_rasterize_fwd_train.argtypes = [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                 c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p,
                                                 c_void_p, c_void_p, c_void_p]
        L.bsplat_rasterize_fwd_train_fast.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                      c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32,
                                                      c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
        L.bsplat_rasterize_bwd.argtypes = [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
        L.bsplat_rasterize_bwd_fast.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p,
                                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                                c_void_p]
        L.bsplat_rasterize_workspace_bytes.restype = c_size_t
        L.bsplat_rasterize_workspace_bytes.argtypes = [c_int64]
        L.bsplat_tile_order.argtypes = [c_int32, c_int32, c_void_p, c_void_p, c_void_p]
        L.bsplat_render_begin.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(BsplatCamera),
                                          c_int32, c_int32, c_void_p, c_size_t, c_void_p, c_void_p]
        L.bsplat_render_end.argtypes = [c_int64, c_int64, c_void_p, c_void_p, c_int32, POINTER(BsplatCamera),
                                        c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_size_t,
                                        POINTER(c_size_t), c_void_p]
        L.bsplat_render_enqueue.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                            c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p,
                                            c_void_p, c_size_t, c_int64, POINTER(c_size_t), c_void_p, c_void_p,
                                            c_void_p, c_void_p]
        L.bsplat_render_enqueue_band.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                                 c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                                 c_void_p, c_void_p, c_size_t, c_int64, POINTER(c_size_t),
                                                 c_void_p, c_void_p, c_void_p, c_void_p]
        L.bsplat_render_enqueue_band_p2p.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                                     c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                                     c_void_p, c_void_p, c_int32, c_void_p, c_size_t, c_int64,
                                                     POINTER(c_size_t), c_void_p, c_void_p, c_void_p, c_void_p]
        L.bsplat_sh_eval.argtypes = [c_int64, c_int32, c_int32, c_void_p, c_void_p, POINTER(c_float * 3), c_void_p,
                                     c_void_p]
        L.bsplat_project_bwd.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, POINTER(BsplatCamera), c_float, c_int32,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
        L.bsplat_sh_bwd.argtypes = [c_int64, c_int32, c_int32, c_void_p, c_void_p, POINTER(c_float * 3), c_void_p,
                                    c_void_p, c_void_p, c_void_p]
        L.bsplat_ssim_workspace_bytes.restype = c_size_t
        L.bsplat_ssim_workspace_bytes.argtypes = [c_int32, c_int32, c_int32]
        L.bsplat_ssim_fwd.restype = ctypes.c_int
        L.bsplat_ssim_fwd.argtypes = [c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_size_t, POINTER(c_size_t), c_void_p]
        L.bsplat_ssim_bwd.restype = ctypes.c_int
        L.bsplat_ssim_bwd.argtypes = [c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p]
        L.bsplat_densify_workspace_bytes.restype = c_size_t
        L.bsplat_densify_workspace_bytes.argtypes = [c_int64]
        L.bsplat_densify_stats.restype = ctypes.c_int
        L.bsplat_densify_stats.argtypes = [c_int64, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                           c_void_p]
        L.bsplat_densify_plan.restype = ctypes.c_int
        L.bsplat_densify_plan.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          POINTER(BsplatDensifyParams), c_void_p, c_size_t, POINTER(c_size_t),
                                          c_void_p, c_void_p]
        L.bsplat_densify_apply.restype = ctypes.c_int
        L.bsplat_densify_apply.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                           POINTER(BsplatDensifyTensor), c_void_p]
        L.bsplat_rasterize_stats.argtypes = [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32,
                                             c_int32, c_void_p, c_void_p, c_void_p]
        L.bsplat_render_workspace_bytes.restype = c_size_t
        L.bsplat_render_workspace_bytes.argtypes = [c_int64, c_int64, c_int32, c_int32, c_int32]
        L.bsplat_render_fwd.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_int32, POINTER(BsplatCamera), c_void_p, c_int32, c_int32,
                                        c_int32, c_void_p, c_void_p, c_size_t, POINTER(c_size_t),
                                        POINTER(BsplatRenderAux), c_void_p]
        L.bsplat_render_host_scratch_bytes.restype = c_size_t
        L.bsplat_render_host_scratch_bytes.argtypes = [c_int64, c_int32, c_int32, c_int32]
        L.bsplat_render_fwd_host.argtypes = [c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_int32, POINTER(BsplatCamera), c_void_p, c_int32, c_int32,
                                             c_int32, c_void_p, c_void_p, c_size_t, c_void_p, c_size_t,
                                             POINTER(c_size_t), POINTER(BsplatRenderAux), c_void_p]
        L.bsplat_microbench.argtypes = [c_int32, c_int32, c_int32, c_void_p, c_void_p]
        L.bsplat_bin2_workspace_bytes.restype = c_size_t
        L.bsplat_bin2_workspace_bytes.argtypes = [c_int64, c_int64, c_int64]
        L.bsplat_bin2_prepare.argtypes = [c_int64, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32,
                                          c_int32, c_int32, c_int32, c_int32, c_void_p, c_size_t, c_void_p,
                                          c_void_p]
        L.bsplat_bin2_finish.argtypes = [c_int64, c_int64, c_void_p, c_void_p, c_int32, c_int32, c_int32,
                                         c_int32, c_int32, c_int32, c_int32, c_void_p, c_size_t, c_void_p,
                                         c_void_p, c_void_p, c_void_p]
        _lib = L
    return _lib


_checked_devices: set = set()


def require_device(device: torch.device) -> ctypes.CDLL:
    """Library + an sm_100 device, or an exception. No CPU path exists."""
    if device.type != "cuda":
        raise RuntimeError("the 'cuda' backend needs CUDA tensors; there is no CPU fallback "
                           f"(got device '{device}')")
    L = load()
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _checked_devices:
        rc = L.bsplat_check_device(idx)
        if rc != OK:
            raise BsplatError(rc, "bsplat_check_device")
        _checked_devices.add(idx)
    return L


def check(rc: int, where: str) -> None:
    if rc != OK:
        raise BsplatError(rc, where)


def stream_ptr(device: torch.device) -> c_void_p:
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t: torch.Tensor | None) -> c_void_p:
    if t is None or t.numel() == 0:
        return c_void_p(0)
    return c_void_p(t.data_ptr())


def camera_struct(camera) -> BsplatCamera:
    """POD copy of a Camera (utils.py). Cached on the object; the view matrix and the intrinsics matrix are read
    back from the device once per (tensor, version).  Like the reference (projection.py:137-140, 156-159) the
    intrinsics come from ``camera.Ks``, not from the scalar fields; a Ks that is not a plain pinhole matrix
    (skew, or a last row other than [0, 0, 1]) has no counterpart in the C ABI and is rejected."""
    vm = camera.view_matrix
    ks = camera.Ks
    key = (vm.data_ptr(), vm._version, ks.data_ptr(), ks._version, camera.H, camera.W, camera.near, camera.far)
    cached = getattr(camera, "_bsplat_cam", None)
    if cached is not None and cached[0] == key:
        return cached[1]
    c = BsplatCamera()
    flat = vm.detach().to(device="cpu", dtype=torch.float32).reshape(16).tolist()
    for k in range(16):
        c.viewmat[k] = flat[k]
    K = ks.detach().to(device="cpu", dtype=torch.float32).reshape(3, 3).tolist()
    if K[0][1] != 0.0 or K[1][0] != 0.0 or K[2] != [0.0, 0.0, 1.0]:
        raise ValueError("camera.Ks must be a pinhole matrix [[fx, 0, cx], [0, fy, cy], [0, 0, 1]] for the CUDA backend")
    c.fx, c.fy, c.cx, c.cy = K[0][0], K[1][1], K[0][2], K[1][2]
    c.width, c.height = int(camera.W), int(camera.H)
    c.near_plane, c.far_plane = float(camera.near), float(camera.far)
    try:
        object.__setattr__(camera, "_bsplat_cam", (key, c))
    except Exception:
        pass
    return c


class Workspace:
    """Grow-only byte buffer per (device, CUDA stream, tag), allocated from torch's caching allocator.  The stream is
    part of the key: two renders issued on different streams of one device must not share scratch memory."""

    def __init__(self):
        self._bufs: dict = {}

    @staticmethod
    def key(device: torch.device, tag: str):
        idx = device.index if device.index is not None else torch.cuda.current_device()
        return (idx, int(torch.cuda.current_stream(device).cuda_stream), tag)

    def get(self, device: torch.device, tag: str, nbytes: int) -> torch.Tensor:
        key = self.key(device, tag)
        buf = self._bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            grow = int(nbytes * 1.25) if buf is not None else int(nbytes)
            self._bufs[key] = buf = torch.empty(max(grow, 256), dtype=torch.uint8, device=device)
        return buf

    def put(self, device: torch.device, tag: str, buf: torch.Tensor) -> None:
        self._bufs[self.key(device, tag)] = buf

    def clear(self):
        self._bufs.clear()


workspace = Workspace()


def as_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if t.dtype != torch.float32:
        t = t.to(torch.float32)
    return t.contiguous()
