"""ctypes front-end of absgrad_ref.c, the fp64 reference of AbsGS's absolute screen-space gradient.  TEST
INFRASTRUCTURE ONLY.

The shared library is compiled with gcc on first use (seconds) into the system temporary directory, keyed by a hash of
the source, so the repository tree is never written to."""
import ctypes
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_SRC = Path(__file__).resolve().with_name("absgrad_ref.c")
_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        src = _SRC.read_bytes()
        out_dir = Path(tempfile.gettempdir()) / f"bsplat_absgrad_ref_{os.getuid()}"
        out_dir.mkdir(exist_ok=True)
        so = out_dir / f"absgrad_ref_{hashlib.sha1(src).hexdigest()[:16]}.so"
        if not so.exists():
            tmp = out_dir / f"{so.name}.{os.getpid()}.tmp"
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC", "-std=c99",
                                   "-o", str(tmp), str(_SRC), "-lm"])
            os.replace(tmp, so)
        _lib = ctypes.CDLL(str(so))
    return _lib


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(ctypes.c_void_p)


def raster_abs_means2d_f64(means2d, conics, colors, opacities, background, tile_ranges, sorted_ids, W, H, tile_size,
                           grad_image):
    """-> (abs_means2d [N,2], signed_means2d [N,2]) float64 for the upstream gradient grad_image [H, W, C]: per
    Gaussian, the sum over the pixels it was composited at of |d L_p / d means2d| and of d L_p / d means2d.  To leave
    out oracle.raster_bwd_f64's borderline pixels, pass grad_image with them zeroed."""
    means2d, conics, colors = _f32(means2d), _f32(conics), _f32(colors)
    opacities = _f32(opacities).reshape(-1)
    background = _f32(background).reshape(-1)
    N, C = colors.shape
    assert 1 <= C <= 16
    ranges = np.ascontiguousarray(np.asarray(tile_ranges, dtype=np.int32))
    ids = np.ascontiguousarray(np.asarray(sorted_ids, dtype=np.int32))
    gimg = _f32(grad_image).reshape(H, W, C)
    out_abs, out_signed = np.empty((N, 2), np.float64), np.empty((N, 2), np.float64)
    lib().absgrad_ref_f64(ctypes.c_int64(N), ctypes.c_int(C), _ptr(means2d), _ptr(conics), _ptr(colors),
                          _ptr(opacities), _ptr(background), _ptr(ranges), _ptr(ids), ctypes.c_int(W), ctypes.c_int(H),
                          ctypes.c_int(tile_size), _ptr(gimg), _ptr(out_abs), _ptr(out_signed))
    return out_abs, out_signed
