"""Shared helpers for the parity tests (CUDA path vs oracle / golden fixtures)."""
import math

import numpy as np
import torch

import mojosplat_b200 as ms
from mojosplat_b200 import synthetic
from oracle import oracle


def camera_from_golden(g, device="cpu"):
    vm = torch.from_numpy(np.asarray(g["viewmat"], np.float32)).to(device)
    fx, fy, cx, cy = [float(v) for v in g["intr"]]
    W, H = [int(v) for v in g["size"]]
    near, far = [float(v) for v in g["clip"]]
    return ms.Camera(R=vm[:3, :3].contiguous(), T=vm[:3, 3].contiguous(), H=H, W=W, fx=fx, fy=fy, cx=cx, cy=cy,
                     near=near, far=far)


def dev(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def oracle_project_scene(sc, semantics=oracle.SEM_TORCH):
    cam = sc.camera
    return oracle.project(sc.means3d.numpy(), sc.log_scales.numpy(), sc.quats.numpy(), sc.opacities.numpy(),
                          cam.view_matrix.numpy(), cam.fx, cam.fy, cam.cx, cam.cy, cam.W, cam.H, cam.near,
                          cam.far, 0.3, semantics)


def scene_on(sc, device):
    return [t.to(device) for t in sc.gaussians()], sc.camera.to(device)


def psnr(a, b):
    mse = float(np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2))
    return 99.0 if mse == 0 else 10.0 * math.log10(1.0 / mse)


def image_gate(img, ref, frac_allowed=1e-4, atol=1e-4, rtol=1e-4, max_err_allowed=0.1 + 2e-4, audit=None):
    """SURVEY H4 gate.  `north_star`: images within 1e-4 max-abs / PSNR > 60 dB.  The alpha >= 1/255 test and the
    T (1 - alpha) <= 1e-4 stop (rasterization.mojo:143-150) make a pixel discontinuous in exp(): two correct fp32
    implementations may take different branches when a value sits within rounding distance of a threshold.  So:

    * >= (1 - frac_allowed) of the values within atol + rtol*|ref| and PSNR > 60 dB;
    * max error bounded by the largest change ONE flipped decision can cause: a skipped / added Gaussian at the alpha
      threshold moves a pixel by <= T c / 255, a flipped stop by <= alpha T c with T (1 - alpha) ~ 1e-4 and
      alpha <= 0.999, i.e. <= 0.0999 c (colours and background <= 1 here);
    * with ``audit`` (the raster inputs: dict with means2d, conics, colors, opacities, background, tile_ranges,
      sorted_ids, W, H, tile_size): EVERY out-of-tolerance pixel must be reproduced by the oracle with one (or two)
      borderline decisions forced the other way (oracle.raster_audit); anything else is a bug, not a discontinuity.
    """
    img = np.asarray(img); ref = np.asarray(ref)
    err = np.abs(img - ref)
    bad = err > (atol + rtol * np.abs(ref))
    bad_px = np.argwhere(bad.any(axis=-1))
    res = dict(frac_bad=float(bad.mean()), max_err=float(err.max()) if err.size else 0.0, psnr=psnr(img, ref),
               n_outliers=int(bad_px.shape[0]), n_unexplained=None)
    ok = bool(res["frac_bad"] <= frac_allowed and res["psnr"] > 60.0 and res["max_err"] <= max_err_allowed)
    if audit is not None and bad_px.shape[0] > 0:
        observed = img[bad_px[:, 0], bad_px[:, 1]]
        explained, n_border = oracle.raster_audit(
            audit["means2d"], audit["conics"], audit["colors"], audit["opacities"], audit["background"],
            audit["tile_ranges"], audit["sorted_ids"], audit["W"], audit["H"], audit.get("tile_size", 16),
            bad_px, observed, atol=atol, rtol=rtol)
        res["n_unexplained"] = int((explained == 0).sum())
        res["flips"] = {"one": int((explained == 1).sum()), "two": int((explained == 2).sum())}
        ok = ok and res["n_unexplained"] == 0
    elif audit is not None:
        res["n_unexplained"] = 0
    res["ok"] = ok
    return res


# rho of the per-entry backward bound (oracle.c: oracle_raster_bwd_f64), from the kernels' arithmetic: 2 x 2^-22 for the
# pair kernel (ex2.approx, lg2.approx, rcp.approx), 4 x 2^-24 for the generic kernel (libdevice expf, IEEE division)
BWD_RHO = {"fast": 2.0 * 2.0 ** -22, "faithful": 4.0 * 2.0 ** -24}
BWD_GRADS = ["means2d", "conics", "colors", "opacities", "background"]


def bwd_entry_ratios(got, ref, rho, n_pixels):
    """err / bound of every gradient entry against oracle.raster_bwd_f64's result `ref`:
    |got - ref| <= rho wmag + n_e 2^-24 mag + 1e-12, n_e the pixels that composited the Gaussian (for the background
    gradient, a torch reduction over the image: n_pixels)."""
    out = {}
    for n in BWD_GRADS:
        if n not in got:
            continue
        cnt = float(n_pixels) if n == "background" else ref["count"].astype(np.float64)
        if n in ("means2d", "conics", "colors"):
            cnt = cnt[:, None]
        bound = rho * ref[f"wmag_{n}"] + cnt * 2.0 ** -24 * ref[f"mag_{n}"] + 1e-12
        out[n] = np.abs(np.asarray(got[n], np.float64) - ref[f"grad_{n}"]) / bound
    return out


def audit_inputs(ref, sc, tile_size=16):
    """Raster inputs of an oracle.render(..., return_all=True) result, for image_gate(audit=...)."""
    return dict(means2d=ref["means2d"], conics=ref["conics"], colors=sc.colors.numpy(), opacities=sc.opacities.numpy(),
                background=sc.background.numpy(), tile_ranges=ref["tile_ranges"], sorted_ids=ref["sorted_ids"],
                W=sc.camera.W, H=sc.camera.H, tile_size=tile_size)
