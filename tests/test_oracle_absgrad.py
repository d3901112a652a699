"""CPU: the fp64 reference of AbsGS's absolute screen-space gradient (gsplat's ``absgrad``; absgrad_ref.c) against fp64
torch autograd, its agreement with oracle.raster_bwd_f64, and its invariants.  No GPU.

The autograd side does not share the reference's arithmetic: it restates test_gpu_raster_bwd.torch_raster with pixel p
reading ``means2d[g] + delta[p, g]``, delta a zero [H, W, N, 2] leaf, so d L / d delta[p, g] is exactly pixel p's term
of d L / d means2d[g], and sum_p |d L / d delta[p, g]| is the definition of the absolute gradient."""
import numpy as np
import pytest
import torch

from absgrad_ref import raster_abs_means2d_f64
from oracle import oracle
from test_gpu_raster_bwd import small_scene
from test_oracle_raster_bwd import AUTOGRAD_CASES


def torch_raster_per_pixel_means(means2d, delta, conics, colors, opac, bg, ranges, ids, H, W, ts):
    """torch_raster with the mean of Gaussian g seen by pixel (y, x) equal to means2d[g] + delta[y, x, g]."""
    C = colors.shape[1]
    image = torch.zeros((H, W, C), dtype=means2d.dtype)
    th, tw = ranges.shape[:2]
    for ty in range(th):
        for tx in range(tw):
            y0, x0 = ty * ts, tx * ts
            y1, x1 = min(y0 + ts, H), min(x0 + ts, W)
            ys = torch.arange(y0, y1, dtype=means2d.dtype) + 0.5
            xs = torch.arange(x0, x1, dtype=means2d.dtype) + 0.5
            py, px = torch.meshgrid(ys, xs, indexing="ij")
            T = torch.ones_like(px)
            out = torch.zeros(px.shape + (C,), dtype=means2d.dtype)
            done = torch.zeros_like(px, dtype=torch.bool)
            for k in range(int(ranges[ty, tx, 0]), int(ranges[ty, tx, 1])):
                g = int(ids[k])
                d = delta[y0:y1, x0:x1, g]
                dx, dy = means2d[g, 0] + d[..., 0] - px, means2d[g, 1] + d[..., 1] - py
                a, b, c = conics[g, 0], conics[g, 1], conics[g, 2]
                sigma = 0.5 * (a * dx * dx + c * dy * dy) + b * dx * dy
                alpha = torch.clamp(opac[g] * torch.exp(-sigma), max=0.999)
                valid = (sigma >= 0) & (alpha >= 1.0 / 255.0) & ~done
                nT = T * (1 - alpha)
                stop = valid & (nT <= 1e-4)
                done = done | stop
                add = valid & ~stop
                out = out + torch.where(add, alpha * T, torch.zeros_like(T)).unsqueeze(-1) * colors[g]
                T = torch.where(add, nT, T)
            image[y0:y1, x0:x1] = out + T.unsqueeze(-1) * bg
    return image


def _autograd_abs(m2, con, c, o, bg, ranges, ids, H, W, ts, gimg):
    """-> (sum_p |d L / d means2d_p|, d L / d means2d) in fp64, L = sum(image * gimg)."""
    t64 = [torch.tensor(x, dtype=torch.float64, requires_grad=True) for x in (m2, con, c, o, bg)]
    delta = torch.zeros((H, W, m2.shape[0], 2), dtype=torch.float64, requires_grad=True)
    img = torch_raster_per_pixel_means(t64[0], delta, *t64[1:], ranges, ids, H, W, ts)
    (img * torch.as_tensor(gimg, dtype=torch.float64)).sum().backward()
    return delta.grad.abs().sum(dim=(0, 1)).numpy(), t64[0].grad.numpy()


def _check(ref, got, signed, want_abs, want_grad):
    """ref: oracle.raster_bwd_f64's result; got, signed: raster_abs_means2d_f64's on the same inputs."""
    mag = ref["mag_means2d"]
    assert got.shape == want_abs.shape == (ref["count"].shape[0], 2)
    # the reference's abs sum against autograd, relative to the sum of magnitudes (as test_oracle_raster_bwd)
    err = np.abs(got - want_abs)
    assert (err <= 1e-10 * mag + 1e-300).all(), float((err / np.maximum(mag, 1e-300)).max())
    # the per-pixel sum of the signed terms is the ordinary gradient, and the same walk as the oracle's
    assert (np.abs(want_grad - ref["grad_means2d"]) <= 1e-10 * mag + 1e-300).all()
    assert (np.abs(signed - ref["grad_means2d"]) <= 1e-12 * mag + 1e-300).all()
    # invariants: |sum| <= sum |.| <= the sum of the termwise magnitudes; nothing where nothing was composited
    g = np.abs(ref["grad_means2d"])
    assert (got >= g * (1 - 1e-12)).all()
    assert (got <= mag * (1 + 1e-12)).all()
    assert (got[ref["count"] == 0] == 0).all()
    assert (got >= 0).all()


@pytest.mark.parametrize("N,HW,ts,C,seed", AUTOGRAD_CASES)
def test_abs_means2d_matches_autograd(N, HW, ts, C, seed):
    cam, m2, con, dep, rad, o, c = small_scene(N, HW, seed, C)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, HW, HW, ts)
    bg = np.linspace(0.1, 0.4, C).astype(np.float32)
    gimg = torch.randn(HW, HW, C, generator=torch.Generator().manual_seed(100 + seed)).numpy()
    want_abs, want_grad = _autograd_abs(m2, con, c, o, bg, ranges, ids, HW, HW, ts, gimg)
    ref = oracle.raster_bwd_f64(m2, con, c, o, bg, ranges, ids, HW, HW, ts, gimg)
    got, signed = raster_abs_means2d_f64(m2, con, c, o, bg, ranges, ids, HW, HW, ts, gimg)
    _check(ref, got, signed, want_abs, want_grad)
    assert got.max() > 0
    if N > 1:
        # a random upstream cancels: the absolute sum exceeds the signed one somewhere by a wide margin
        assert (got > 2.0 * np.abs(ref["grad_means2d"])).any()


def test_abs_means2d_saturated_stack_matches_autograd():
    """The opaque stack of test_oracle_raster_bwd: early stops and the 0.999 clamp (no gradient through it)."""
    N, HW = 60, 32
    g = torch.Generator().manual_seed(11)
    m2 = (torch.rand(N, 2, generator=g) * 12 + 10).numpy().astype(np.float32)
    con = np.tile(np.array([[0.02, 0.0, 0.02]], np.float32), (N, 1))
    dep = np.arange(N, dtype=np.float32) + 1
    rad = np.full((N, 2), 40, np.int32)
    o = np.full(N, 1.0, np.float32); o[::3] = 0.9
    c = torch.rand(N, 3, generator=g).numpy()
    ids, ranges = oracle.bin_tiles(m2, rad, dep, HW, HW, 16)
    bg = np.array([0.5, 0.5, 0.5], np.float32)
    for gimg in (np.ones((HW, HW, 3), np.float32),
                 torch.randn(HW, HW, 3, generator=torch.Generator().manual_seed(12)).numpy()):
        want_abs, want_grad = _autograd_abs(m2, con, c, o, bg, ranges, ids, HW, HW, 16, gimg)
        ref = oracle.raster_bwd_f64(m2, con, c, o, bg, ranges, ids, HW, HW, 16, gimg)
        _check(ref, *raster_abs_means2d_f64(m2, con, c, o, bg, ranges, ids, HW, HW, 16, gimg), want_abs, want_grad)


def test_abs_means2d_masking_by_zeroed_upstream():
    """Borderline pixels are left out by zeroing them in grad_image: the signed sums then equal the oracle's with
    mask_borderline=True, on a scene where the flag fires."""
    cam, m2, con, dep, rad, o, c = small_scene(60, 64, 7)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, 64, 64, 32)
    bg = np.linspace(0.1, 0.4, 3).astype(np.float32)
    gimg = torch.randn(64, 64, 3, generator=torch.Generator().manual_seed(107)).numpy()
    ref = oracle.raster_bwd_f64(m2, con, c, o, bg, ranges, ids, 64, 64, 32, gimg, mask_borderline=True)
    assert ref["borderline"].any()
    gm = np.where(ref["borderline"][..., None], np.float32(0), gimg)
    got, signed = raster_abs_means2d_f64(m2, con, c, o, bg, ranges, ids, 64, 64, 32, gm)
    assert (np.abs(signed - ref["grad_means2d"]) <= 1e-12 * ref["mag_means2d"] + 1e-300).all()
    assert (got <= ref["mag_means2d"] * (1 + 1e-12)).all()

