"""CPU: the fp64 compositing backward of the oracle (oracle.raster_bwd_f64) against fp64 torch autograd through the
pure-torch restatement of the forward (test_gpu_raster_bwd.torch_raster), its invariants, and its borderline flag on
constructed pixels.  No GPU: this anchors the reference the full-size GPU parity tests (test_gpu_raster_bwd_full.py)
bound every gradient entry against."""
import numpy as np
import pytest
import torch

from helpers import oracle_project_scene
from mojosplat_b200 import synthetic
from oracle import oracle
from test_gpu_raster_bwd import small_scene, torch_raster

NAMES = ["means2d", "conics", "colors", "opacities", "background"]

# every parameter set of test_gpu_raster_bwd.test_backward_matches_torch_autograd
AUTOGRAD_CASES = [(1, 32, 16, 3, 0), (40, 48, 16, 3, 1), (150, 64, 16, 3, 2), (60, 40, 10, 3, 3), (80, 48, 16, 1, 4),
                  (80, 48, 16, 4, 5), (400, 32, 16, 3, 6), (80, 42, 16, 3, 12), (120, 57, 16, 3, 13),
                  (60, 64, 32, 3, 7), (60, 64, 32, 4, 8), (60, 62, 31, 3, 9), (60, 64, 32, 2, 10)]


def _autograd(m2, con, c, o, bg, ranges, ids, H, W, ts, gimg):
    t64 = [torch.tensor(x, dtype=torch.float64, requires_grad=True) for x in (m2, con, c, o, bg)]
    img = torch_raster(*t64, ranges, ids, H, W, ts)
    (img * torch.as_tensor(gimg, dtype=torch.float64)).sum().backward()
    return img.detach().numpy(), [t.grad.numpy() for t in t64]


def _assert_matches(ref, want, rel=1e-10):
    for name, w in zip(NAMES, want):
        got, mag = ref[f"grad_{name}"], ref[f"mag_{name}"]
        assert got.shape == w.shape, name
        err = np.abs(got - w)
        bound = rel * mag + 1e-300
        assert (err <= bound).all(), (name, float((err / np.maximum(mag, 1e-300)).max()))


def _check_invariants(ref):
    for name in NAMES:
        g, m, wm = ref[f"grad_{name}"], ref[f"mag_{name}"], ref[f"wmag_{name}"]
        assert (m >= np.abs(g) * (1 - 1e-12)).all(), name
        assert (wm >= m).all(), name   # every weight is >= 2
    assert (ref["kappa"] >= 0).all()
    assert (ref["weight"] >= 0).all()
    assert (ref["count"] >= 0).all()


@pytest.mark.parametrize("N,HW,ts,C,seed", AUTOGRAD_CASES)
def test_raster_bwd_f64_matches_autograd(N, HW, ts, C, seed):
    cam, m2, con, dep, rad, o, c = small_scene(N, HW, seed, C)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, HW, HW, ts)
    bg = np.linspace(0.1, 0.4, C).astype(np.float32)
    gimg = torch.randn(HW, HW, C, generator=torch.Generator().manual_seed(100 + seed)).numpy()
    img, want = _autograd(m2, con, c, o, bg, ranges, ids, HW, HW, ts, gimg)
    ref = oracle.raster_bwd_f64(m2, con, c, o, bg, ranges, ids, HW, HW, ts, gimg)
    _assert_matches(ref, want)
    _check_invariants(ref)
    assert np.abs(ref["grad_means2d"]).max() > 0 or N == 0
    # final T: image = composite + T bg, so T is recovered from a zero-colour forward
    zero_c = np.zeros_like(c)
    t_img = oracle.rasterize_f64(m2, con, zero_c, o, np.ones(C, np.float32), ranges, ids, HW, HW, ts)
    np.testing.assert_allclose(ref["final_T"], t_img[..., 0], rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(img, oracle.rasterize_f64(m2, con, c, o, bg, ranges, ids, HW, HW, ts),
                               rtol=1e-12, atol=1e-15)


def test_raster_bwd_f64_saturated_stack_matches_autograd():
    """The opaque stack of test_gpu_raster_bwd.test_backward_saturated_pixels_and_clamp: early stops and the clamp."""
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
        _, want = _autograd(m2, con, c, o, bg, ranges, ids, HW, HW, 16, gimg)
        ref = oracle.raster_bwd_f64(m2, con, c, o, bg, ranges, ids, HW, HW, 16, gimg)
        _assert_matches(ref, want)
        _check_invariants(ref)
    # the stack saturates: some pixels stop before the end of their list, and the clamp zeroes some opacity terms
    r1 = ranges[..., 1].repeat(16, 0).repeat(16, 1)[:HW, :HW]
    assert (ref["last_idx"] < r1 - 1).sum() > 100
    assert ref["final_T"].min() < 1e-3


def _one_gaussian_pixel(opacity, mean=(8.5 + 1.5, 8.5), conic=(1.0, 0.0, 1.0), HW=16):
    m2 = np.array([mean], np.float32)
    con = np.array([conic], np.float32)
    o = np.array([opacity], np.float32)
    c = np.array([[0.3, 0.6, 0.9]], np.float32)
    ids = np.zeros((1,), np.int32)
    ranges = np.array([[[0, 1]]], np.int32)
    gimg = np.ones((HW, HW, 3), np.float32)
    return oracle.raster_bwd_f64(m2, con, c, o, np.zeros(3, np.float32), ranges, ids, HW, HW, 16, gimg)


@pytest.mark.parametrize("rel", [1e-6, -1e-6])
def test_borderline_alpha_threshold(rel):
    # alpha = o exp(-sigma) = (1/255)(1 + rel) at pixel (8, 8): dx = 1.5, dy = 0, sigma = 1.125
    o = np.float32(np.exp(1.125) / 255.0 * (1.0 + rel))
    ref = _one_gaussian_pixel(o)
    assert ref["borderline"][8, 8]
    assert ref["borderline"].sum() <= 4
    # a clear margin is not borderline
    o = np.float32(np.exp(1.125) / 255.0 * (1.0 + 1e3 * rel))
    assert not _one_gaussian_pixel(o)["borderline"][8, 8]


@pytest.mark.parametrize("rel", [5e-7, -5e-7])
def test_borderline_clamp(rel):
    # the mean on the pixel centre (sigma = 0): alpha = o, just under and over 0.999 (the window there is
    # 2 e u = 2 (2 - ln 0.999) 2^-22 ~ 9.5e-7 in log space)
    o = np.float32(0.999 * (1.0 + rel))
    ref = _one_gaussian_pixel(o, mean=(8.5, 8.5))
    assert ref["borderline"][8, 8]
    assert ref["borderline"].sum() == 1
    clamped = np.float32(0.999 * (1.0 + 1e3 * rel))
    assert not _one_gaussian_pixel(clamped, mean=(8.5, 8.5))["borderline"][8, 8]


@pytest.mark.parametrize("eps", [1e-6, -1e-6])
def test_borderline_early_stop(eps):
    # four Gaussians centred on pixel (8, 8) (sigma = 0, alpha = o): T after the fourth lands on 1e-4 (1 + eps)
    def stack(eps):
        o = np.array([0.9, 0.9, 0.9, 0.0], np.float32)
        T3 = float(np.prod(1.0 - o[:3].astype(np.float64)))
        o[3] = np.float32(1.0 - 1e-4 * (1.0 + eps) / T3)
        m2 = np.full((4, 2), 8.5, np.float32)
        con = np.tile(np.array([[0.5, 0.0, 0.5]], np.float32), (4, 1))
        c = np.full((4, 3), 0.5, np.float32)
        ranges = np.array([[[0, 4]]], np.int32)
        return oracle.raster_bwd_f64(m2, con, c, o, np.zeros(3, np.float32), ranges, np.arange(4, dtype=np.int32),
                                     16, 16, 16, np.ones((16, 16, 3), np.float32))
    ref = stack(eps)
    assert ref["borderline"][8, 8]
    assert ref["last_idx"][8, 8] == (3 if eps > 0 else 2)
    far = stack(1e4 * eps)
    assert not far["borderline"][8, 8]


def test_borderline_rare_on_generic_scene():
    sc = synthetic.make_scene("config1_1k_256")
    cam = sc.camera
    m2, con, dep, rad = oracle_project_scene(sc)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, cam.H, cam.W, 16)
    gimg = torch.randn(cam.H, cam.W, 3, generator=torch.Generator().manual_seed(1)).numpy()
    ref = oracle.raster_bwd_f64(m2, con, sc.colors.numpy(), sc.opacities.numpy(), sc.background.numpy(), ranges, ids,
                                cam.W, cam.H, 16, gimg)
    frac = float(ref["borderline"].mean())
    print(f"\n[config1] borderline fraction {frac:.2e}, max kappa {ref['kappa'].max():.1f}")
    assert frac < 1e-3
    _check_invariants(ref)
    # masking: borderline pixels contribute nothing, the rest is unchanged (the backward is linear in grad_image)
    masked = oracle.raster_bwd_f64(m2, con, sc.colors.numpy(), sc.opacities.numpy(), sc.background.numpy(), ranges,
                                   ids, cam.W, cam.H, 16, gimg, mask_borderline=True)
    g0 = gimg.copy(); g0[ref["borderline"]] = 0
    again = oracle.raster_bwd_f64(m2, con, sc.colors.numpy(), sc.opacities.numpy(), sc.background.numpy(), ranges,
                                  ids, cam.W, cam.H, 16, g0)
    for name in NAMES:
        np.testing.assert_allclose(masked[f"grad_{name}"], again[f"grad_{name}"], rtol=1e-12,
                                   atol=1e-12 * float(np.abs(again[f"mag_{name}"]).max()))
