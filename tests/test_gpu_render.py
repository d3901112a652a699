"""GPU: end-to-end render_gaussians (fused C path) vs the oracle; API behaviour of render.py."""
import numpy as np
import pytest
import torch

import mojosplat_b200 as ms
from helpers import audit_inputs, image_gate, scene_on
from mojosplat_b200 import binning, synthetic
from oracle import oracle

pytestmark = pytest.mark.gpu


def oracle_render(sc, **kw):
    cam = sc.camera
    return oracle.render(sc.means3d.numpy(), sc.log_scales.numpy(), sc.quats.numpy(), sc.opacities.numpy(),
                         sc.colors.numpy(), cam.view_matrix.numpy(), cam.fx, cam.fy, cam.cx, cam.cy, cam.W, cam.H,
                         cam.near, cam.far, background=sc.background.numpy(), return_all=True, **kw)


@pytest.mark.parametrize("cfg,N", [("config1_1k_256", None), ("config2_100k_1080p", 20_000),
                                   ("config3_1m_1080p", 200_000), ("config3_1m_1080p", 1_000_000)])
def test_render_end_to_end_vs_oracle_and_single_level(cuda_device, cfg, N):
    sc = synthetic.make_scene(cfg, N=N)
    ref = oracle_render(sc)
    (m, s, q, o, c), cam = scene_on(sc, cuda_device)
    img = ms.render_gaussians(m, s, q, o, c, cam, background_color=sc.background.to(cuda_device), backend="cuda")
    assert img.shape == (cam.H, cam.W, 3) and img.dtype == torch.float32 and img.device.type == "cuda"
    # end to end the projected values differ from the oracle's in the last bits (libdevice vs glibc expf, conic
    # reciprocal), so a few more threshold decisions flip than with identical raster inputs: every one is audited
    r = image_gate(img.cpu().numpy(), ref["image"], frac_allowed=2e-4, audit=audit_inputs(ref, sc))
    assert r["ok"], r
    # stage outputs of the fused path: binning must be bit-exact when the projected inputs agree
    img2, aux = ms.render_fused(m, s, q, o, c, cam, sc.background.to(cuda_device), return_aux=True)
    assert torch.equal(img, img2)
    # the frame's two-level lists equal the stand-alone single-level binning of its own stage outputs
    ids1, ranges1 = binning.bin_gaussians_to_tiles_cuda(aux["means2d"], aux["radii"], aux["depths"], cam.H, cam.W, 16,
                                                        algo="single")
    assert torch.equal(aux["tile_ranges"], ranges1)
    assert aux["sorted_ids"] is not None and torch.equal(aux["sorted_ids"], ids1)
    assert aux["n_isect"] == ref["sorted_ids"].shape[0] or abs(aux["n_isect"] - ref["sorted_ids"].shape[0]) <= 8
    if np.array_equal(aux["radii"].cpu().numpy(), ref["radii"]) and \
            np.array_equal(aux["means2d"].cpu().numpy(), ref["means2d"]):
        assert np.array_equal(aux["tile_ranges"].cpu().numpy(), ref["tile_ranges"])


def test_render_host_path_equals_device_path(cuda_device):
    sc = synthetic.make_scene("config1_1k_256")
    (m, s, q, o, c), cam = scene_on(sc, cuda_device)
    img = ms.render_gaussians(m, s, q, o, c, cam, background_color=sc.background.to(cuda_device))
    host = ms.render_gaussians_host(*sc.gaussians(), sc.camera, background_color=sc.background)
    assert not host.is_cuda and torch.equal(host, img.cpu())


def test_render_api_behaviour(cuda_device):
    sc = synthetic.make_scene("config1_1k_256", N=64)
    (m, s, q, o, c), cam = scene_on(sc, cuda_device)
    with pytest.raises(ValueError, match="CUDA tensors"):
        ms.render_gaussians(m.cpu(), s, q, o, c, cam)                      # render.py:44-46
    with pytest.raises(ValueError, match="Background color channels"):
        ms.render_gaussians(m, s, q, o, c, cam, background_color=torch.zeros(4))  # render.py:57-58
    with pytest.raises(ValueError, match="Invalid backend"):
        ms.render_gaussians(m, s, q, o, c, cam, backend="nope")
    img = ms.render_gaussians(m, s, q, o, c, cam, background_color=[0.1, 0.1, 0.1])  # non-tensor background
    assert img.shape == (cam.H, cam.W, 3)
    img0 = ms.render_gaussians(m, s, q, o, c, cam)                           # default background zeros
    assert torch.isfinite(img0).all()
    # empty scene -> all zeros, not background (render.py:73-76)
    far = m.clone(); far[:, 2] += 1e6
    z = lambda *sh: torch.zeros(*sh, device=cuda_device)
    with pytest.warns(UserWarning):
        e = ms.render_gaussians(z(0, 3), z(0, 3), z(0, 4), z(0), z(0, 3), cam, background_color=torch.ones(3))
    assert (e == 0).all()


def test_render_single_gaussian_centre(cuda_device):
    """tests/test_render.py:60-86 with a camera that sees the scene (SURVEY section 4 caveat)."""
    cam = ms.Camera(R=torch.eye(3, device=cuda_device), T=torch.tensor([0.0, 0.0, 5.0], device=cuda_device),
                    H=64, W=64, fx=100.0, fy=100.0, cx=32.0, cy=32.0)
    d = lambda a: torch.tensor(a, dtype=torch.float32, device=cuda_device)
    img = ms.render_gaussians(d([[0.0, 0.0, 0.0]]), torch.log(d([[0.3, 0.3, 0.3]])), d([[1.0, 0, 0, 0]]), d([0.9]),
                              d([[1.0, 0.0, 0.0]]), cam, background_color=d([0.0, 0.0, 1.0]))
    assert img[32, 32, 0] > 0.5
    for y, x in ((0, 0), (0, 63), (63, 0), (63, 63)):
        assert (img[y, x] - d([0.0, 0.0, 1.0])).abs().max() < 1e-2
