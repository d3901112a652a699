"""Photometric training loss (ssim, l1_dssim_loss; bsplat_ssim_fwd / bsplat_ssim_bwd) against fp64 torch autograd.

The oracle is autograd through a pure-torch restatement of 3DGS's ``ssim`` (grouped ``F.conv2d`` with the normalised
11x11 Gaussian window, ``padding=5``) plus ``abs().mean()``, evaluated in float64: no hand-derived formula on the
checking side.  The argument checks at the top need no GPU.
"""
import math

import pytest
import torch
import torch.nn.functional as F

import mojosplat_b200 as ms
from mojosplat_b200 import _lib
from mojosplat_b200.loss import ssim_l1
from test_gpu_train import e2e_scene


def gaussian_window(C, dtype, device):
    g = torch.tensor([math.exp(-(x - 5) ** 2 / float(2 * 1.5 ** 2)) for x in range(11)], dtype=dtype)
    g = g / g.sum()
    w2 = g[:, None] @ g[None, :]
    return w2.expand(C, 1, 11, 11).contiguous().to(device)


def torch_ssim_l1(img, target):
    """3DGS's ssim (loss_utils.py: _ssim with size_average) on (H, W, C) images, and mean |img - target|."""
    C = img.shape[-1]
    x, y = img.permute(2, 0, 1)[None], target.permute(2, 0, 1)[None]
    w = gaussian_window(C, img.dtype, img.device)
    conv = lambda t: F.conv2d(t, w, padding=5, groups=C)  # noqa: E731
    mu1, mu2 = conv(x), conv(y)
    mu1_sq, mu2_sq, mu1_mu2 = mu1 * mu1, mu2 * mu2, mu1 * mu2
    sigma1_sq = conv(x * x) - mu1_sq
    sigma2_sq = conv(y * y) - mu2_sq
    sigma12 = conv(x * y) - mu1_mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    ssim_map = ((2 * mu1_mu2 + C1) * (2 * sigma12 + C2)) / ((mu1_sq + mu2_sq + C1) * (sigma1_sq + sigma2_sq + C2))
    return ssim_map.mean(), (img - target).abs().mean()


UPSTREAMS = {
    "ssim": lambda s, l: s,
    "l1_dssim": lambda s, l: 0.8 * l + 0.2 * (1.0 - s),
    "mixed": lambda s, l: 2.0 * s - 3.0 * l,
}


def grad_err(got, want):
    """Max |got - want| over max|want|, but at least over 1 / (HWC): the natural scale of the gradient of a mean (the
    gradient of ssim(x, x) is ~0, and a relative error against ~0 means nothing)."""
    return float((got.double() - want).abs().max()) / max(float(want.abs().max()), 1.0 / want.numel())


def compare(img, target):
    """Max errors of the fused loss against fp64 autograd: (scalar error, {upstream: gradient error, see grad_err})."""
    x64 = img.detach().double().requires_grad_(True)
    s64, l64 = torch_ssim_l1(x64, target.double())
    errs = {}
    x = img.detach().clone().requires_grad_(True)
    s, l = ssim_l1(x, target)
    scalar_err = max(abs(float(s.detach()) - float(s64.detach())), abs(float(l.detach()) - float(l64.detach())))
    for name, fn in UPSTREAMS.items():
        (gw,) = torch.autograd.grad(fn(s64, l64), x64, retain_graph=True)
        x.grad = None
        s, l = ssim_l1(x, target)
        fn(s, l).backward()
        errs[name] = grad_err(x.grad, gw)
    # the public wrappers are the same Function
    xs = img.detach().clone().requires_grad_(True)
    ms.ssim(xs, target).backward()
    (gw,) = torch.autograd.grad(s64, x64, retain_graph=True)
    errs["ssim()"] = grad_err(xs.grad, gw)
    xl = img.detach().clone().requires_grad_(True)
    ms.l1_dssim_loss(xl, target).backward()
    (gw,) = torch.autograd.grad(0.8 * l64 + 0.2 * (1.0 - s64), x64)
    errs["l1_dssim_loss()"] = grad_err(xl.grad, gw)
    return scalar_err, errs


# fp32 against fp64.  Measured on a B200 (1000 W): random images <= 4.2e-8 on the scalars and <= 1.6e-6 on the gradients
# (1080p), renders <= 1.5e-7 and <= 1.6e-5.
SCALAR_TOL = 1e-5
GRAD_TOL = 1e-4
# Constant images are ill-conditioned in fp32: sigma^2 = E[x^2] - mu^2 cancels to ~1e-8, which only C2 = 9e-4 holds
# off, so S and its gradient carry relative errors near 1e-5 / 1e-4.  torch's own fp32 evaluation of the same formula
# is 5.1e-5 off on the 0.2 / 0.7 pair below; the fused kernels measured 2.1e-5 there and 1.6e-4 on a gradient.
CONST_SCALAR_TOL = 1e-4
CONST_GRAD_TOL = 1e-3


# ---------------------------------------------------------------- argument checks (no GPU) --------------------------

def test_workspace_query_needs_no_gpu():
    L = _lib.load() if _lib.LIB_PATH.exists() else None
    if L is None:
        pytest.skip("libbsplat.so not built")
    assert L.bsplat_ssim_workspace_bytes(1080, 1920, 3) == 60 * 34 * 8
    assert L.bsplat_ssim_workspace_bytes(1, 1, 1) == 8
    assert L.bsplat_ssim_workspace_bytes(8, 8, 5) == 0 and L.bsplat_ssim_workspace_bytes(0, 8, 3) == 0


def test_arguments_rejected():
    a = torch.rand(8, 9, 3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ms.ssim(a, a.clone())
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ms.l1_dssim_loss(a.clone().requires_grad_(True), a)
    with pytest.raises(ValueError, match="H, W, C"):
        ms.ssim(a, torch.rand(8, 10, 3))
    with pytest.raises(ValueError, match="H, W, C"):
        ms.ssim(a[..., 0], a[..., 0])
    with pytest.raises(ValueError, match="1 <= C <= 4"):
        ms.ssim(torch.rand(8, 9, 5), torch.rand(8, 9, 5))
    with pytest.raises(ValueError, match="target must not require grad"):
        ms.l1_dssim_loss(a, a.clone().requires_grad_(True))


@pytest.mark.gpu
def test_arguments_rejected_on_gpu(cuda_device):
    a = torch.rand(8, 9, 3, device=cuda_device)
    with pytest.raises(ValueError, match="1 <= C <= 4"):
        ms.ssim(torch.rand(8, 9, 5, device=cuda_device), torch.rand(8, 9, 5, device=cuda_device))
    with pytest.raises(ValueError, match="H, W, C"):
        ms.ssim(a, torch.rand(9, 8, 3, device=cuda_device))
    with pytest.raises(ValueError, match="target must not require grad"):
        ms.ssim(a, a.clone().requires_grad_(True))
    with pytest.raises(ValueError, match="different devices"):
        ms.ssim(a, a.cpu())


# ---------------------------------------------------------------- parity ---------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("H,W,C,seed", [
    (37, 53, 3, 0), (1, 1, 3, 1), (3, 7, 2, 2), (64, 64, 1, 3), (64, 64, 4, 4), (33, 97, 2, 5), (100, 31, 4, 6),
    (1080, 1920, 3, 7)])
def test_loss_matches_fp64_autograd(cuda_device, H, W, C, seed):
    """Random images in [0, 1] (odd seeds: a correlated pair).  Measured maxima next to SCALAR_TOL / GRAD_TOL."""
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(H, W, C, generator=g).to(cuda_device)
    target = torch.rand(H, W, C, generator=g).to(cuda_device)
    if seed % 2:
        target = (0.7 * img + 0.3 * target).contiguous()  # correlated pair: SSIM well inside (0, 1)
    scalar_err, errs = compare(img, target)
    print(f"{H}x{W}x{C}: scalar {scalar_err:.2e} grads " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert scalar_err <= SCALAR_TOL, scalar_err
    for k, v in errs.items():
        assert v <= GRAD_TOL, (k, v)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3])
def test_loss_on_renders_matches_fp64_autograd(cuda_device, C):
    """Two renders of the same scene from perturbed parameters (render_gaussians), as in a training step."""
    cam, m, s, q, o, c, _ = e2e_scene(300, 96, 11, C)
    g = torch.Generator().manual_seed(12)
    bg = torch.linspace(0.1, 0.4, C).to(cuda_device)
    target = ms.render_gaussians(*[x.to(cuda_device) for x in (m, s, q, o, c)], cam, background_color=bg)
    m2 = m + 0.03 * torch.randn(m.shape, generator=g)
    img = ms.render_gaussians(*[x.to(cuda_device) for x in (m2, s, q, o, c)], cam, background_color=bg)
    assert img.shape == (96, 96, C)
    scalar_err, errs = compare(img, target)
    print(f"render C={C}: scalar {scalar_err:.2e} grads " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert scalar_err <= SCALAR_TOL, scalar_err
    for k, v in errs.items():
        assert v <= GRAD_TOL, (k, v)


# ---------------------------------------------------------------- known answers --------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("H,W,C", [(37, 53, 3), (1, 1, 1), (64, 64, 4)])
def test_identical_images(cuda_device, H, W, C):
    """ssim(x, x) = 1 within fp32 rounding with a vanishing gradient; the L1 gradient is exactly zero."""
    x = torch.rand(H, W, C, generator=torch.Generator().manual_seed(H + C)).to(cuda_device)
    p = x.clone().requires_grad_(True)
    s, l = ssim_l1(p, x)
    s_val, l_val = float(s.detach()), float(l.detach())
    assert abs(s_val - 1.0) <= 1e-6 and l_val == 0.0
    (gs,) = torch.autograd.grad(s, p, retain_graph=True)
    print(f"ssim(x, x) - 1 = {s_val - 1.0:.2e}, max |grad| * HWC = {float(gs.abs().max()) * H * W * C:.2e}")
    assert float(gs.abs().max()) * (H * W * C) <= 1e-3, float(gs.abs().max())
    (gl,) = torch.autograd.grad(l, p)
    assert torch.equal(gl, torch.zeros_like(gl))


@pytest.mark.gpu
@pytest.mark.parametrize("a,b,H,W,C", [(0.5, 0.5, 40, 50, 3), (0.2, 0.7, 40, 50, 3), (1.0, 0.0, 23, 17, 2),
                                       (0.0, 0.0, 12, 12, 1), (0.9, 0.3, 1, 1, 4)])
def test_constant_images(cuda_device, a, b, H, W, C):
    """Constant images: sigma = 0 in the interior, so only C1 / C2 keep S finite; at the border the zero padding makes
    mu and sigma differ from the interior values.  (1x1: a 1-pixel image.)"""
    img = torch.full((H, W, C), a, device=cuda_device)
    target = torch.full((H, W, C), b, device=cuda_device)
    scalar_err, errs = compare(img, target)
    print(f"constant {a}/{b} {H}x{W}x{C}: scalar {scalar_err:.2e} grads "
          + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert scalar_err <= CONST_SCALAR_TOL, scalar_err
    for k, v in errs.items():
        assert v <= CONST_GRAD_TOL, (k, v)


@pytest.mark.gpu
def test_one_pixel_image(cuda_device):
    """A 1x1 image: every window tap but the centre falls into the padding."""
    img = torch.tensor([[[0.3, 0.8, 0.1]]], device=cuda_device)
    target = torch.tensor([[[0.6, 0.8, 0.0]]], device=cuda_device)
    s64, l64 = torch_ssim_l1(img.double(), target.double())
    s, l = ssim_l1(img, target)
    assert abs(float(s) - float(s64)) <= SCALAR_TOL and abs(float(l) - float(l64)) <= 1e-7
    scalar_err, errs = compare(img, target)
    for k, v in errs.items():
        assert v <= GRAD_TOL, (k, v)


# ---------------------------------------------------------------- determinism ----------------------------------------

@pytest.mark.gpu
def test_deterministic_at_1080p(cuda_device):
    g = torch.Generator().manual_seed(21)
    img = torch.rand(1080, 1920, 3, generator=g).to(cuda_device)
    target = torch.rand(1080, 1920, 3, generator=g).to(cuda_device)
    res = []
    for _ in range(2):
        x = img.clone().requires_grad_(True)
        s, l = ssim_l1(x, target)
        (2.0 * s - 3.0 * l).backward()
        res.append((s.detach().clone(), l.detach().clone(), x.grad))
    for a, b in zip(*res):
        assert torch.equal(a, b)


# ---------------------------------------------------------------- fitting --------------------------------------------

@pytest.mark.gpu
def test_fit_small_scene_l1_dssim(cuda_device):
    """300 Adam steps of l1_dssim_loss from perturbed parameters back towards a rendered target, through
    render_gaussians_diff (the setting of test_gpu_train.test_fit_small_scene).  Measured on a B200: the loss falls
    1.419e-1 -> 1.012e-3 (x140); the test asks for x20."""
    torch.manual_seed(0)
    cam, m, s, q, o, c, _ = e2e_scene(200, 64, 42, 3)
    target = ms.render_gaussians_diff(*[x.to(cuda_device) for x in (m, s, q, o, c)], cam).detach()
    g = torch.Generator().manual_seed(7)
    params = [(m + 0.05 * torch.randn(m.shape, generator=g)),
              (s + 0.2 * torch.randn(s.shape, generator=g)),
              (q + 0.2 * torch.randn(q.shape, generator=g)),
              (o + 0.1 * torch.randn(o.shape, generator=g)).clamp(0.05, 0.99),
              (c + 0.2 * torch.randn(c.shape, generator=g)).clamp(0.0, 1.0)]
    params = [p.to(cuda_device).requires_grad_(True) for p in params]
    lrs = [2e-3, 1e-2, 1e-2, 1e-2, 1e-2]
    opt = torch.optim.Adam([{"params": [p], "lr": lr} for p, lr in zip(params, lrs)])
    losses = []
    for step in range(300):
        opt.zero_grad()
        img = ms.render_gaussians_diff(*params, cam)
        loss = ms.l1_dssim_loss(img, target)
        loss.backward()
        if step == 0:
            for p in params:
                assert float(p.grad.abs().sum()) > 0
        opt.step()
        losses.append(float(loss))
    ratio = losses[0] / losses[-1]
    print(f"fit (l1_dssim): loss {losses[0]:.3e} -> {losses[-1]:.3e} (x{ratio:.1f})")
    assert ratio >= 20.0, (losses[0], losses[-1])
