"""GPU: rasterization backward (SURVEY.md 8f rank 1) against torch autograd.

The reference is forward-only (render.py:11), gsplat is not installable here, so the gradient oracle is
torch autograd (fp64) through a pure-torch restatement of kernels/rasterization.mojo:138-162 -- written
below with whole-tile tensor ops, no hand-derived formula on the checking side.  The forward half
(image, final transmittance, last composited index) is checked against the C oracle / the faithful kernel.
"""
import numpy as np
import pytest
import torch

import mojosplat_b200 as ms
from helpers import BWD_RHO, bwd_entry_ratios, dev, image_gate
from mojosplat_b200 import rasterization
from oracle import oracle

pytestmark = pytest.mark.gpu


def torch_raster(means2d, conics, colors, opac, bg, ranges, ids, H, W, ts):
    """Differentiable restatement of rasterization.mojo:138-162 (fp64, CPU), one tile at a time."""
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
                dx, dy = means2d[g, 0] - px, means2d[g, 1] - py
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


def small_scene(N, HW, seed, C=3, opacity_lo=0.3):
    g = torch.Generator().manual_seed(seed)
    m = torch.randn(N, 3, generator=g) * 0.6
    m[:, 2] = torch.rand(N, generator=g) * 3.0 + 1.5
    s = torch.ones(N, 3) * -2.2 + torch.randn(N, 3, generator=g) * 0.3
    q = torch.nn.functional.normalize(torch.randn(N, 4, generator=g), dim=1)
    o = torch.rand(N, generator=g) * (0.98 - opacity_lo) + opacity_lo
    c = torch.rand(N, C, generator=g)
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=HW, W=HW, fx=60.0, fy=60.0, cx=HW / 2, cy=HW / 2)
    m2, con, dep, rad = oracle.project(m.numpy(), s.numpy(), q.numpy(), o.numpy(), cam.view_matrix.numpy(),
                                       cam.fx, cam.fy, cam.cx, cam.cy, HW, HW)
    return cam, m2, con, dep, rad, o.numpy(), c.numpy()


@pytest.mark.parametrize("N,HW,ts,C,seed", [(1, 32, 16, 3, 0), (40, 48, 16, 3, 1), (150, 64, 16, 3, 2),
                                            (60, 40, 10, 3, 3), (80, 48, 16, 1, 4), (80, 48, 16, 4, 5),
                                            (400, 32, 16, 3, 6),
                                            # partial tiles / image width not a multiple of 4 in the pair-layout kernels
                                            (80, 42, 16, 3, 12), (120, 57, 16, 3, 13),
                                            # tile sizes 31 / 32: > 48 KB of dynamic shared memory (opt-in attribute)
                                            (60, 64, 32, 3, 7), (60, 64, 32, 4, 8), (60, 62, 31, 3, 9),
                                            (60, 64, 32, 2, 10)])
def test_backward_matches_torch_autograd(cuda_device, N, HW, ts, C, seed):
    _check_backward(cuda_device, N, HW, ts, C, seed, "fast")  # (16x16 RGB: the pair-layout kernels; else the generic ones)


@pytest.mark.parametrize("N,HW,seed", [(1, 32, 0), (40, 48, 1), (150, 64, 2), (400, 32, 6)])
def test_backward_faithful_mode_matches_torch_autograd(cuda_device, N, HW, seed):
    _check_backward(cuda_device, N, HW, 16, 3, seed, "faithful")


def _check_backward(cuda_device, N, HW, ts, C, seed, mode):
    cam, m2, con, dep, rad, o, c = small_scene(N, HW, seed, C)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, HW, HW, ts)
    bg = np.linspace(0.1, 0.4, C).astype(np.float32)
    gen = torch.Generator().manual_seed(100 + seed)
    gimg = torch.randn(HW, HW, C, generator=gen)

    # oracle side: fp64 autograd on the CPU
    t64 = [torch.tensor(x, dtype=torch.float64, requires_grad=True) for x in (m2, con, c, o, bg)]
    ref_img = torch_raster(*t64, ranges, ids, HW, HW, ts)
    (ref_img * gimg.double()).sum().backward()

    # CUDA side, through the autograd.Function over the C ABI
    t32 = [dev(x, cuda_device).requires_grad_(True) for x in (m2, con, c, o, bg)]
    img = rasterization.rasterize_gaussians_diff(t32[0], t32[1], t32[2], t32[3], t32[4], dev(ranges, cuda_device),
                                                 dev(ids, cuda_device), cam, ts, mode=mode)
    np.testing.assert_allclose(img.detach().cpu().numpy(), ref_img.detach().numpy(), atol=1e-4, rtol=1e-4)
    (img * gimg.to(cuda_device)).sum().backward()
    names = ["means2d", "conics", "colors", "opacities", "background"]
    for name, a, b in zip(names, t32, t64):
        got, want = a.grad.cpu().double().numpy(), b.grad.numpy()
        assert got.shape == want.shape
        scale = np.abs(want).max() + 1e-12
        # fp32 compositing + atomics vs fp64 autograd: 1e-3 of the largest entry, plus 1e-3 relative
        np.testing.assert_allclose(got, want, atol=1e-3 * scale, rtol=1e-3, err_msg=name)
        assert np.abs(want).max() > 0 or N == 0, name
    rho = BWD_RHO["fast" if (mode == "fast" and ts == 16 and C == 3) else "faithful"]
    _assert_every_entry(cuda_device, (m2, con, c, o, bg), ranges, ids, cam, ts, mode, gimg.numpy(), rho)


def _assert_every_entry(cuda_device, inputs, ranges, ids, cam, ts, mode, gimg, rho):
    """Every gradient entry within the per-entry bound against the fp64 reference (oracle.raster_bwd_f64), with the
    upstream gradient zeroed on the reference's borderline pixels (on both sides)."""
    m2, con, c, o, bg = inputs
    H, W = int(cam.H), int(cam.W)
    ref = oracle.raster_bwd_f64(m2, con, c, o, bg, ranges, ids, W, H, ts, gimg, mask_borderline=True)
    gm = np.where(ref["borderline"][..., None], np.float32(0), gimg.astype(np.float32))
    t32 = [dev(x, cuda_device).requires_grad_(True) for x in inputs]
    img = rasterization.rasterize_gaussians_diff(*t32, dev(ranges, cuda_device), dev(ids, cuda_device), cam, ts,
                                                 mode=mode)
    img.backward(dev(gm, cuda_device))
    got = {n: x.grad.cpu().double().numpy() for n, x in zip(["means2d", "conics", "colors", "opacities",
                                                             "background"], t32)}
    assert float(ref["borderline"].mean()) <= 0.05
    for n, r in bwd_entry_ratios(got, ref, rho, H * W).items():
        assert r.max() <= 1.0, (n, float(r.max()), np.unravel_index(int(r.argmax()), r.shape))


def test_train_forward_equals_faithful_kernel(cuda_device):
    """Same operation order as the faithful kernel => identical image; final_T / last_idx consistent."""
    cam, m2, con, dep, rad, o, c = small_scene(300, 96, 7)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, 96, 96, 16)
    bg = np.array([0.1, 0.2, 0.3], np.float32)
    a = [dev(m2, cuda_device), dev(con, cuda_device), dev(c, cuda_device), dev(o, cuda_device),
         dev(bg, cuda_device), dev(ranges, cuda_device), dev(ids, cuda_device)]
    faithful = rasterization.rasterize_gaussians_cuda(*a, cam, 16, mode="faithful")
    img = rasterization.rasterize_gaussians_diff(*a, cam, 16, mode="faithful")
    assert torch.equal(img, faithful)
    ref = oracle.rasterize(m2, con, c, o, bg, ranges, ids, 96, 96, 16)
    assert image_gate(img.cpu().numpy(), ref)["ok"]


def _train_forward_raw(a, H, W, fast, cuda_device):
    """(image, final_T, last_idx) of the two training-side forward entry points, straight through the C ABI."""
    from mojosplat_b200 import _lib
    L = _lib.load()
    m2, con, c, o, bg, ranges, ids = a
    N = m2.shape[0]
    image = torch.empty((H, W, 3), dtype=torch.float32, device=cuda_device)
    final_T = torch.empty((H, W), dtype=torch.float32, device=cuda_device)
    last = torch.empty((H, W), dtype=torch.int32, device=cuda_device)
    sp = _lib.stream_ptr(torch.device(cuda_device))
    if fast:
        rc = L.bsplat_rasterize_fwd_train_fast(N, _lib.ptr(m2), _lib.ptr(con), _lib.ptr(c), _lib.ptr(o), _lib.ptr(bg),
                                               _lib.ptr(ranges), None, _lib.ptr(ids), ids.numel(), W, H,
                                               _lib.ptr(image), _lib.ptr(final_T), _lib.ptr(last), None, 0, sp)
    else:
        rc = L.bsplat_rasterize_fwd_train(N, 3, _lib.ptr(m2), _lib.ptr(con), _lib.ptr(c), _lib.ptr(o), _lib.ptr(bg),
                                          _lib.ptr(ranges), _lib.ptr(ids), ids.numel(), W, H, 16, _lib.ptr(image),
                                          _lib.ptr(final_T), _lib.ptr(last), sp)
    assert rc == 0
    torch.cuda.synchronize()
    return image, final_T, last


@pytest.mark.parametrize("scene", ["plain", "opaque"])
def test_fast_train_forward(cuda_device, scene):
    """The training-side forward through the pair kernel: image == the inference kernel's bit for bit (with and without
    the record workspace), final transmittance within the float tolerance of the faithful forward's, and last_idx
    consistent with it: never in front of the faithful 'last composited' index (entries behind it fail the alpha test
    again in the backward pass), equal to it + 0 wherever the pixel saturated."""
    if scene == "plain":
        cam, m2, con, dep, rad, o, c = small_scene(300, 96, 7)
        HW = 96
    else:  # opaque stacks: most pixels saturate long before the end of their list
        N, HW = 80, 64
        g = torch.Generator().manual_seed(3)
        m2 = (torch.rand(N, 2, generator=g) * 40 + 12).numpy().astype(np.float32)
        con = np.tile(np.array([[0.02, 0.0, 0.02]], np.float32), (N, 1))
        dep = np.arange(N, dtype=np.float32) + 1
        rad = np.full((N, 2), 40, np.int32)
        o = np.full(N, 0.95, np.float32)
        c = torch.rand(N, 3, generator=g).numpy()
        cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=HW, W=HW, fx=60.0, fy=60.0, cx=32.0, cy=32.0)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, HW, HW, 16)
    bg = np.array([0.1, 0.2, 0.3], np.float32)
    a = [dev(m2, cuda_device), dev(con, cuda_device), dev(c, cuda_device), dev(o, cuda_device),
         dev(bg, cuda_device), dev(ranges, cuda_device).to(torch.int32).contiguous(),
         dev(ids, cuda_device).to(torch.int32).contiguous()]
    infer = rasterization.rasterize_gaussians_cuda(*a, cam, 16)
    img_ws = rasterization.rasterize_gaussians_diff(*a, cam, 16)          # records + tile order
    img_raw, T_fast, last_fast = _train_forward_raw(a, HW, HW, True, cuda_device)   # workspace-free staging
    assert torch.equal(img_ws, infer) and torch.equal(img_raw, infer)
    img_f, T_f, last_f = _train_forward_raw(a, HW, HW, False, cuda_device)
    assert float((T_fast - T_f).abs().max()) <= 1e-5
    r1 = a[5][..., 1].repeat_interleave(16, 0).repeat_interleave(16, 1)[:HW, :HW]
    saturated = last_fast < r1 - 1
    assert bool((last_fast >= last_f).all())
    if scene == "opaque":
        assert int(saturated.sum()) > 100
    # and never past the end of the tile's list
    assert bool((last_fast <= r1 - 1).all())


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_backward_saturated_pixels_and_clamp(cuda_device, mode):
    """Opaque stacks: pixels stop early (the stopping Gaussian gets no gradient) and alpha hits the 0.999 clamp
    (no gradient through it). Still equal to autograd."""
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
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=HW, W=HW, fx=60.0, fy=60.0, cx=16.0, cy=16.0)
    t64 = [torch.tensor(x, dtype=torch.float64, requires_grad=True) for x in (m2, con, c, o, bg)]
    ref_img = torch_raster(*t64, ranges, ids, HW, HW, 16)
    ref_img.sum().backward()
    t32 = [dev(x, cuda_device).requires_grad_(True) for x in (m2, con, c, o, bg)]
    img = rasterization.rasterize_gaussians_diff(*t32, dev(ranges, cuda_device), dev(ids, cuda_device), cam, 16,
                                                 mode=mode)
    img.sum().backward()
    np.testing.assert_allclose(img.detach().cpu().numpy(), ref_img.detach().numpy(), atol=1e-4, rtol=1e-4)
    for a, b in zip(t32, t64):
        want = b.grad.numpy(); scale = np.abs(want).max() + 1e-12
        np.testing.assert_allclose(a.grad.cpu().double().numpy(), want, atol=2e-3 * scale, rtol=2e-3)
    rho = BWD_RHO[mode]
    for gimg in (np.ones((HW, HW, 3), np.float32),
                 torch.randn(HW, HW, 3, generator=torch.Generator().manual_seed(12)).numpy()):
        _assert_every_entry(cuda_device, (m2, con, c, o, bg), ranges, ids, cam, 16, mode, gimg, rho)
    # Gaussians that autograd says never contributed (behind saturated pixels everywhere) get exactly zero
    never = (t64[2].grad.abs().sum(dim=1) == 0).numpy()
    assert float(t32[2].grad.cpu()[torch.from_numpy(never)].abs().sum()) == 0.0
    # and saturation did happen: some pixel stopped before the end of its list
    assert float(ref_img.detach().max()) > 0 and never.sum() >= 0


def test_backward_empty_and_linearity(cuda_device):
    cam, m2, con, dep, rad, o, c = small_scene(120, 64, 21)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, 64, 64, 16)
    bg = np.zeros(3, np.float32)
    base = [dev(m2, cuda_device), dev(con, cuda_device), dev(c, cuda_device), dev(o, cuda_device)]

    def grads(gimg):
        t = [x.clone().requires_grad_(True) for x in base]
        img = rasterization.rasterize_gaussians_diff(*t, dev(bg, cuda_device), dev(ranges, cuda_device),
                                                     dev(ids, cuda_device), cam, 16)
        img.backward(gimg)
        return [x.grad for x in t]
    g1 = torch.randn(64, 64, 3, device=cuda_device); g2 = torch.randn(64, 64, 3, device=cuda_device)
    a, b, ab = grads(g1), grads(g2), grads(g1 + g2)
    for x, y, z in zip(a, b, ab):  # the backward pass is linear in grad_image
        scale = float(z.abs().max()) + 1e-12
        assert float((x + y - z).abs().max()) <= 1e-4 * scale
    # empty lists: background only, zero gradients
    empty_ranges = torch.zeros_like(dev(ranges, cuda_device))
    t = [x.clone().requires_grad_(True) for x in base]
    img = rasterization.rasterize_gaussians_diff(*t, dev(bg + 0.25, cuda_device), empty_ranges,
                                                 dev(ids, cuda_device), cam, 16)
    img.sum().backward()
    assert float((img - 0.25).abs().max()) == 0.0
    assert all(float(x.grad.abs().max()) == 0.0 for x in t)


def test_backward_100k_gaussians_vs_finite_differences(cuda_device):
    """Backward at scale (100 k Gaussians @1080p, M ~ 8 M) against central finite differences of the forward pass, on a
    random subset of parameters.  The loss is a fixed random projection of the image; the forward used for the
    differences is the train forward in fp32, so the step is chosen large enough for its rounding noise (1e-7
    relative on a sum of ~6 M terms) and parameters whose two-sided difference crosses a threshold decision (alpha
    1/255, saturation: the loss is discontinuous there) are recognised by a mismatch between the h and h/2
    differences and skipped."""
    from mojosplat_b200 import synthetic
    sc = synthetic.make_scene("config2_100k_1080p")
    cam = sc.camera
    g = [t.to(cuda_device) for t in sc.gaussians()]
    bg = sc.background.to(cuda_device)
    _, aux = ms.render_fused(*g, cam.to(cuda_device), bg, return_aux=True)
    _, aux = ms.render_fused(*g, cam.to(cuda_device), bg, return_aux=True)
    ids, ranges = aux["sorted_ids"], aux["tile_ranges"]
    assert ids is not None and ids.numel() > 5_000_000
    gen = torch.Generator().manual_seed(5)
    gimg = torch.randn(cam.H, cam.W, 3, generator=gen).to(cuda_device)
    base = [aux["means2d"].double(), aux["conics"].double(), g[4].double(), g[3].double()]

    def loss(params):
        img = rasterization.rasterize_gaussians_diff(params[0].float(), params[1].float(), params[2].float(),
                                                     params[3].float(), bg, ranges, ids, cam, 16)
        return float((img.double() * gimg.double()).sum())

    t = [x.float().clone().requires_grad_(True) for x in base]
    img = rasterization.rasterize_gaussians_diff(*t, bg, ranges, ids, cam, 16)
    (img * gimg).sum().backward()
    torch.cuda.synchronize()
    # visible Gaussians with a sizeable gradient
    vis = torch.nonzero((aux["radii"] > 0).all(-1)).flatten().cpu()
    pick = vis[torch.randperm(vis.numel(), generator=gen)[:12]]
    # The alpha >= 1/255 ring of a Gaussian is ~60 pixels long: a step moves a few of them across the threshold and each
    # crossing jumps the loss by ~T c / 255.  Their contribution to the difference quotient falls like 1 / sqrt(h)
    # while the truncation error of a ~3 px wide Gaussian is (h / sigma)^2 / 6: fairly large steps are the accurate ones.
    steps = {0: 0.25, 1: None, 2: 5e-2, 3: 5e-2}   # means2d (px), conics (relative), colours, opacities
    checked = 0
    for which, name in enumerate(["means2d", "conics", "colors", "opacities"]):
        for gi in pick.tolist():
            comp = 0 if which == 3 else int(gi) % base[which].shape[1]
            analytic = float(t[which].grad[gi] if which == 3 else t[which].grad[gi, comp])
            x0 = float(base[which][gi] if which == 3 else base[which][gi, comp])
            h = steps[which] if steps[which] is not None else 0.05 * abs(x0) + 1e-5
            fd = []
            for hh in (h, h / 2):
                vals = []
                for sgn in (+1, -1):
                    p = [x.clone() for x in base]
                    if which == 3:
                        p[which][gi] = x0 + sgn * hh
                    else:
                        p[which][gi, comp] = x0 + sgn * hh
                    vals.append(loss(p))
                fd.append((vals[0] - vals[1]) / (2 * hh))
            scale = max(abs(fd[0]), abs(fd[1]), abs(analytic), 1e-6)
            if abs(fd[0] - fd[1]) > 0.1 * scale:
                continue   # threshold crossings dominate inside [x - h, x + h]: no derivative to compare with
            checked += 1
            assert abs(analytic - fd[0]) <= 0.1 * scale + 2e-3, (name, gi, comp, analytic, fd)
    assert checked >= 24, checked
    # the two backward implementations (pair layout / generic) on the same inputs, every gradient entry: float rounding
    # of two different summation orders plus the rare alpha decisions that ex2.approx and expf take differently
    t2 = [x.float().clone().requires_grad_(True) for x in base]
    img2 = rasterization.rasterize_gaussians_diff(*t2, bg, ranges, ids, cam, 16, mode="faithful")
    (img2 * gimg).sum().backward()
    for name, a, b in zip(["means2d", "conics", "colors", "opacities"], t, t2):
        scale = float(b.grad.abs().max()) + 1e-12
        diff = (a.grad - b.grad).abs()
        assert float(diff.max()) <= 2e-2 * scale, (name, float(diff.max()), scale)
        assert float((diff > 1e-3 * scale).float().mean()) <= 1e-4, name
