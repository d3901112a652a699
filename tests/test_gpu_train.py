"""Differentiable rendering from the 3D parameters: projection backward (bsplat_project_bwd), SH backward
(bsplat_sh_bwd) and render_gaussians_diff, against fp64 torch autograd.

The oracle is autograd through pure-torch restatements of the forwards (no hand-derived formula on the checking
side, like test_gpu_raster_bwd.py).  The projection restatement is anchored to the repository's own forward by the
CPU tests at the top: the torch rules against oracle.project_f64, the gsplat rules against oracle.project.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import mojosplat_b200 as ms
from helpers import dev
from mojosplat_b200 import projection, sh
from oracle import oracle
from oracle.oracle_np import sh_eval_np
from test_gpu_raster_bwd import torch_raster


def lims_f32(cam):
    """Jacobian clamp limits as the kernels compute them (fp32, projection.cuh: make_proj_cam)."""
    f = np.float32
    W, H, fx, fy, cx, cy = f(cam.W), f(cam.H), f(cam.fx), f(cam.fy), f(cam.cx), f(cam.cy)
    tx, ty = f(0.5) * W / fx, f(0.5) * H / fy
    return (float((W - cx) / fx + f(0.3) * tx), float(cx / fx + f(0.3) * tx),
            float((H - cy) / fy + f(0.3) * ty), float(cy / fy + f(0.3) * ty))


def lims_f64(cam):
    """The same limits in double precision (oracle.project_f64)."""
    tx, ty = 0.5 * cam.W / cam.fx, 0.5 * cam.H / cam.fy
    return ((cam.W - cam.cx) / cam.fx + 0.3 * tx, cam.cx / cam.fx + 0.3 * tx,
            (cam.H - cam.cy) / cam.fy + 0.3 * ty, cam.cy / cam.fy + 0.3 * ty)


def torch_project(means3d, log_scales, quats, opacities, cam, lims, semantics=oracle.SEM_TORCH, eps2d=0.3):
    """Differentiable restatement of projection.cu: project_core (fp64 tensors in).
    -> (means2d, conics, depths, radii_real [N,2] (extent * sqrt(c) before ceil), visible [N] bool)."""
    vm = cam.view_matrix.to(torch.float64)
    Rv, t = vm[:3, :3], vm[:3, 3]
    fx, fy, cx, cy = float(cam.fx), float(cam.fy), float(cam.cx), float(cam.cy)
    mc = means3d @ Rv.T + t
    q = F.normalize(quats, dim=1, eps=1e-12)
    w, x, y, z = q.unbind(1)
    R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                     2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                     2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], 1).reshape(-1, 3, 3)
    M = R * torch.exp(log_scales)[:, None, :]
    Sc = Rv @ (M @ M.transpose(1, 2)) @ Rv.T
    tz = mc[:, 2]
    lxp, lxn, lyp, lyn = lims
    tx = tz * torch.clamp(mc[:, 0] / tz, -lxn, lxp)
    ty = tz * torch.clamp(mc[:, 1] / tz, -lyn, lyp)
    zero = torch.zeros_like(tz)
    J = torch.stack([torch.stack([fx / tz, zero, -fx * tx / tz ** 2], 1),
                     torch.stack([zero, fy / tz, -fy * ty / tz ** 2], 1)], 1)
    cov = J @ Sc @ J.transpose(1, 2)
    c00, c01, c10, c11 = cov[:, 0, 0] + eps2d, cov[:, 0, 1], cov[:, 1, 0], cov[:, 1, 1] + eps2d
    det = c00 * c11 - c01 * c10
    if semantics == oracle.SEM_TORCH:
        det = torch.clamp(det, min=1e-10)
    conics = torch.stack([c11 / det, -(c01 + c10) / 2 / det, c00 / det], 1)
    means2d = torch.stack([(fx * mc[:, 0] + cx * tz) / tz, (fy * mc[:, 1] + cy * tz) / tz], 1)
    with torch.no_grad():
        m2x, m2y = means2d[:, 0], means2d[:, 1]
        if semantics == oracle.SEM_TORCH:
            rx, ry = 3.33 * torch.sqrt(c00), 3.33 * torch.sqrt(c11)
            vis = (det > 0) & (tz > cam.near) & (tz < cam.far)
            vis &= (m2x + torch.ceil(rx) > 0) & (m2x - torch.ceil(rx) < cam.W) & \
                   (m2y + torch.ceil(ry) > 0) & (m2y - torch.ceil(ry) < cam.H)
        else:
            op = opacities.to(torch.float64)
            ext = torch.clamp(torch.sqrt(2 * torch.log(torch.clamp(op * 255.0, min=1.0))), max=3.33)
            rx, ry = ext * torch.sqrt(c00), ext * torch.sqrt(c11)
            Rx, Ry = torch.ceil(rx), torch.ceil(ry)
            vis = (tz > cam.near) & (tz < cam.far) & (op >= 1 / 255.0)
            vis &= ~((Rx <= 0) & (Ry <= 0)) & (m2x + Rx > 0) & (m2x - Rx < cam.W) & (m2y + Ry > 0) & (m2y - Ry < cam.H)
        radii = torch.where(vis[:, None], torch.stack([rx, ry], 1), torch.zeros_like(means2d))
    return means2d, conics, tz, radii, vis


def torch_sh(degree, coeffs, means3d, campos):
    """Differentiable fp64 form of oracle_np.sh_eval_np."""
    c = coeffs
    d = means3d - campos[None, :]
    d = d / torch.clamp(torch.linalg.norm(d, dim=1, keepdim=True), min=1e-15)
    x, y, z = d[:, 0:1], d[:, 1:2], d[:, 2:3]
    out = 0.28209479177387814 * c[:, 0]
    if degree >= 1:
        out = out + 0.4886025119029199 * (-y * c[:, 1] + z * c[:, 2] - x * c[:, 3])
    if degree >= 2:
        xx, yy, zz, xy, yz, xz = x * x, y * y, z * z, x * y, y * z, x * z
        out = out + (1.0925484305920792 * xy * c[:, 4] - 1.0925484305920792 * yz * c[:, 5]
                     + 0.31539156525252005 * (2 * zz - xx - yy) * c[:, 6] - 1.0925484305920792 * xz * c[:, 7]
                     + 0.5462742152960396 * (xx - yy) * c[:, 8])
    if degree >= 3:
        out = out + (-0.5900435899266435 * y * (3 * xx - yy) * c[:, 9] + 2.890611442640554 * xy * z * c[:, 10]
                     - 0.4570457994644658 * y * (4 * zz - xx - yy) * c[:, 11]
                     + 0.3731763325901154 * z * (2 * zz - 3 * xx - 3 * yy) * c[:, 12]
                     - 0.4570457994644658 * x * (4 * zz - xx - yy) * c[:, 13]
                     + 1.445305721320277 * z * (xx - yy) * c[:, 14] - 0.5900435899266435 * x * (xx - 3 * yy) * c[:, 15])
    return torch.clamp(out + 0.5, min=0.0)


def rotated_camera(HW, seed, f=60.0):
    """A camera with a non-trivial world->camera rotation (a transposed Rv would not go unnoticed)."""
    g = torch.Generator().manual_seed(1000 + seed)
    q = F.normalize(torch.tensor([1.0, 0.0, 0.0, 0.0]) + 0.3 * torch.randn(4, generator=g), dim=0)
    w, x, y, z = q.tolist()
    R = torch.tensor([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                      [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                      [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]], dtype=torch.float32)
    T = torch.randn(3, generator=g) * 0.5
    return ms.Camera(R=R, T=T, H=HW, W=HW, fx=f, fy=f, cx=HW / 2, cy=HW / 2)


def proj_scene(N, seed, HW=64, extremes=True):
    """Gaussians placed in camera space (then mapped to the world): mostly ordinary ones; with `extremes` also rows whose
    x/z or y/z is clamped but which stay visible (large, just off the image), rows behind the near plane,
    unnormalised quaternions (norms 0.3-3) and anisotropic scales."""
    cam = rotated_camera(HW, seed)
    g = torch.Generator().manual_seed(seed)
    mcam = torch.randn(N, 3, generator=g) * 0.6
    mcam[:, 2] = torch.rand(N, generator=g) * 3.0 + 1.5
    ls = -2.2 + torch.randn(N, 3, generator=g) * 0.5
    if extremes and N > 1:
        k = torch.arange(N)
        clampx, clampy, behind = (k % 10 == 3), (k % 10 == 6), (k % 20 == 9)
        mcam[clampx, 2] = 2.0
        mcam[clampx, 0] = 1.6 * torch.sign(torch.randn(int(clampx.sum()), generator=g))   # x/z = +-0.8
        mcam[clampy, 2] = 2.0
        mcam[clampy, 1] = 1.6 * torch.sign(torch.randn(int(clampy.sum()), generator=g))
        ls[clampx | clampy] = -1.2 + torch.randn(int((clampx | clampy).sum()), 3, generator=g) * 0.1
        mcam[behind, 2] = -torch.rand(int(behind.sum()), generator=g)
    means = (mcam - cam.T) @ cam.R          # world = R^T (mu_c - T)
    q = F.normalize(torch.randn(N, 4, generator=g), dim=1) * (0.3 + 2.7 * torch.rand(N, 1, generator=g))
    o = torch.rand(N, generator=g) * 0.95 + 0.05
    return cam, means.float().contiguous(), ls.float().contiguous(), q.float().contiguous(), o.float().contiguous()


def _f64(*a):
    return [torch.as_tensor(np.asarray(x), dtype=torch.float64) for x in a]


# ---------------------------------------------------------------- 1. the restatement is anchored (CPU) ----------

def test_restatement_matches_oracle_torch_rules():
    cam, m, s, q, o = proj_scene(1000, 0)
    m2, con, dep, rad, vis = torch_project(*_f64(m, s, q, o), cam, lims_f64(cam))
    om2, ocon, odep, orad = oracle.project_f64(m.numpy(), s.numpy(), q.numpy(), cam.view_matrix.numpy(), cam.fx,
                                               cam.fy, cam.cx, cam.cy, cam.W, cam.H)
    ovis = (orad > 0).any(axis=1)
    assert np.array_equal(vis.numpy(), ovis) and ovis.sum() > 500
    for got, want in ((m2, om2), (con, ocon), (dep, odep), (rad, orad)):
        np.testing.assert_allclose(got.numpy()[ovis], want[ovis], rtol=1e-9, atol=0)


def test_restatement_matches_oracle_gsplat_rules():
    cam, m, s, q, o = proj_scene(1000, 1)
    m2, con, dep, rad, vis = torch_project(*_f64(m, s, q, o), cam, lims_f32(cam), semantics=oracle.SEM_GSPLAT)
    om2, ocon, odep, orad = oracle.project(m.numpy(), s.numpy(), q.numpy(), o.numpy(), cam.view_matrix.numpy(),
                                           cam.fx, cam.fy, cam.cx, cam.cy, cam.W, cam.H,
                                           semantics=oracle.SEM_GSPLAT)
    ovis = (orad > 0).any(axis=1)
    assert np.array_equal(vis.numpy(), ovis) and 500 < ovis.sum() < 1000
    assert np.array_equal(np.ceil(rad.numpy()[ovis]), orad[ovis])
    for got, want in ((m2, om2), (con, ocon), (dep, odep)):
        got, want = got.numpy()[ovis], want[ovis].astype(np.float64)
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5 * np.abs(want).max())


def test_render_diff_rejects_cpu_tensors():
    z = torch.zeros
    cam = ms.Camera(R=torch.eye(3), T=z(3), H=8, W=8, fx=1.0, fy=1.0, cx=4.0, cy=4.0)
    with pytest.raises(ValueError, match="CUDA tensors"):
        ms.render_gaussians_diff(z(1, 3), z(1, 3), z(1, 4), z(1), z(1, 3), cam)


# ---------------------------------------------------------------- 2. projection backward ----------------------------

def _assert_grad_close(got, want, name):
    scale = np.abs(want).max() + 1e-12
    np.testing.assert_allclose(got, want, atol=1e-3 * scale, rtol=1e-3, err_msg=name)


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["cuda", "cuda_gsplat"])
@pytest.mark.parametrize("N", [0, 1, 37, 256, 1000, 5003])
def test_projection_backward_matches_autograd(cuda_device, backend, N):
    sem = projection.CUDA_BACKENDS[backend]
    cam, m, s, q, o = proj_scene(N, 10 + N)
    gen = torch.Generator().manual_seed(N)
    g_m2, g_con, g_dep = torch.randn(N, 2, generator=gen), torch.randn(N, 3, generator=gen), torch.randn(N, generator=gen)

    t32 = [dev(x.numpy(), cuda_device).requires_grad_(True) for x in (m, s, q)]
    o32 = dev(o.numpy(), cuda_device)
    m2, con, dep, rad = projection.project_gaussians_diff(*t32, o32, cam, backend=backend)
    assert not rad.requires_grad
    ref = projection.project_gaussians(*[t.detach() for t in t32], o32, cam, backend=backend)
    for a, b in zip((m2, con, dep, rad), ref):
        assert torch.equal(a.detach(), b)
    if N == 0:
        return
    got = torch.autograd.grad((m2, con, dep), t32, (g_m2.to(cuda_device), g_con.to(cuda_device),
                                                     g_dep.to(cuda_device)))
    vis = (rad.cpu() != 0).any(dim=1).numpy()

    t64 = [x.double().requires_grad_(True) for x in (m, s, q)]
    w_m2, w_con, w_dep, _, _ = torch_project(*t64, o.double(), cam, lims_f32(cam), semantics=sem)
    want = torch.autograd.grad((w_m2, w_con, w_dep), t64, (g_m2.double(), g_con.double(), g_dep.double()))
    for name, a, b in zip(["means3d", "log_scales", "quats"], got, want):
        a = a.cpu().double().numpy()
        assert np.isfinite(a).all(), name
        assert (a[~vis] == 0).all(), name          # culled rows (behind the camera included): exact zeros
        _assert_grad_close(a[vis], b.numpy()[vis], name)
    if N >= 256:
        lxp, lxn, lyp, lyn = lims_f32(cam)
        mc = (m.double() @ cam.R.double().T + cam.T.double())
        rxz, ryz = mc[:, 0] / mc[:, 2], mc[:, 1] / mc[:, 2]
        clamped = ((rxz > lxp) | (rxz < -lxn) | (ryz > lyp) | (ryz < -lyn)).numpy()
        behind = (mc[:, 2] < 0.1).numpy()
        assert (clamped & vis).sum() >= 5 and behind.sum() > 0 and not (behind & vis).any()


# ---------------------------------------------------------------- 3. SH backward ------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("degree,K", [(0, 1), (0, 16), (1, 4), (2, 9), (2, 16), (3, 16), (1, 9)])
def test_sh_backward_matches_autograd(cuda_device, degree, K):
    N = 3001
    g = torch.Generator().manual_seed(degree * 100 + K)
    coeffs = torch.randn(N, K, 3, generator=g) * 0.6
    coeffs[::7, 0] = -3.0                   # r + 0.5 < 0 on most channels of these rows
    means = torch.randn(N, 3, generator=g) * 2
    cam = rotated_camera(64, degree)
    gcol = torch.randn(N, 3, generator=g)
    c32, m32 = coeffs.to(cuda_device).requires_grad_(True), means.to(cuda_device).requires_grad_(True)
    col = sh.eval_sh_diff(degree, c32, m32, cam)
    assert torch.equal(col.detach(), sh.eval_sh(degree, c32.detach(), m32.detach(), cam))
    col.backward(gcol.to(cuda_device))

    c64, m64 = coeffs.double().requires_grad_(True), means.double().requires_grad_(True)
    pos = sh.camera_position(cam).double()
    full = torch.cat([c64, torch.zeros(N, 16 - K, 3, dtype=torch.float64)], 1) if K < 16 else c64
    ref = torch_sh(degree, full, m64, pos)
    np.testing.assert_allclose(ref.detach().numpy(), sh_eval_np(degree, full.detach().numpy(), means.numpy(),
                                                                pos.numpy()), rtol=1e-12, atol=1e-12)
    ref.backward(gcol.double())
    assert int((ref.detach() == 0).sum()) > N // 10   # the clamp is active on many entries
    gc = c32.grad.cpu().double().numpy()
    used = (degree + 1) ** 2
    assert (gc[:, used:] == 0).all()
    _assert_grad_close(gc, c64.grad.numpy(), "coeffs")
    gm = m32.grad.cpu().double().numpy()
    if degree == 0:
        assert (gm == 0).all()
    else:
        _assert_grad_close(gm, m64.grad.numpy(), "means3d")
        assert np.abs(gm).max() > 0


# ---------------------------------------------------------------- 4. end to end -------------------------------------

def e2e_scene(N, HW, seed, C):
    g = torch.Generator().manual_seed(seed)
    m = torch.randn(N, 3, generator=g) * 0.6
    m[:, 2] = torch.rand(N, generator=g) * 3.0 + 1.5
    s = torch.ones(N, 3) * -2.2 + torch.randn(N, 3, generator=g) * 0.3
    q = F.normalize(torch.randn(N, 4, generator=g), dim=1) * (0.5 + torch.rand(N, 1, generator=g))
    o = torch.rand(N, generator=g) * 0.68 + 0.3
    c = torch.rand(N, C, generator=g)
    coeffs = torch.randn(N, 16, 3, generator=g) * 0.3
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=HW, W=HW, fx=60.0, fy=60.0, cx=HW / 2, cy=HW / 2)
    return cam, m, s, q, o, c, coeffs


@pytest.mark.gpu
@pytest.mark.parametrize("N,HW,ts,C,use_sh,backend,seed", [
    (200, 64, 16, 3, False, "cuda", 0), (300, 96, 16, 3, True, "cuda", 1), (150, 64, 32, 3, False, "cuda", 2),
    (120, 48, 16, 1, False, "cuda_gsplat", 3), (120, 48, 16, 4, False, "cuda", 4),
    (400, 96, 16, 3, True, "cuda_gsplat", 5), (50, 48, 32, 4, False, "cuda_gsplat", 6),
    (200, 64, 16, 3, False, "cuda_gsplat", 7), (100, 64, 32, 3, True, "cuda", 8)])
def test_render_diff_matches_autograd(cuda_device, N, HW, ts, C, use_sh, backend, seed):
    cam, m, s, q, o, c, coeffs = e2e_scene(N, HW, seed, C)
    feats = coeffs if use_sh else c
    bg = torch.linspace(0.1, 0.4, C)
    sem = projection.CUDA_BACKENDS[backend]
    gen = torch.Generator().manual_seed(100 + seed)
    gimg = torch.randn(HW, HW, C, generator=gen)

    t32 = [x.to(cuda_device).requires_grad_(True) for x in (m, s, q, o, feats, bg)]
    img, aux = ms.render_gaussians_diff(*t32[:5], cam, sh_degree=3 if use_sh else None, background_color=t32[5],
                                        tile_size=ts, backend=backend, return_aux=True)
    if ts == 16 and C == 3:
        # every stage is bit-identical to its counterpart inside the fused frame
        ref = ms.render_gaussians(*[t.detach() for t in t32[:5]], cam, sh_degree=3 if use_sh else None,
                                  background_color=t32[5].detach(), tile_size=ts, backend=backend)
        assert torch.equal(img.detach(), ref)
    (img * gimg.to(cuda_device)).sum().backward()

    # oracle: fp64 autograd through the restatements and torch_raster, on the lists the CUDA forward produced.  The
    # values fed to torch_raster are the kernels' fp32 ones (straight-through: x64 + (x32 - x64).detach()), so that a
    # threshold of the compositing (alpha >= 1/255, the saturation stop) decides the same way on both sides; the
    # gradients are fp64 autograd's.  Culled rows are constants (the documented contract of the projection backward).
    t64 = [x.double().requires_grad_(True) for x in (m, s, q, o, feats, bg)]
    m2, con, _, _, _ = torch_project(t64[0], t64[1], t64[2], o.double(), cam, lims_f32(cam), semantics=sem)
    vis = (aux["radii"].cpu() != 0).any(dim=1)[:, None]

    def st(x64, x32):
        x = x64 + (x32.detach().cpu().double() - x64).detach()
        return torch.where(vis, x, x.detach())
    m2 = st(m2, aux["means2d"])
    con = st(con, aux["conics"])
    if use_sh:
        col = torch_sh(3, t64[4], t64[0], sh.camera_position(cam).double())
        col = col + (sh.eval_sh(3, t32[4].detach(), t32[0].detach(), cam).cpu().double() - col).detach()
    else:
        col = t64[4]
    ref_img = torch_raster(m2, con, col, t64[3], t64[5], aux["tile_ranges"].cpu(), aux["sorted_ids"].cpu(),
                           HW, HW, ts)
    np.testing.assert_allclose(img.detach().cpu().numpy(), ref_img.detach().numpy(), atol=1e-4, rtol=1e-4)
    (ref_img * gimg.double()).sum().backward()
    for name, a, b in zip(["means3d", "log_scales", "quats", "opacities", "features", "background"], t32, t64):
        got, want = a.grad.cpu().double().numpy(), b.grad.numpy()
        _assert_grad_close(got, want, name)
        assert np.abs(want).max() > 0, name


@pytest.mark.gpu
def test_render_diff_empty_is_background(cuda_device):
    """No intersection (every Gaussian culled by the gsplat rules): the background, still differentiable."""
    cam, m, s, q, o, c, _ = e2e_scene(20, 32, 0, 3)
    m[:, 2] = -1.0
    bg = torch.tensor([0.1, 0.2, 0.3], device=cuda_device, requires_grad=True)
    with pytest.warns(UserWarning):
        img = ms.render_gaussians_diff(*[x.to(cuda_device) for x in (m, s, q, o, c)], cam, background_color=bg,
                                       backend="cuda_gsplat")
    assert img.shape == (32, 32, 3) and torch.equal(img[5, 7], bg.detach())
    img.sum().backward()
    assert torch.equal(bg.grad, torch.full((3,), 32.0 * 32.0, device=cuda_device))


# ---------------------------------------------------------------- 5. fitting smoke test -----------------------------

@pytest.mark.gpu
def test_fit_small_scene(cuda_device):
    """300 Adam steps of L2 loss from perturbed parameters back towards a rendered target.  Measured on a B200: the
    loss falls 1.39e-2 -> 1.23e-5 (x1127); the test asks for x10."""
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
        loss = ((img - target) ** 2).mean()
        loss.backward()
        if step == 0:
            for p in params:
                assert float(p.grad.abs().sum()) > 0
        opt.step()
        losses.append(float(loss))
    ratio = losses[0] / losses[-1]
    print(f"fit: loss {losses[0]:.3e} -> {losses[-1]:.3e} (x{ratio:.1f})")
    assert ratio >= 10.0, (losses[0], losses[-1])
