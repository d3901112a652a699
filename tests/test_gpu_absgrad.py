"""AbsGS's absolute screen-space gradient (gsplat's ``absgrad``): ``bsplat_rasterize_bwd[_fast]_abs``,
``rasterize_gaussians_diff(..., means2d_absgrad=)`` and ``render_gaussians_diff(..., absgrad=True)``.

Every entry of the absolute gradient is checked against the fp64 reference (absgrad_ref.c, anchored to autograd in
test_oracle_absgrad.py) with oracle.raster_bwd_f64's per-entry bound of the signed mean gradient,
``rho * wmag + n_e 2^-24 mag + 1e-12``: |sum |x_p| - sum |y_p|| <= sum |x_p - y_p|, so the bound on the signed terms
covers their absolute values, and ``mag`` is >= the absolute sums.  As in test_gpu_raster_bwd_full, the upstream
gradient is zeroed on the reference's borderline pixels.  The argument checks at the top need no GPU.
"""
import ctypes

import numpy as np
import pytest
import torch

import mojosplat_b200 as ms
from absgrad_ref import raster_abs_means2d_f64
from helpers import BWD_RHO, bwd_entry_ratios, oracle_project_scene
from mojosplat_b200 import _lib, rasterization, synthetic
from mojosplat_b200.densify import DensifyStats, densify_and_prune
from mojosplat_b200.loss import l1_dssim_loss
from oracle import oracle
from test_gpu_densify import sparse_fit
from test_gpu_raster_bwd import small_scene
from test_gpu_raster_bwd_full import CASES, MASKED_LIMIT, _camera, _dev, _scene, _upstreams
from test_oracle_raster_bwd import AUTOGRAD_CASES

GRADS = ["means2d", "conics", "colors", "opacities"]
ABSGS_THRESHOLD = 0.0008  # gsplat's grow_grad2d with absgrad=True


# ---------------------------------------------------------------- arguments and ABI (no GPU) -------------------------

@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        _lib.build()
    return _lib.load()


def test_tensor_arguments_rejected_without_gpu():
    N = 5
    m2, con, col, op, bg = torch.zeros(N, 2), torch.zeros(N, 3), torch.zeros(N, 3), torch.zeros(N), torch.zeros(3)
    ranges, ids = torch.zeros(1, 1, 2, dtype=torch.int32), torch.zeros(0, dtype=torch.int32)
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=16, W=16, fx=10.0, fy=10.0, cx=8.0, cy=8.0)
    bad = {"shape": torch.zeros(N, 3), "rows": torch.zeros(N + 1, 2), "dtype": torch.zeros(N, 2, dtype=torch.float64),
           "contiguity": torch.zeros(2, N).t(), "device": torch.zeros(N, 2, device="meta"), "type": np.zeros((N, 2))}
    for name, t in bad.items():
        with pytest.raises(ValueError, match="means2d_absgrad"):
            rasterization.rasterize_gaussians_diff(m2, con, col, op, bg, ranges, ids, cam, means2d_absgrad=t)
    with pytest.raises(ValueError, match="return_aux"):
        ms.render_gaussians_diff(torch.zeros(N, 3), torch.zeros(N, 3), torch.zeros(N, 4), op, col, cam, absgrad=True)


def test_c_abi_rejections_without_gpu(lib):
    """Argument rules of the two _abs entry points: every one of these returns before anything reaches a device."""
    f = [ctypes.c_void_p(0x10000 * (i + 1)) for i in range(16)]
    (m2, con, col, op, bg, ranges, order, ids, fT, last, gimg, gm, gabs, gk, gc, go) = f
    ws, nws = ctypes.c_void_p(0x200000), lib.bsplat_rasterize_workspace_bytes(10)

    def fast(N=10, M=100, m2=m2, gabs=gabs, ws=ws, nws=nws):
        return lib.bsplat_rasterize_bwd_fast_abs(N, m2, con, col, op, bg, ranges, order, ids, M, 32, 32, fT, last, gimg,
                                                 gm, gabs, gk, gc, go, ws, nws, None)

    def generic(N=10, M=100, channels=3, ts=16, gabs=gabs):
        return lib.bsplat_rasterize_bwd_abs(N, channels, m2, con, col, op, bg, ranges, ids, M, 32, 32, ts, fT, last,
                                            gimg, gm, gabs, gk, gc, go, None)

    for call in (fast, generic):
        assert call(gabs=None) == _lib.E_ARG                      # NULL absolute-gradient array, N > 0
        assert call(gabs=None, M=0) == _lib.E_ARG                 # ... checked before the M == 0 early return
        assert call(N=0, gabs=None) == _lib.OK                    # N = 0: nothing to write, nothing launched
        assert call(M=0) == _lib.OK                               # no pairs: nothing launched
        assert call(N=-1) == _lib.E_ARG
    assert fast(m2=ctypes.c_void_p(0x10004)) == _lib.E_ARG           # means2d not 8-byte aligned
    assert fast(ws=ctypes.c_void_p(0x200008)) == _lib.E_WORKSPACE    # workspace not 16-byte aligned
    assert fast(ws=None) == _lib.E_WORKSPACE
    assert fast(nws=nws - 1) == _lib.E_WORKSPACE
    assert generic(channels=5) == _lib.E_ARG
    assert generic(channels=0) == _lib.E_ARG
    assert generic(ts=33) == _lib.E_ARG


# ---------------------------------------------------------------- every entry against the fp64 reference -------------

def _check_abs(got, ref, abs_ref, rho, tag):
    """got: dict of the signed gradients and "abs"; ref: oracle.raster_bwd_f64's result, abs_ref the fp64 absolute
    sums, both for the same (masked) upstream; each entry within the bound of the reference's."""
    assert (ref["mag_means2d"] >= abs_ref * (1 - 1e-12)).all(), tag
    cnt = ref["count"].astype(np.float64)[:, None]
    bound = rho * ref["wmag_means2d"] + cnt * 2.0 ** -24 * ref["mag_means2d"] + 1e-12
    r = np.abs(got["abs"] - abs_ref) / bound
    ratios = bwd_entry_ratios({k: v for k, v in got.items() if k != "abs"}, ref, rho, 0)
    worst = {n: float(x.max()) for n, x in ratios.items()}
    print(f"\n[absgrad {tag}] abs max err/bound {r.max():.3g}; signed {worst}")
    assert r.max() <= 1.0, (tag, float(r.max()), np.unravel_index(int(r.argmax()), r.shape))
    for n, x in ratios.items():
        assert x.max() <= 1.0, (tag, n, float(x.max()))


def _gpu_abs(t, cam, ts, gimg, mode):
    """Signed gradients and the absolute mean gradient of one backward through rasterize_gaussians_diff."""
    p = [t[k].clone().requires_grad_(True) for k in ("m2", "con", "col", "op")]
    absgrad = torch.zeros_like(t["m2"])
    img = rasterization.rasterize_gaussians_diff(*p, t["bg"], t["ranges"], t["ids"], cam, ts, mode=mode,
                                                 means2d_absgrad=absgrad)
    img.backward(gimg)
    torch.cuda.synchronize()
    out = {n: x.grad.double().cpu().numpy() for n, x in zip(GRADS, p)}
    out["abs"] = absgrad.double().cpu().numpy()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("N,HW,ts,C,seed", AUTOGRAD_CASES)
def test_absgrad_small_scenes(cuda_device, N, HW, ts, C, seed):
    """16x16 RGB selects the pair kernel, every other shape the generic one."""
    cam, m2, con, dep, rad, o, c = small_scene(N, HW, seed, C)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, HW, HW, ts)
    bg = np.linspace(0.1, 0.4, C).astype(np.float32)
    gimg = torch.randn(HW, HW, C, generator=torch.Generator().manual_seed(100 + seed)).numpy()
    ref = oracle.raster_bwd_f64(m2, con, c, o, bg, ranges, ids, HW, HW, ts, gimg, mask_borderline=True)
    assert float(ref["borderline"].mean()) <= 0.05
    gm = np.where(ref["borderline"][..., None], np.float32(0), gimg.astype(np.float32))
    s = dict(m2=m2, con=con, col=c, op=o, bg=bg, ranges=ranges, ids=ids)
    got = _gpu_abs(_dev(s, cuda_device), cam, ts, torch.from_numpy(gm).to(cuda_device), "fast")
    abs_ref, _ = raster_abs_means2d_f64(m2, con, c, o, bg, ranges, ids, HW, HW, ts, gm)
    rho = BWD_RHO["fast" if (ts == 16 and C == 3) else "faithful"]
    _check_abs(got, ref, abs_ref, rho, f"N={N} HW={HW} ts={ts} C={C}")
    assert got["abs"].max() > 0


def _config1():
    sc = synthetic.make_scene("config1_1k_256")
    m2, con, dep, rad = oracle_project_scene(sc)
    W, H = sc.camera.W, sc.camera.H
    ids, ranges = oracle.bin_tiles(m2, rad, dep, H, W, 16)
    return dict(m2=m2, con=con, col=sc.colors.numpy(), op=sc.opacities.numpy(), bg=sc.background.numpy(),
                ranges=ranges, ids=ids, W=W, H=H, ts=16, C=3)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["config1", "config2_100k", "big_gaussians"])
def test_absgrad_full_frame(cuda_device, case):
    """Both kernels, both upstream gradients (random normal, and the real d L / d img of l1_dssim_loss)."""
    s = _config1() if case == "config1" else _scene(case)
    kernels = ("fast", "faithful") if case == "config1" else CASES[case][0]
    t = _dev(s, cuda_device)
    H, W = s["H"], s["W"]
    for up_name, gimg in _upstreams(s, t, kernels[0], cuda_device):
        ref = oracle.raster_bwd_f64(s["m2"], s["con"], s["col"], s["op"], s["bg"], s["ranges"], s["ids"], W, H,
                                    s["ts"], gimg.cpu().numpy(), mask_borderline=True)
        border = ref["borderline"]
        assert float(border.mean()) <= MASKED_LIMIT, case
        gm = gimg.clone()
        gm[torch.from_numpy(border).to(cuda_device)] = 0.0
        abs_ref, _ = raster_abs_means2d_f64(s["m2"], s["con"], s["col"], s["op"], s["bg"], s["ranges"], s["ids"], W,
                                            H, s["ts"], gm.cpu().numpy())
        for mode in kernels:
            got = _gpu_abs(t, _camera(s), s["ts"], gm, mode)
            _check_abs(got, ref, abs_ref, BWD_RHO[mode], f"{case} {mode} {up_name}")
        # the statistic is not the signed one: cancellation makes it larger on some of the composited Gaussians
        seen = ref["count"] > 0
        assert (abs_ref[seen] > 2.0 * np.abs(ref["grad_means2d"][seen])).any()


# ---------------------------------------------------------------- cancellation: split with absgrad, kept without -----

def _stripes_case(dev):
    """One large Gaussian at the image centre over vertical stripes that are symmetric about its mean: pixels on the
    two sides pull the mean in opposite directions, so the signed gradient cancels."""
    W = H = 64
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=H, W=W, fx=100.0, fy=100.0, cx=32.0, cy=32.0)
    params = dict(means3d=torch.tensor([[0.0, 0.0, 4.0]]), scales=torch.full((1, 3), -0.7),
                  quats=torch.tensor([[1.0, 0.0, 0.0, 0.0]]), opacities=torch.tensor([0.8]),
                  colors=torch.full((1, 3), 0.5))
    params = {k: v.to(dev).requires_grad_(True) for k, v in params.items()}
    r = (torch.arange(W, dtype=torch.float64) + 0.5 - 32.0).abs()       # distance of the pixel centre from the mean
    stripe = ((r // 3) % 2).float()
    target = stripe.expand(H, W).unsqueeze(-1).expand(H, W, 3).contiguous().to(dev)
    return params, cam, target


def _stats_after_one_view(params, cam, target, absgrad):
    img, aux = ms.render_gaussians_diff(*[params[k] for k in ("means3d", "scales", "quats", "opacities", "colors")],
                                        cam, return_aux=True, absgrad=absgrad)
    aux["means2d"].retain_grad()
    l1_dssim_loss(img, target).backward()
    st = DensifyStats(1, params["means3d"].device)
    st.accumulate(aux["means2d_absgrad"] if absgrad else aux["means2d"].grad, aux["radii"], cam.W, cam.H)
    return st, aux


@pytest.mark.gpu
def test_cancellation_split_with_absgrad_only(cuda_device):
    results = {}
    for absgrad in (False, True):
        params, cam, target = _stripes_case(cuda_device)
        st, aux = _stats_after_one_view(params, cam, target, absgrad)
        assert (aux["means2d"].detach().cpu() - 32.0).abs().max() <= 1e-4   # the stripes' axis of symmetry
        grad2d = float(st.grad2d[0])
        new, counts = densify_and_prune({k: v.detach() for k, v in params.items()}, st, 1.0,
                                        grad_threshold=ABSGS_THRESHOLD,
                                        generator=torch.Generator(device=cuda_device).manual_seed(0))
        results[absgrad] = (grad2d, counts, new["means3d"].shape[0])
    (g_signed, c_signed, n_signed), (g_abs, c_abs, n_abs) = results[False], results[True]
    print(f"\n[absgrad stripes] grad2d signed {g_signed:.3e}, absolute {g_abs:.3e}, threshold {ABSGS_THRESHOLD}")
    assert g_signed < 0.1 * ABSGS_THRESHOLD and g_abs > 10.0 * ABSGS_THRESHOLD
    assert c_signed["n_split"] == 0 and c_signed["n_clone"] == 0 and n_signed == 1
    assert c_abs["n_split"] == 1 and n_abs == 2


# ---------------------------------------------------------------- through render_gaussians_diff ----------------------

def _render_scene(dev):
    g = torch.Generator().manual_seed(21)
    m = torch.randn(300, 3, generator=g) * 0.6
    m[:, 2] = torch.rand(300, generator=g) * 3.0 + 1.5
    s = torch.randn(300, 3, generator=g) * 0.3 - 2.2
    q = torch.nn.functional.normalize(torch.randn(300, 4, generator=g), dim=1)
    o, c = torch.rand(300, generator=g) * 0.68 + 0.3, torch.rand(300, 3, generator=g)
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=96, W=96, fx=60.0, fy=60.0, cx=48.0, cy=48.0)
    params = [x.to(dev).requires_grad_(True) for x in (m, s, q, o, c)]
    bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    target = torch.rand(96, 96, 3, generator=g).to(dev)
    return params, cam, bg, target


@pytest.mark.gpu
def test_render_absgrad_matches_direct_call_and_accumulates(cuda_device):
    params, cam, bg, target = _render_scene(cuda_device)
    img0 = ms.render_gaussians_diff(*params, cam, background_color=bg)
    img, aux = ms.render_gaussians_diff(*params, cam, background_color=bg, return_aux=True, absgrad=True)
    assert "means2d_absgrad" not in ms.render_gaussians_diff(*params, cam, background_color=bg, return_aux=True)[1]
    assert torch.equal(img.detach(), img0.detach())          # the forward is the same kernel: bit for bit
    a = aux["means2d_absgrad"]
    assert a.shape == (300, 2) and a.dtype == torch.float32 and (a == 0).all()
    img.retain_grad()
    loss = l1_dssim_loss(img, target)
    loss.backward(retain_graph=True)
    first = a.clone()
    gimg = img.grad.detach().clone()
    # the same backward straight through the rasterizer on the aux tensors
    direct = torch.zeros_like(a)
    x = [aux["means2d"].detach().clone().requires_grad_(True), aux["conics"].detach(), params[4].detach(),
         params[3].detach(), bg]
    out = rasterization.rasterize_gaussians_diff(*x, aux["tile_ranges"], aux["sorted_ids"], cam, 16,
                                                 means2d_absgrad=direct)
    out.backward(gimg)
    ref = oracle.raster_bwd_f64(x[0].detach().cpu().numpy(), x[1].cpu().numpy(), x[2].cpu().numpy(), x[3].cpu().numpy(),
                                bg.cpu().numpy(), aux["tile_ranges"].cpu().numpy(), aux["sorted_ids"].cpu().numpy(),
                                cam.W, cam.H, 16, gimg.cpu().numpy())
    # two runs of the same kernel on the same inputs differ only in the order of the float atomics
    cnt = ref["count"].astype(np.float64)[:, None]
    bound = torch.from_numpy(2.0 * cnt * 2.0 ** -24 * ref["mag_means2d"] + 1e-12)
    assert ((first.double().cpu() - direct.double().cpu()).abs() <= bound).all()
    assert first.max() > 0
    # a second backward adds the same sums again
    loss.backward()
    assert ((a.double().cpu() - 2.0 * first.double().cpu()).abs() <= 2.0 * bound).all()


@pytest.mark.gpu
def test_render_absgrad_no_overlap_stays_zero(cuda_device):
    params, cam, bg, _ = _render_scene(cuda_device)
    with torch.no_grad():
        params[0][:, 2] = -5.0
    # gsplat rules + every Gaussian behind the camera: no pairs (the torch rules bin a culled row into one tile)
    with pytest.warns(UserWarning, match="No Gaussian overlaps"):
        _, aux = ms.render_gaussians_diff(*params, cam, background_color=bg, backend="cuda_gsplat", return_aux=True,
                                          absgrad=True)
    assert aux["sorted_ids"].numel() == 0
    assert aux["means2d_absgrad"].shape == (300, 2) and (aux["means2d_absgrad"] == 0).all()


# ---------------------------------------------------------------- a short fit with absgrad statistics ---------------

def absgrad_fit(dev, steps=300, every=100):
    """test_gpu_densify.sparse_fit's scene and loop, densifying on the absolute gradient at gsplat's threshold."""
    g = torch.Generator().manual_seed(31)
    N = 3000
    z = torch.rand(N, generator=g) * 2.0 + 2.0
    m = torch.stack([(torch.rand(N, generator=g) * 2 - 1) * 0.66 * z, (torch.rand(N, generator=g) * 2 - 1) * 0.66 * z,
                     z], 1)
    s = torch.randn(N, 3, generator=g) * 0.3 - 3.4
    q = torch.randn(N, 4, generator=g)
    o = torch.rand(N, generator=g) * 0.5 + 0.45
    c = torch.rand(N, 3, generator=g)
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=128, W=128, fx=100.0, fy=100.0, cx=64.0, cy=64.0)
    target = ms.render_gaussians_diff(*[x.to(dev) for x in (m, s, q, o, c)], cam).detach()
    pick = torch.randperm(N, generator=g)[:150]
    params = dict(means3d=m[pick], scales=s[pick] + 1.0, quats=q[pick], opacities=o[pick] * 0 + 0.5, colors=c[pick])
    params = {k: v.to(dev).requires_grad_(True) for k, v in params.items()}
    lrs = dict(means3d=2e-3, scales=1e-2, quats=1e-2, opacities=1e-2, colors=1e-2)
    opt = torch.optim.Adam([{"params": [params[k]], "lr": lrs[k]} for k in params])
    stats = DensifyStats(150, dev)
    gen = torch.Generator(device=dev).manual_seed(5)
    sizes, losses = [150], []
    for step in range(1, steps + 1):
        opt.zero_grad()
        img, aux = ms.render_gaussians_diff(*[params[k] for k in ("means3d", "scales", "quats", "opacities",
                                                                   "colors")], cam, return_aux=True, absgrad=True)
        loss = ms.l1_dssim_loss(img, target)
        loss.backward()
        losses.append(float(loss.detach()))
        stats.accumulate(aux["means2d_absgrad"], aux["radii"], cam.W, cam.H)
        opt.step()
        with torch.no_grad():
            params["opacities"].clamp_(0.0, 1.0)
        if step % every == 0 and step < steps:
            params, _ = densify_and_prune(params, stats, 4.0, grad_threshold=ABSGS_THRESHOLD, optimizer=opt,
                                          generator=gen)
            sizes.append(params["means3d"].shape[0])
    return losses, sizes


@pytest.mark.gpu
def test_training_from_sparse_start_with_absgrad(cuda_device):
    losses, sizes = absgrad_fit(cuda_device)
    loss_n, _ = sparse_fit(cuda_device, False, steps=300)
    print(f"\n[absgrad fit] N {sizes}, loss {losses[0]:.4e} -> {losses[-1]:.4e}; without densification {loss_n:.4e}")
    assert sizes[-1] > sizes[0], sizes
    assert losses[-1] < 0.9 * losses[0]
