"""GPU: the compositing backward at full frame size against the fp64 reference (oracle.raster_bwd_f64), every gradient
entry.

Both sides get identical fp32 inputs (oracle projection and binning).  The upstream gradient is zeroed on the pixels
the reference flags as borderline (a decision within rounding distance of its threshold): the backward is linear in
grad_image and such a pixel then contributes exactly zero to every gradient, which removes the only legitimate
discontinuity.  Every entry e of every gradient must then satisfy

    |got - ref| <= rho * wmag_e + n_e 2^-24 mag_e + 1e-12

mag_e = sum_p |term_p| (the reference's sum of absolute values), wmag_e = sum_p w_p |term_p| with w_p the per-term
rounding-error weight in units of 2^-22 that oracle.c derives from the kernels' arithmetic (alpha's relative error
grows with the exponent's size, the recovered transmittance's with kappa = sum alpha / (1 - alpha) and with the
number of steps), n_e the number of pixels that composited the Gaussian (a count of the fp32 additions, atomics
included).  rho comes from the arithmetic, not from observed errors: 2 x 2^-22 for the pair kernel (ex2.approx,
lg2.approx, rcp.approx; oracle.c's error model is written for it), 4 x 2^-24 for the generic kernel (libdevice expf,
IEEE division), whose alpha error 2^-24 (4 s + 5) fits in the same weights.
"""
import time

import numpy as np
import pytest
import torch

import mojosplat_b200 as ms
from helpers import BWD_RHO, bwd_entry_ratios, oracle_project_scene
from mojosplat_b200 import _lib, rasterization, synthetic
from mojosplat_b200.loss import l1_dssim_loss
from oracle import oracle

pytestmark = pytest.mark.gpu

RHO = BWD_RHO
MASKED_LIMIT = 0.01   # largest fraction of pixels whose upstream gradient may be zeroed as borderline
GRADS = ["means2d", "conics", "colors", "opacities"]

# scene -> (kernels, what it reaches)
CASES = {
    "config3_1m": (("fast", "faithful"), "the bench workload: lists up to ~10 k entries, ~78 batches of 128"),
    "config2_100k": (("fast", "faithful"), "the most pairs per pixel (M ~ 8.4 M)"),
    "config2_opaque": (("fast", "faithful"), "opacities 0.995-1.0: special records, the clamp, early stops"),
    "config2_1917x1079": (("fast",), "partial tiles on both edges"),
    "config3_offscreen": (("fast",), "1 M, a third of the means off screen: border lists > 16 k entries"),
    "big_gaussians": (("fast", "faithful"), "~50 frame-covering Gaussians: millions of pixels per entry"),
    "config2_ts8_c1": (("faithful",), "generic kernel, 8x8 tiles, one channel"),
    "config2_ts8_c4": (("faithful",), "generic kernel, 8x8 tiles, four channels"),
    "config2_ts32_c1": (("faithful",), "generic kernel, 32x32 tiles (opt-in shared memory), one channel"),
    "config2_ts32_c4": (("faithful",), "generic kernel, 32x32 tiles (opt-in shared memory), four channels"),
}


def _big_gaussians(W=1920, H=1080, n_small=2950, n_big=50, seed=7):
    rng = np.random.default_rng(seed)
    N = n_small + n_big
    m2 = np.stack([rng.uniform(0, W, N), rng.uniform(0, H, N)], 1)
    sd = np.concatenate([rng.uniform(1.0, 8.0, (n_small, 2)), rng.uniform(700.0, 1500.0, (n_big, 2))])
    th = rng.uniform(0, np.pi, N)
    cs, sn = np.cos(th), np.sin(th)
    # covariance R diag(sd^2) R^T + 0.3 I, conic = its inverse
    cxx = cs * cs * sd[:, 0] ** 2 + sn * sn * sd[:, 1] ** 2 + 0.3
    cyy = sn * sn * sd[:, 0] ** 2 + cs * cs * sd[:, 1] ** 2 + 0.3
    cxy = cs * sn * (sd[:, 0] ** 2 - sd[:, 1] ** 2)
    det = cxx * cyy - cxy * cxy
    con = np.stack([cyy / det, -cxy / det, cxx / det], 1)
    rad = np.ceil(3.33 * np.sqrt(np.stack([cxx, cyy], 1)))
    op = np.concatenate([rng.uniform(0.05, 0.95, n_small), rng.uniform(0.01, 0.08, n_big)])
    col = rng.uniform(0, 1, (N, 3))
    dep = rng.uniform(1.0, 50.0, N)
    f = np.float32
    return m2.astype(f), con.astype(f), dep.astype(f), rad.astype(np.int32), op.astype(f), col.astype(f), W, H


def _scene(case):
    ts, C = 16, 3
    if case == "big_gaussians":
        m2, con, dep, rad, op, col, W, H = _big_gaussians()
        bg = np.array([0.1, 0.2, 0.3], np.float32)
    else:
        sc = synthetic.make_scene("config3_1m_1080p" if case.startswith("config3") else "config2_100k_1080p")
        gen = torch.Generator().manual_seed(3)
        if case == "config2_opaque":
            sc.opacities = (0.995 + 0.005 * torch.rand(sc.N, generator=gen)).clamp(max=1.0).contiguous()
        elif case == "config2_1917x1079":
            sc.camera = synthetic.make_camera(1917, 1079, 500.0)
        elif case == "config3_offscreen":
            sc.means3d[::3] *= 6.0   # as test_long_list_prepass_is_exact: lists of culled Gaussians in border tiles
        elif "_ts" in case:
            ts, C = int(case.split("_ts")[1].split("_")[0]), int(case.split("_c")[-1])
            sc.colors = torch.rand(sc.N, C, generator=gen).contiguous()
        m2, con, dep, rad = oracle_project_scene(sc)
        op, col, W, H = sc.opacities.numpy(), sc.colors.numpy(), sc.camera.W, sc.camera.H
        bg = np.linspace(0.1, 0.4, C).astype(np.float32)
    ids, ranges = oracle.bin_tiles(m2, rad, dep, H, W, ts)
    return dict(m2=m2, con=con, col=col, op=op, bg=bg, ranges=ranges, ids=ids, W=W, H=H, ts=ts, C=C)


def _camera(s):
    return ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=s["H"], W=s["W"], fx=500.0, fy=500.0, cx=s["W"] / 2,
                     cy=s["H"] / 2)


def _dev(s, d):
    return {k: torch.from_numpy(np.ascontiguousarray(s[k])).to(d) for k in ("m2", "con", "col", "op", "bg", "ranges",
                                                                           "ids")}


def _gpu_grads(s, t, gimg, mode):
    p = [t[k].clone().requires_grad_(True) for k in ("m2", "con", "col", "op", "bg")]
    img = rasterization.rasterize_gaussians_diff(*p, t["ranges"], t["ids"], _camera(s), s["ts"], mode=mode)
    img.backward(gimg)
    torch.cuda.synchronize()
    return {n: x.grad.double().cpu().numpy() for n, x in zip(GRADS + ["background"], p)}


def _raw_forward(s, t, mode, d):
    """(final_T, last_idx) of the training-side forward, straight through the C ABI (no tile order, no workspace)."""
    L = _lib.load()
    H, W, C = s["H"], s["W"], s["C"]
    image = torch.empty((H, W, C), dtype=torch.float32, device=d)
    final_T = torch.empty((H, W), dtype=torch.float32, device=d)
    last = torch.empty((H, W), dtype=torch.int32, device=d)
    N, M, sp = t["m2"].shape[0], t["ids"].numel(), _lib.stream_ptr(d)
    ptr = _lib.ptr
    if mode == "fast":
        rc = L.bsplat_rasterize_fwd_train_fast(N, ptr(t["m2"]), ptr(t["con"]), ptr(t["col"]), ptr(t["op"]),
                                               ptr(t["bg"]), ptr(t["ranges"]), None, ptr(t["ids"]), M, W, H,
                                               ptr(image), ptr(final_T), ptr(last), None, 0, sp)
    else:
        rc = L.bsplat_rasterize_fwd_train(N, C, ptr(t["m2"]), ptr(t["con"]), ptr(t["col"]), ptr(t["op"]),
                                          ptr(t["bg"]), ptr(t["ranges"]), ptr(t["ids"]), M, W, H, s["ts"], ptr(image),
                                          ptr(final_T), ptr(last), sp)
    assert rc == 0
    torch.cuda.synchronize()
    return final_T, last


def _raw_backward_fast_no_order(s, t, final_T, last, gimg, d):
    """bsplat_rasterize_bwd_fast with tile_order = NULL (the Python path always passes an order)."""
    L = _lib.load()
    N, M, ptr = t["m2"].shape[0], t["ids"].numel(), _lib.ptr
    out = [torch.zeros_like(t[k]) for k in ("m2", "con", "col", "op")]
    ws = torch.empty((L.bsplat_rasterize_workspace_bytes(N),), dtype=torch.uint8, device=d)
    rc = L.bsplat_rasterize_bwd_fast(N, ptr(t["m2"]), ptr(t["con"]), ptr(t["col"]), ptr(t["op"]), ptr(t["bg"]),
                                     ptr(t["ranges"]), None, ptr(t["ids"]), M, s["W"], s["H"], ptr(final_T), ptr(last),
                                     ptr(gimg), ptr(out[0]), ptr(out[1]), ptr(out[2]), ptr(out[3]), ptr(ws), ws.numel(),
                                     _lib.stream_ptr(d))
    assert rc == 0
    torch.cuda.synchronize()
    return {n: x.double().cpu().numpy() for n, x in zip(GRADS, out)}


def _upstreams(s, t, mode, d):
    """Random normal (signed: it cancels), and the real dL/dimg of l1_dssim_loss against a perturbed target."""
    H, W, C = s["H"], s["W"], s["C"]
    gen = torch.Generator().manual_seed(11)
    yield "randn", torch.randn(H, W, C, generator=gen).to(d)
    with torch.no_grad():
        img = rasterization.rasterize_gaussians_diff(t["m2"], t["con"], t["col"], t["op"], t["bg"], t["ranges"],
                                                     t["ids"], _camera(s), s["ts"], mode=mode)
    target = (img + 0.05 * torch.randn(H, W, C, generator=gen).to(d)).clamp(0.0, 1.0)
    x = img.clone().requires_grad_(True)
    l1_dssim_loss(x, target).backward()
    yield "l1_dssim", x.grad.detach().contiguous()


def _report(tag, ratios, masked, secs):
    allr = np.concatenate([r.ravel() for r in ratios.values()])
    worst = {n: float(r.max()) for n, r in ratios.items()}
    print(f"\n[bwd-full {tag}] max err/bound {allr.max():.3g}  p99.9 {np.quantile(allr, 0.999):.3g}  "
          f"masked {masked:.2e}  {secs:.1f}s  per gradient {worst}")
    for n, r in ratios.items():
        assert r.max() <= 1.0, (tag, n, float(r.max()), np.unravel_index(int(r.argmax()), r.shape))


@pytest.mark.parametrize("case", list(CASES))
def test_backward_full_size_every_entry(cuda_device, case):
    kernels, _ = CASES[case]
    t0 = time.time()
    s = _scene(case)
    t = _dev(s, cuda_device)
    H, W = s["H"], s["W"]
    if case == "config3_offscreen":
        r = s["ranges"].reshape(-1, 2)
        assert int((r[:, 1] - r[:, 0]).max()) > 16384
    fwd = {}
    for up_name, gimg in _upstreams(s, t, kernels[0], cuda_device):
        ref = oracle.raster_bwd_f64(s["m2"], s["con"], s["col"], s["op"], s["bg"], s["ranges"], s["ids"], W, H,
                                    s["ts"], gimg.cpu().numpy(), mask_borderline=True)
        border = ref["borderline"]
        masked = float(border.mean())
        assert masked <= MASKED_LIMIT, (case, masked)
        gm = gimg.clone()
        gm[torch.from_numpy(border).to(cuda_device)] = 0.0
        for mode in kernels:
            t1 = time.time()
            got = _gpu_grads(s, t, gm, mode)
            _report(f"{case} {mode} {up_name}", bwd_entry_ratios(got, ref, RHO[mode], H * W), masked,
                    time.time() - t1)
            if mode not in fwd:
                # the forward's transmittance (and, for the generic kernel, the last composited index) on the
                # unmasked pixels: the borderline flag does not depend on the upstream gradient
                fwd[mode] = final_T, last = _raw_forward(s, t, mode, cuda_device)
                keep = ~border
                T_got = final_T.double().cpu().numpy()
                T_bound = RHO[mode] * (2.0 + ref["weight"]) * ref["final_T"] + 1e-12
                assert (np.abs(T_got - ref["final_T"])[keep] <= T_bound[keep]).all(), (case, mode)
                if mode == "faithful":
                    assert np.array_equal(last.cpu().numpy()[keep], ref["last_idx"][keep]), (case, mode)
        if case == "config2_100k":
            raw = _raw_backward_fast_no_order(s, t, *fwd["fast"], gm, cuda_device)
            _report(f"{case} fast C-ABI tile_order=NULL {up_name}", bwd_entry_ratios(raw, ref, RHO["fast"], H * W),
                    masked, 0.0)
    print(f"[bwd-full {case}] {CASES[case][1]}; max kappa {ref['kappa'].max():.1f}, "
          f"max weight {ref['weight'].max():.0f}, max count {int(ref['count'].max())}, total {time.time() - t0:.1f}s")
