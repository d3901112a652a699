"""compute-sanitizer workload: every kernel of libbsplat.so on small scenes (both rule sets, packed layout, row bands,
long-list pre-pass, sync-free / captured frames, backward with and without the absolute mean gradient, SH, projection /
SH backward, SSIM + L1 loss, densification, MCMC noise / relocation / sample-add).  Run as

    compute-sanitizer --tool memcheck  python benchmarks/sanitize.py
    compute-sanitizer --tool racecheck python benchmarks/sanitize.py
    compute-sanitizer --tool synccheck python benchmarks/sanitize.py

and keep the summaries under profiles/ (the raster staging double buffer, the onesweep / scan look-back chains and
the multi-CTA tile finish are the kernels that need it)."""
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch

import mojosplat_b200 as ms
from mojosplat_b200 import binning, parallel, rasterization, synthetic
from mojosplat_b200.pipeline import GraphRenderer, OverlappedPipeline

dev = torch.device("cuda:0")
small = "--small" in sys.argv
for cfg, N, sem in [("config1_1k_256", None, "cuda"), ("config3_1m_1080p", 8000 if small else 30000, "cuda"),
                    ("config3_1m_1080p", 8000 if small else 30000, "cuda_gsplat"),
                    ("config2_100k_1080p", 1500 if small else 3000, "cuda")]:
    sc = synthetic.make_scene(cfg, N=N)
    g = [t.to(dev) for t in sc.gaussians()]
    bg = sc.background.to(dev)
    img = ms.render_gaussians(*g, sc.camera, background_color=bg, backend=sem)
    semv = ms.projection.CUDA_BACKENDS[sem]
    img2, aux = ms.render_fused(*g, sc.camera, bg, 16, semantics=semv, return_aux=True)
    img2, aux = ms.render_fused(*g, sc.camera, bg, 16, semantics=semv, return_aux=True)
    img3, _ = ms.render_fused(*g, sc.camera, bg, 16, semantics=semv, return_aux=True, packed=True)
    assert torch.equal(img2, img3)
    # single-level binning of the frame's stage outputs: the same lists as the frame's two-level binning
    ids1, ranges1 = binning.bin_gaussians_to_tiles_cuda(aux["means2d"], aux["radii"], aux["depths"], sc.camera.H,
                                                        sc.camera.W, 16, semantics=semv, algo="single")
    assert torch.equal(ranges1, aux["tile_ranges"]) and torch.equal(ids1, aux["sorted_ids"])
    for mode in ["fast", "faithful", "fast_nocull"]:
        rasterization.rasterize_gaussians_cuda(aux["means2d"], aux["conics"], g[4], g[3], bg, aux["tile_ranges"],
                                               aux["sorted_ids"], sc.camera, 16, mode=mode)
    # small tiles: more than 65 536 tile ids (3-pass tile sort), stage-level binning with and without compaction
    for ts, packed in ((4, False), (4, True), (16, True)):
        binning.bin_gaussians_to_tiles_cuda(aux["means2d"], aux["radii"], aux["depths"], sc.camera.H, sc.camera.W, ts,
                                            semantics=semv, packed=packed)
    t = [aux["means2d"].clone().requires_grad_(True), aux["conics"].clone().requires_grad_(True),
         g[4].clone().requires_grad_(True), g[3].clone().requires_grad_(True)]
    for mode in ("fast", "faithful"):  # pair-layout kernels / generic kernels
        out = rasterization.rasterize_gaussians_diff(*t, bg, aux["tile_ranges"], aux["sorted_ids"], sc.camera, 16,
                                                     mode=mode)
        out.sum().backward()
        # ... and their AbsGS instantiations (bsplat_rasterize_bwd[_fast]_abs)
        absgrad = torch.zeros_like(aux["means2d"])
        out = rasterization.rasterize_gaussians_diff(*t, bg, aux["tile_ranges"], aux["sorted_ids"], sc.camera, 16,
                                                     mode=mode, means2d_absgrad=absgrad)
        out.sum().backward()
        assert bool(torch.isfinite(absgrad).all()) and bool((absgrad >= 0).all())
    pipe = OverlappedPipeline(dev, sc.N, sc.camera.W, sc.camera.H, semantics=semv, m_capacity=200 * sc.N + 4096)
    cams = synthetic.orbit_cameras(4, sc.camera.W, sc.camera.H, sc.camera.fx)
    pipe.render(*g, cams, bg); pipe.check()
    tiny = OverlappedPipeline(dev, sc.N, sc.camera.W, sc.camera.H, m_capacity=500)
    tiny.render(*g, cams[:2], bg); tiny.check()
    gr = GraphRenderer(*g, sc.camera, bg, semantics=semv, m_capacity=200 * sc.N + 4096)
    gr.render(cams[1]); gr.check()
    full = ms.render_fused(*g, sc.camera, bg, 16, semantics=semv)
    assert torch.equal(parallel.render_frame_row_split(*g, sc.camera, bg, semantics=semv), full)
    rb_img = torch.zeros_like(full)
    th = (sc.camera.H + 15) // 16
    for bi, band in enumerate(((0, th // 3), (th // 3, th // 3), (th // 3, th // 2), (th // 2, th))):   # (one empty band)
        # (torch rules: bands 0..2 through the band pre-test + candidate-list projection, the last one without)
        rb = parallel.RowBandRenderer(sc.N, sc.camera, semantics=semv, pretest=bi < 3, m_capacity=200 * sc.N + 4096)
        rb.bands = [band]
        rb.render(*g, sc.camera, bg); rb.check()
        r0, r1 = band[0] * 16, min(band[1] * 16, sc.camera.H)
        rb_img[r0:r1] = rb.image[r0:r1]
    assert torch.equal(rb_img, full)
    coeffs = torch.randn(sc.N, 16, 3, device=dev)
    ms.eval_sh(3, coeffs, g[0], sc.camera)
    # differentiable frame from the 3D parameters: SH, projection and raster backward
    p3 = [x.clone().requires_grad_(True) for x in (g[0], g[1], g[2], coeffs)]
    ms.render_gaussians_diff(p3[0], p3[1], p3[2], g[3], p3[3], sc.camera, sh_degree=3, background_color=bg,
                             backend=sem).sum().backward()
    # photometric loss: fused SSIM + L1 forward (with the gradient maps) and backward
    li = img2.detach().clone().requires_grad_(True)
    ms.l1_dssim_loss(li, img.detach()).backward()
    # adaptive density control: statistics, plan and one apply over every tensor role (clones, splits and prunes)
    st = ms.DensifyStats(sc.N, dev)
    st.accumulate(torch.randn(sc.N, 2, device=dev) * 1e-3, aux["radii"], sc.camera.W, sc.camera.H)
    dp = dict(means3d=g[0], scales=g[1], quats=g[2], opacities=g[3], colors=g[4], sh=coeffs)
    dp = {k: v.clone().requires_grad_(True) for k, v in dp.items()}
    dopt = torch.optim.Adam(list(dp.values()))
    for v in dp.values():
        v.grad = torch.ones_like(v)
    dopt.step()
    dnew, dcounts = ms.densify_and_prune(dp, st, 1.0, min_opacity=0.3, optimizer=dopt)
    assert dcounts["n_out"] == dnew["sh"].shape[0] > 0
    # MCMC densification: noise, relocation (in place, Adam state zeroed) and sample-add (out of place)
    mp = {k: v.detach().clone().requires_grad_(True) for k, v in dnew.items()}
    mopt = torch.optim.Adam(list(mp.values()))
    for v in mp.values():
        v.grad = torch.ones_like(v)
    mopt.step()
    ms.mcmc_inject_noise(mp, 1e3)
    mnew, mcounts = ms.mcmc_refine(mp, cap_max=2 * dcounts["n_out"], min_opacity=0.5, optimizer=mopt)
    assert mcounts["n_relocated"] > 0 and mcounts["n_out"] == mnew["sh"].shape[0] > dcounts["n_out"]
    torch.cuda.synchronize()
    print(cfg, sem, "ok", float(img.mean()), flush=True)
