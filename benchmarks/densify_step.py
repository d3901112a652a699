"""Adaptive density control on the GPU (DensifyStats, densify_and_prune; bsplat_densify_*) against the same work in torch.

Workloads: config 3 (1 M Gaussians) and config 5's 6 M scene, each with (N, 16, 3) SH coefficients, opacities and Adam
state (exp_avg, exp_avg_sq) for every parameter: 59 floats of parameters and 118 of moments, 708 B per Gaussian.  The
statistics are seeded so that about 10 % of the Gaussians clone, 10 % split and 5 % are pruned.  CUDA events; the L2 is
overwritten (512 MiB memset) before every timed call.  Reported per workload:
  - densify_stats: one accumulate() call against the torch statement of the same update (element-wise ops);
  - densify_and_prune (plan, the one read-back, apply over 15 tensors) against densify_reference, the torch restatement
    of tests/test_gpu_densify.py, on the same inputs, with a check that both give the same outputs;
  - the apply kernel alone through bsplat_densify_apply, with its algorithmic bytes sum_t 4 w_t (N + N') and their
    share of the HBM peak (MEASURED_PEAKS.json if present, else 6.65 TB/s).
And one config-3 training step (render_gaussians_diff -> l1_dssim_loss -> backward, SH degree 3) with and without
DensifyStats.accumulate.

    python benchmarks/densify_step.py [--reps 20] [--steps 20] [--warmup 3]
"""
import argparse
import ctypes
import json
import math
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "benchmarks"))
sys.path.insert(0, str(ROOT / "tests"))
import torch

import mojosplat_b200 as ms
from mojosplat_b200 import _lib, synthetic
from mojosplat_b200.densify import DensifyStats, densify_and_prune
from test_gpu_densify import densify_reference
from train_step import hbm_peak_gbs, power_limit, timed

KEYS = ("means3d", "scales", "quats", "opacities", "sh")


def make_workload(name, dev):
    sc = synthetic.make_scene(name)
    N = sc.N
    g = torch.Generator().manual_seed(7)
    m, s, q, o, _ = sc.gaussians()
    sh = torch.randn(N, 16, 3, generator=g) * 0.3
    params = {k: v.to(dev).contiguous() for k, v in zip(KEYS, (m, s, q, o, sh))}
    state = {(k, sk): torch.randn(params[k].shape, generator=g).abs().to(dev) * 1e-3
             for k in KEYS for sk in ("exp_avg", "exp_avg_sq")}
    high = torch.rand(N, generator=g) < 0.2
    count = torch.full((N,), 5, dtype=torch.int32)
    grad2d = torch.where(high, 5 * 3e-4, 5 * 1e-4).float()
    smax = s.max(dim=1).values
    extent = math.exp(float(smax.median())) / 0.01            # the clone / split cut at the median scale
    min_opacity = float(o.kthvalue(max(1, N // 20)).values)   # ~5 % pruned
    max_radius = torch.randint(0, 40, (N,), generator=g, dtype=torch.int32)
    return N, params, state, grad2d.to(dev), count.to(dev), max_radius.to(dev), extent, min_opacity


def with_optimizer(params, state):
    """A fresh Adam over the params whose state tensors are the given ones (no copies)."""
    ps = {k: v.requires_grad_(True) for k, v in params.items()}
    opt = torch.optim.Adam([{"params": [p], "lr": 1e-3} for p in ps.values()])
    for k, p in ps.items():
        opt.state[p] = {"step": torch.tensor(10.0), "exp_avg": state[(k, "exp_avg")],
                        "exp_avg_sq": state[(k, "exp_avg_sq")]}
    return ps, opt


def timed_setup(setup, fn, flush, reps):
    """Mean device ms of fn(setup()) over reps calls (after one untimed call); setup and the L2 flush are outside."""
    fn(setup())
    total = 0.0
    for _ in range(reps):
        arg = setup()
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn(arg)
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    return total / reps


def densify_times(name, reps, flush, dev, hbm):
    L = _lib.load()
    N, params, state, grad2d, count, max_radius, extent, min_opacity = make_workload(name, dev)
    kw = dict(grad_threshold=2e-4, percent_dense=0.01, min_opacity=min_opacity)

    # ---- statistics: one view ----
    gen = torch.Generator().manual_seed(3)
    v2d = (torch.randn(N, 2, generator=gen) * 1e-6).to(dev)
    radii = torch.randint(0, 30, (N, 2), generator=gen, dtype=torch.int32).to(dev)
    st = DensifyStats(N, dev)
    W, H = 1920, 1080
    stats_ms = timed(lambda: st.accumulate(v2d, radii, W, H), flush, reps)
    tg, tc, tr = torch.zeros(N, device=dev), torch.zeros(N, dtype=torch.int32, device=dev), torch.zeros(
        N, dtype=torch.int32, device=dev)

    def torch_stats():
        rmax = radii.max(dim=1).values
        vis = rmax > 0
        nrm = torch.sqrt((v2d[:, 0] * (W / 2)) ** 2 + (v2d[:, 1] * (H / 2)) ** 2)
        tg.add_(torch.where(vis, nrm, 0.0))
        tc.add_(vis.int())
        torch.maximum(tr, torch.where(vis, rmax, tr), out=tr)
    torch_stats_ms = timed(torch_stats, flush, reps)

    # ---- densify_and_prune against the torch restatement ----
    def setup():
        ps, opt = with_optimizer({k: v.detach() for k, v in params.items()}, state)
        s = DensifyStats(N, dev)
        s.grad2d.copy_(grad2d); s.count.copy_(count); s.max_radius.copy_(max_radius)
        return ps, opt, s

    def fused(arg):
        ps, opt, s = arg
        return densify_and_prune(ps, s, extent, optimizer=opt, generator=torch.Generator(device=dev).manual_seed(1),
                                 **kw)

    def reference(_):
        return densify_reference(params, grad2d, count, max_radius, extent, params["opacities"], state=state,
                                 generator=torch.Generator(device=dev).manual_seed(1), **kw)

    fused_ms = timed_setup(setup, fused, flush, reps)
    ref_ms = timed_setup(lambda: None, reference, flush, max(3, reps // 4))
    # same outputs
    ps, opt, s = setup()
    new, counts = fused((ps, opt, s))
    ref, ref_state, ref_counts, extra = densify_reference(params, grad2d, count, max_radius, extent,
                                                          params["opacities"], state=state,
                                                          generator=torch.Generator(device=dev).manual_seed(1), **kw)
    child = extra["child"]
    agree = counts == ref_counts and all(torch.equal(new[k].detach(), ref[k]) for k in KEYS if k != "means3d") and \
        torch.equal(new["means3d"].detach()[~child], ref["means3d"][~child]) and all(
            torch.equal(opt.state[new[k]][sk], ref_state[(k, sk)]) for k in KEYS for sk in ("exp_avg", "exp_avg_sq"))
    mean_err = float(((new["means3d"].detach()[child].double() - extra["means64"]).abs() / extra["tol_scale"]).max())
    del new, ref, ref_state, extra, ps, opt, s

    # ---- the apply kernel alone ----
    n_out, n_split = counts["n_out"], counts["n_split"]
    ws = torch.empty(L.bsplat_densify_workspace_bytes(N), dtype=torch.uint8, device=dev)
    counts_host = torch.zeros(4, dtype=torch.int64).pin_memory()
    prm = _lib.BsplatDensifyParams()
    prm.grad_threshold = float(torch.tensor(2e-4, dtype=torch.float64).float())
    prm.log_clone_max_scale = float(torch.tensor(math.log(0.01 * extent), dtype=torch.float64).float())
    prm.min_opacity = float(torch.tensor(min_opacity, dtype=torch.float64).float())
    prm.log_max_world_scale, prm.max_screen_radius = math.inf, 0x7fffffff
    sp = _lib.stream_ptr(dev)
    _lib.check(L.bsplat_densify_plan(N, _lib.ptr(grad2d), _lib.ptr(count), _lib.ptr(max_radius),
                                     _lib.ptr(params["scales"]), _lib.ptr(params["opacities"]), ctypes.byref(prm),
                                     _lib.ptr(ws), ws.numel(), None, ctypes.c_void_p(counts_host.data_ptr()), sp),
               "bsplat_densify_plan")
    torch.cuda.synchronize()
    assert counts_host.tolist() == [n_out, counts["n_clone"], n_split, counts["n_pruned"]]
    noise = torch.randn((n_split, 2, 3), device=dev)
    srcs = [(params[k], _lib.DENSIFY_MEANS if k == "means3d" else _lib.DENSIFY_LOG_SCALES if k == "scales"
             else _lib.DENSIFY_COPY) for k in KEYS] + [(state[(k, sk)], _lib.DENSIFY_STATE) for k in KEYS
                                                        for sk in ("exp_avg", "exp_avg_sq")]
    outs = [torch.empty((n_out, *t.shape[1:]), device=dev) for t, _ in srcs]
    desc = (_lib.BsplatDensifyTensor * len(srcs))()
    floats_per_row = 0
    for d, (t, role), o in zip(desc, srcs, outs):
        d.src, d.dst, d.width, d.role = t.data_ptr(), o.data_ptr(), t[0].numel(), role
        floats_per_row += t[0].numel()

    def apply():
        _lib.check(L.bsplat_densify_apply(N, _lib.ptr(ws), _lib.ptr(params["means3d"]), _lib.ptr(params["scales"]),
                                          _lib.ptr(params["quats"]), _lib.ptr(noise), len(srcs), desc, sp),
                   "bsplat_densify_apply")

    def plan():
        _lib.check(L.bsplat_densify_plan(N, _lib.ptr(grad2d), _lib.ptr(count), _lib.ptr(max_radius),
                                         _lib.ptr(params["scales"]), _lib.ptr(params["opacities"]), ctypes.byref(prm),
                                         _lib.ptr(ws), ws.numel(), None, ctypes.c_void_p(counts_host.data_ptr()), sp),
                   "bsplat_densify_plan")
    plan_ms = timed(plan, flush, reps)
    apply_ms = timed(apply, flush, reps)
    apply_bytes = 4 * floats_per_row * (N + n_out)
    return dict(workload=name, N=N, n_out=n_out, n_clone=counts["n_clone"], n_split=n_split,
                n_pruned=counts["n_pruned"], floats_per_row=floats_per_row, bytes_per_row=4 * floats_per_row,
                tensors=len(srcs),
                stats_ms=round(stats_ms, 4), torch_stats_ms=round(torch_stats_ms, 4),
                stats_speedup=round(torch_stats_ms / stats_ms, 2),
                densify_and_prune_ms=round(fused_ms, 4), torch_reference_ms=round(ref_ms, 4),
                densify_speedup=round(ref_ms / fused_ms, 2),
                outputs_agree=bool(agree), split_mean_max_err_over_tol_scale=mean_err,
                plan_kernel_ms=round(plan_ms, 4), apply_kernel_ms=round(apply_ms, 4), apply_bytes=apply_bytes,
                apply_gbs=round(apply_bytes / (apply_ms * 1e-3) / 1e9, 1),
                apply_frac_hbm=round(apply_bytes / (apply_ms * 1e-3) / (hbm * 1e9), 3),
                apply_least_time_ms=round(apply_bytes / (hbm * 1e9) * 1e3, 4))


def train_steps(sc, with_stats, steps, warmup, flush, dev):
    N = sc.N
    m, s, q, o, _ = [t.to(dev) for t in sc.gaussians()]
    sh = (torch.randn(N, 16, 3, generator=torch.Generator().manual_seed(3)) * 0.3).to(dev)
    params = [t.clone().requires_grad_(True) for t in (m, s, q, o, sh)]
    cam, bg = sc.camera, sc.background.to(dev)
    target = torch.rand(cam.H, cam.W, 3, generator=torch.Generator().manual_seed(5)).to(dev)
    st = DensifyStats(N, dev)
    times = []
    for k in range(warmup + steps):
        for p in params:
            p.grad = None
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        img, aux = ms.render_gaussians_diff(*params, cam, sh_degree=3, background_color=bg, return_aux=True)
        if with_stats:
            aux["means2d"].retain_grad()
        ms.l1_dssim_loss(img, target).backward()
        if with_stats:
            st.accumulate(aux["means2d"].grad, aux["radii"], cam.W, cam.H)
        b.record()
        torch.cuda.synchronize()
        if k >= warmup:
            times.append(a.elapsed_time(b))
    ms_ = sum(times) / steps
    return dict(step_ms=round(ms_, 4), steps_per_s=round(1000.0 / ms_, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("densify_step.py needs a CUDA device")
    dev = torch.device("cuda:0")
    _lib.require_device(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    hbm, hbm_src = hbm_peak_gbs()
    out = dict(gpu=torch.cuda.get_device_name(dev), power_limit=power_limit(),
               l2="512 MiB memset before every timed call / step", reps=args.reps,
               hbm_peak_gbs=hbm, hbm_peak_source=hbm_src,
               apply_bytes_note="sum over tensors of 4 w_t (N + N'): every source row read once, every output row "
                                "written once")
    out["config3_1m"] = densify_times("config3_1m_1080p", args.reps, flush, dev, hbm)
    torch.cuda.empty_cache()
    out["config5_6m"] = densify_times("config5_6m_4k", args.reps, flush, dev, hbm)
    torch.cuda.empty_cache()
    sc = synthetic.make_scene("config3_1m_1080p")
    out["train_step_config3"] = dict(
        workload="config3_1m_1080p, SH degree 3, render_gaussians_diff -> l1_dssim_loss -> backward", N=sc.N,
        without_stats=train_steps(sc, False, args.steps, args.warmup, flush, dev),
        with_accumulate=train_steps(sc, True, args.steps, args.warmup, flush, dev))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
