"""One training step at config 3 (1 M Gaussians @1920x1080) through render_gaussians_diff:
render_gaussians_diff(...) -> (img * g).sum().backward(), once with RGB features and once with random degree-3 SH
coefficients ([N, 16, 3]).  CUDA events, the L2 overwritten (512 MiB memset) before every timed step and kernel
(the raster backward, timed through its autograd wrapper, back to back after one memset).

Prints one JSON line: steps/s, forward / backward ms, the backward split into its three kernels (each timed alone
through its C entry point on the tensors of the same step: raster bwd, projection bwd, SH bwd), and the bytes the
projection and SH backward kernels have to move with their fraction of the HBM peak (MEASURED_PEAKS.json if present,
else the fallback bench.py uses).

    python benchmarks/train_step.py [--steps 20] [--warmup 3]
"""
import argparse
import json
import subprocess
import sys
from ctypes import byref, c_float
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch

import mojosplat_b200 as ms
from mojosplat_b200 import _lib, rasterization, synthetic
from mojosplat_b200.sh import camera_position

PROJ_BWD_BYTES = 72 + 40          # per Gaussian: means3d, log_scales, quats, radii, v_means2d, v_conics, v_depths in
SH3_BWD_BYTES = 4 * (48 + 3 + 3) + 4 * (48 + 3)   # coeffs, means3d, v_colors in; v_coeffs, v_means3d out (K = 16)


def hbm_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30)
        return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unknown"
    except Exception:
        return "unknown"


def timed(fn, flush, reps):
    """Mean device ms of fn() over reps calls (after one untimed call), the L2 overwritten before each."""
    fn()
    total = 0.0
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    return total / reps


def timed_back_to_back(fn, flush, reps):
    """Mean device ms of fn() over reps calls issued back to back between two events (the L2 overwritten once before):
    for calls whose host-side cost (autograd) would otherwise show up as idle device time after each flush."""
    fn()
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def run(sc, use_sh, steps, warmup, flush, dev):
    L = _lib.load()
    N = sc.N
    m, s, q, o, c = [t.to(dev) for t in sc.gaussians()]
    feats = (torch.randn(N, 16, 3, generator=torch.Generator().manual_seed(3)) * 0.3).to(dev) if use_sh else c
    params = [t.clone().requires_grad_(True) for t in (m, s, q, o, feats)]
    cam, bg = sc.camera, sc.background.to(dev)
    gimg = torch.randn(cam.H, cam.W, 3, generator=torch.Generator().manual_seed(5)).to(dev)
    deg = 3 if use_sh else None

    fwd, bwd = [], []
    for k in range(warmup + steps):
        for p in params:
            p.grad = None
        flush.zero_()
        e0, e1, e2 = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e0.record()
        img, aux = ms.render_gaussians_diff(*params, cam, sh_degree=deg, background_color=bg, return_aux=True)
        e1.record()
        (img * gimg).sum().backward()
        e2.record()
        torch.cuda.synchronize()
        if k >= warmup:
            fwd.append(e0.elapsed_time(e1)); bwd.append(e1.elapsed_time(e2))
    fwd_ms, bwd_ms = sum(fwd) / steps, sum(bwd) / steps

    # the three backward kernels alone, through their entry points, on this step's tensors
    sp = _lib.stream_ptr(dev)
    reps = max(steps, 10)
    t = [aux["means2d"].detach().clone().requires_grad_(True), aux["conics"].detach().clone().requires_grad_(True),
         (ms.eval_sh(3, feats, m, cam) if use_sh else feats).detach().clone().requires_grad_(True),
         o.clone().requires_grad_(True)]
    out = rasterization.rasterize_gaussians_diff(*t, bg, aux["tile_ranges"], aux["sorted_ids"], cam, 16)
    raster_ms = timed_back_to_back(lambda: out.backward(gimg, retain_graph=True), flush, reps)

    cam_s = _lib.camera_struct(cam)
    gm2, gcon, gdep = torch.randn(N, 2, device=dev), torch.randn(N, 3, device=dev), torch.randn(N, device=dev)
    vm, vs, vq = torch.empty(N, 3, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, 4, device=dev)
    radii = aux["radii"]

    def proj_bwd():
        _lib.check(L.bsplat_project_bwd(N, _lib.ptr(m), _lib.ptr(s), _lib.ptr(q), byref(cam_s), 0.3, _lib.SEM_TORCH,
                                        _lib.ptr(radii), _lib.ptr(gm2), _lib.ptr(gcon), _lib.ptr(gdep), _lib.ptr(vm),
                                        _lib.ptr(vs), _lib.ptr(vq), sp), "bsplat_project_bwd")
    proj_ms = timed(proj_bwd, flush, reps)
    peak, peak_src = hbm_peak_gbs()
    res = dict(features="sh3" if use_sh else "rgb", steps_per_s=round(1000.0 / (fwd_ms + bwd_ms), 2),
               forward_ms=round(fwd_ms, 4), backward_ms=round(bwd_ms, 4), raster_bwd_ms=round(raster_ms, 4),
               projection_bwd_ms=round(proj_ms, 4), projection_bwd_bytes=PROJ_BWD_BYTES * N,
               projection_bwd_frac_hbm=round(PROJ_BWD_BYTES * N / (proj_ms * 1e-3) / (peak * 1e9), 3))
    if use_sh:
        pos = camera_position(cam)
        cpos = (c_float * 3)(float(pos[0]), float(pos[1]), float(pos[2]))
        gcol = torch.randn(N, 3, device=dev)
        vc, vm3 = torch.empty_like(feats), torch.empty(N, 3, device=dev)

        def sh_bwd():
            _lib.check(L.bsplat_sh_bwd(N, 3, 16, _lib.ptr(feats), _lib.ptr(m), byref(cpos), _lib.ptr(gcol),
                                       _lib.ptr(vc), _lib.ptr(vm3), sp), "bsplat_sh_bwd")
        sh_ms = timed(sh_bwd, flush, reps)
        res.update(sh_bwd_ms=round(sh_ms, 4), sh_bwd_bytes=SH3_BWD_BYTES * N,
                   sh_bwd_frac_hbm=round(SH3_BWD_BYTES * N / (sh_ms * 1e-3) / (peak * 1e9), 3))
    res["hbm_peak_gbs"], res["hbm_peak_source"] = peak, peak_src
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("train_step.py needs a CUDA device")
    dev = torch.device("cuda:0")
    sc = synthetic.make_scene("config3_1m_1080p")
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    out = dict(workload="config3_1m_1080p", N=sc.N, gpu=torch.cuda.get_device_name(dev), power_limit=power_limit(),
               steps=args.steps, l2="512 MiB memset before every timed step / projection and SH kernel; raster bwd back to back after one")
    out["rgb"] = run(sc, False, args.steps, args.warmup, flush, dev)
    out["sh3"] = run(sc, True, args.steps, args.warmup, flush, dev)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
