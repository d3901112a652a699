"""The photometric training loss on the GPU: fused SSIM + L1 (bsplat_ssim_fwd / bsplat_ssim_bwd) against the same loss
written in torch (3DGS's `ssim` with five grouped 11x11 `conv2d`s, plus `abs().mean()`, fp32, autograd backward).

Images 1920x1080x3 (config 3) and 3840x2160x3 (config 5), random in [0, 1]: the loss's cost does not depend on the
pixel values.  CUDA events; the L2 is overwritten (512 MiB memset) before every timed call, because a 1080p pair fits in
the 126 MB L2.  Reported per size:
  - fused forward (ssim_fwd_kernel + ssim_finish_kernel, with the gradient maps) and fused backward kernel times,
    through the C entry points;
  - fused loss forward + backward through `l1_dssim_loss(...).backward()`, and the torch loss forward + backward (the
    baseline), on the same inputs;
  - algorithmic bytes and FP32 instructions per element, with each kernel's share of the HBM peak (MEASURED_PEAKS.json
    if present, else 6.65 TB/s) and of the FFMA issue rate measured in this run (bsplat_microbench).
And one config-3 training step (render_gaussians_diff -> loss -> backward, 1 M Gaussians @1080p) with either loss.

    python benchmarks/loss_step.py [--reps 50] [--steps 20] [--warmup 3]
"""
import argparse
import json
import math
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "benchmarks"))
import torch
import torch.nn.functional as F

import mojosplat_b200 as ms
from mojosplat_b200 import _lib, synthetic
from train_step import hbm_peak_gbs, power_limit, timed

# per image element (H * W * C):
FWD_BYTES = 4 + 4 + 3 * 4          # img, target in; the three gradient maps out
BWD_BYTES = 3 * 4 + 4 + 4 + 4      # maps, img, target in; v_img out
# FP32 instructions per element, an FMA counted once: the products (3), two 11-tap passes over five planes (110) and the
# SSIM value, its derivatives and the L1 term (~35) forward; two 11-tap passes over three planes (66) and the
# combination (~8) backward.  The kernels execute more: the horizontal pass also runs over the 10 halo rows of a
# 32-row tile (x 42 / 32).
FWD_OPS = 3 + 2 * 5 * 11 + 35
BWD_OPS = 2 * 3 * 11 + 8


def torch_l1_dssim(img, target, lam=0.2):
    """3DGS's loss in torch on (H, W, C) images: (1 - lam) mean|x - y| + lam (1 - ssim), ssim with 11x11 conv2d."""
    C = img.shape[-1]
    g = torch.tensor([math.exp(-(x - 5) ** 2 / float(2 * 1.5 ** 2)) for x in range(11)])
    g = g / g.sum()
    w = (g[:, None] @ g[None, :]).expand(C, 1, 11, 11).contiguous().to(img.device)
    x, y = img.permute(2, 0, 1)[None], target.permute(2, 0, 1)[None]
    mu1 = F.conv2d(x, w, padding=5, groups=C)
    mu2 = F.conv2d(y, w, padding=5, groups=C)
    mu1_sq, mu2_sq, mu1_mu2 = mu1.pow(2), mu2.pow(2), mu1 * mu2
    sigma1_sq = F.conv2d(x * x, w, padding=5, groups=C) - mu1_sq
    sigma2_sq = F.conv2d(y * y, w, padding=5, groups=C) - mu2_sq
    sigma12 = F.conv2d(x * y, w, padding=5, groups=C) - mu1_mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    ssim_map = ((2 * mu1_mu2 + C1) * (2 * sigma12 + C2)) / ((mu1_sq + mu2_sq + C1) * (sigma1_sq + sigma2_sq + C2))
    return (1.0 - lam) * (img - target).abs().mean() + lam * (1.0 - ssim_map.mean())


def ffma_rate(L, dev):
    """FFMA lane-instructions per second (FFMA chain micro-benchmark, as bench.py measures it)."""
    out = torch.empty(1, dtype=torch.float32, device=dev)
    blocks, iters = 148 * 8, 8192
    best = 1e9
    for _ in range(4):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(L.bsplat_microbench(0, blocks, iters, _lib.ptr(out), _lib.stream_ptr(dev)), "microbench")
        b.record()
        torch.cuda.synchronize(dev)
        best = min(best, a.elapsed_time(b))
    return blocks * 256 * 8 * iters / (best * 1e-3)


def loss_times(H, W, C, reps, flush, dev, hbm, ffma):
    L = _lib.load()
    gen = torch.Generator().manual_seed(H)
    img = torch.rand(H, W, C, generator=gen).to(dev)
    target = torch.rand(H, W, C, generator=gen).to(dev)
    n = H * W * C
    out2 = torch.empty(2, device=dev)
    maps = torch.empty(3, H, W, C, device=dev)
    v_out2 = torch.tensor([-0.2, 0.8], device=dev)
    v_img = torch.empty_like(img)
    ws = torch.empty(L.bsplat_ssim_workspace_bytes(H, W, C), dtype=torch.uint8, device=dev)
    sp = _lib.stream_ptr(dev)

    def fwd():
        _lib.check(L.bsplat_ssim_fwd(H, W, C, _lib.ptr(img), _lib.ptr(target), _lib.ptr(out2), _lib.ptr(maps),
                                     _lib.ptr(ws), ws.numel(), None, sp), "bsplat_ssim_fwd")

    def bwd():
        _lib.check(L.bsplat_ssim_bwd(H, W, C, _lib.ptr(img), _lib.ptr(target), _lib.ptr(maps), _lib.ptr(v_out2),
                                     _lib.ptr(v_img), sp), "bsplat_ssim_bwd")

    def fused_loss():
        x = img.clone().requires_grad_(True)
        ms.l1_dssim_loss(x, target).backward()

    def torch_loss():
        x = img.clone().requires_grad_(True)
        torch_l1_dssim(x, target).backward()

    fwd_ms, bwd_ms = timed(fwd, flush, reps), timed(bwd, flush, reps)
    fused_ms, torch_ms = timed(fused_loss, flush, reps), timed(torch_loss, flush, reps)
    # the two losses agree (value and gradient) on these inputs
    x1, x2 = img.clone().requires_grad_(True), img.clone().requires_grad_(True)
    l1 = ms.l1_dssim_loss(x1, target); l1.backward()
    l2 = torch_l1_dssim(x2, target); l2.backward()
    gmax = float(x2.grad.abs().max())

    def share(nbytes, ops, ms_):
        t_hbm = nbytes * n / (hbm * 1e9)
        t_fp32 = ops * n / ffma
        bound = "fp32" if t_fp32 > t_hbm else "hbm"
        return dict(bytes=nbytes * n, fp32_instr=ops * n, frac_hbm=round(t_hbm / (ms_ * 1e-3), 3),
                    frac_fp32=round(t_fp32 / (ms_ * 1e-3), 3), bound=bound,
                    least_time_us=round(max(t_hbm, t_fp32) * 1e6, 2))

    return dict(shape=[H, W, C], elements=n,
                fused_fwd_ms=round(fwd_ms, 4), fused_bwd_ms=round(bwd_ms, 4),
                fused_fwd=share(FWD_BYTES, FWD_OPS, fwd_ms), fused_bwd=share(BWD_BYTES, BWD_OPS, bwd_ms),
                fused_loss_fwd_bwd_ms=round(fused_ms, 4),
                torch_baseline_fwd_bwd_ms=round(torch_ms, 4),
                torch_baseline="3DGS loss in torch fp32: 5 grouped 11x11 conv2d + elementwise, autograd backward",
                speedup_vs_torch=round(torch_ms / fused_ms, 2),
                loss_abs_diff_vs_torch=float((l1 - l2).detach().abs()),
                grad_max_abs_diff_vs_torch_rel=float((x1.grad - x2.grad).abs().max()) / max(gmax, 1e-30))


def train_steps(sc, loss_fn, steps, warmup, flush, dev):
    m, s, q, o, c = [t.to(dev) for t in sc.gaussians()]
    params = [t.clone().requires_grad_(True) for t in (m, s, q, o, c)]
    cam, bg = sc.camera, sc.background.to(dev)
    target = torch.rand(cam.H, cam.W, 3, generator=torch.Generator().manual_seed(5)).to(dev)
    times = []
    for k in range(warmup + steps):
        for p in params:
            p.grad = None
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        img = ms.render_gaussians_diff(*params, cam, background_color=bg)
        loss_fn(img, target).backward()
        b.record()
        torch.cuda.synchronize()
        if k >= warmup:
            times.append(a.elapsed_time(b))
    ms_ = sum(times) / steps
    return dict(step_ms=round(ms_, 4), steps_per_s=round(1000.0 / ms_, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("loss_step.py needs a CUDA device")
    dev = torch.device("cuda:0")
    L = _lib.require_device(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    hbm, hbm_src = hbm_peak_gbs()
    ffma = ffma_rate(L, dev)
    out = dict(gpu=torch.cuda.get_device_name(dev), power_limit=power_limit(),
               l2="512 MiB memset before every timed call / step", reps=args.reps,
               hbm_peak_gbs=hbm, hbm_peak_source=hbm_src, ffma_per_s=ffma,
               ffma_source="measured in this run (FFMA chain micro-benchmark, bsplat_microbench)",
               op_count_note="fp32_instr: FP32 instructions per element (FMA = 1) x elements, algorithmic (no halo "
                             "recomputation); frac_fp32 = that count at the FFMA issue rate / kernel time")
    out["config3_1080p"] = loss_times(1080, 1920, 3, args.reps, flush, dev, hbm, ffma)
    out["config5_4k"] = loss_times(2160, 3840, 3, args.reps, flush, dev, hbm, ffma)
    sc = synthetic.make_scene("config3_1m_1080p")
    out["train_step_config3"] = dict(
        workload="config3_1m_1080p, RGB, render_gaussians_diff -> loss -> backward", N=sc.N,
        fused_l1_dssim=train_steps(sc, ms.l1_dssim_loss, args.steps, args.warmup, flush, dev),
        torch_l1_dssim=train_steps(sc, torch_l1_dssim, args.steps, args.warmup, flush, dev))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
