"""Cost of AbsGS's absolute screen-space gradient (``absgrad``) at config 3 (1 M Gaussians, 1080p, SH degree 3).

Two measurements, each alternating the two variants call by call in one run (the order swapped every repetition), with
the L2 overwritten (512 MiB memset) before every timed call or step, CUDA events:
  - the pair-kernel backward alone, ``bsplat_rasterize_bwd_fast`` against ``bsplat_rasterize_bwd_fast_abs``, on the
    same forward's final_T / last_idx and a random upstream gradient (gradient arrays zeroed outside the window);
  - a training step, render_gaussians_diff -> l1_dssim_loss -> backward -> DensifyStats.accumulate, on the signed
    gradient (``aux["means2d"].grad``) against ``absgrad=True`` (``aux["means2d_absgrad"]``).
The signed gradients of the two backwards are compared entry by entry (float atomics: neither run is bit-reproducible).

    python benchmarks/absgrad_step.py [--reps 30] [--steps 20] [--warmup 3] [--out result.json]
"""
import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "benchmarks"))
import torch

import mojosplat_b200 as ms
from mojosplat_b200 import _lib, synthetic
from mojosplat_b200.densify import DensifyStats
from train_step import power_limit


def scene_tensors(sc, dev):
    m, s, q, o, _ = [t.to(dev) for t in sc.gaussians()]
    sh = (torch.randn(sc.N, 16, 3, generator=torch.Generator().manual_seed(3)) * 0.3).to(dev)
    return [m, s, q, o, sh]


def backward_times(sc, dev, flush, reps):
    L = _lib.load()
    m, s, q, o, sh = scene_tensors(sc, dev)
    cam, bg = sc.camera, sc.background.to(dev)
    with torch.no_grad():
        colors = ms.eval_sh(3, sh, m, cam).float().contiguous()
        _, aux = ms.render_gaussians_diff(m, s, q, o, colors, cam, background_color=bg, return_aux=True)
    N, W, H = sc.N, cam.W, cam.H
    m2, con = aux["means2d"].detach().contiguous(), aux["conics"].detach().contiguous()
    ranges, ids = aux["tile_ranges"], aux["sorted_ids"]
    M, p, sp = ids.numel(), _lib.ptr, _lib.stream_ptr(dev)
    order = torch.empty(ranges.shape[0] * ranges.shape[1], dtype=torch.int32, device=dev)
    _lib.check(L.bsplat_tile_order(0, order.numel(), p(ranges), p(order), sp), "bsplat_tile_order")
    ws = torch.empty(L.bsplat_rasterize_workspace_bytes(N), dtype=torch.uint8, device=dev)
    image = torch.empty(H, W, 3, device=dev)
    final_T = torch.empty(H, W, device=dev)
    last = torch.empty(H, W, dtype=torch.int32, device=dev)
    _lib.check(L.bsplat_rasterize_fwd_train_fast(N, p(m2), p(con), p(colors), p(o), p(bg), p(ranges), p(order), p(ids),
                                                 M, W, H, p(image), p(final_T), p(last), p(ws), ws.numel(), sp),
               "bsplat_rasterize_fwd_train_fast")
    gimg = torch.randn(H, W, 3, generator=torch.Generator().manual_seed(5)).to(dev)
    outs = {v: [torch.zeros_like(m2), torch.zeros_like(con), torch.zeros_like(colors), torch.zeros_like(o),
                torch.zeros_like(m2)] for v in ("plain", "abs")}

    def call(v):
        gm, gk, gc, go, ga = outs[v]
        head = (N, p(m2), p(con), p(colors), p(o), p(bg), p(ranges), p(order), p(ids), M, W, H, p(final_T), p(last),
                p(gimg))
        tail = (p(gk), p(gc), p(go), p(ws), ws.numel(), sp)
        if v == "abs":
            return L.bsplat_rasterize_bwd_fast_abs(*head, p(gm), p(ga), *tail)
        return L.bsplat_rasterize_bwd_fast(*head, p(gm), *tail)

    times = {"plain": [], "abs": []}
    for k in range(reps + 1):
        for v in (("plain", "abs") if k % 2 == 0 else ("abs", "plain")):
            for t in outs[v]:
                t.zero_()
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _lib.check(call(v), v)
            b.record()
            torch.cuda.synchronize()
            if k > 0:   # the first round warms both up
                times[v].append(a.elapsed_time(b))
    # outputs of the last round: the signed gradients agree up to the order of the float atomics
    agree = {}
    for i, name in enumerate(("means2d", "conics", "colors", "opacities")):
        x, y = outs["plain"][i].double(), outs["abs"][i].double()
        agree[name] = float(((x - y).abs().max() / y.abs().max().clamp_min(1e-30)))
    ga, gm = outs["abs"][4], outs["abs"][0]
    res = {v: round(sum(t) / len(t), 4) for v, t in times.items()}
    return dict(M=M, plain_ms=res["plain"], abs_ms=res["abs"], abs_over_plain=round(res["abs"] / res["plain"], 4),
                signed_grads_max_diff_over_max=agree, absgrad_finite=bool(torch.isfinite(ga).all()),
                absgrad_ge_signed=bool((ga >= gm.abs() * (1 - 1e-5) - 1e-12).all()))


def step_times(sc, dev, flush, steps, warmup):
    m, s, q, o, sh = scene_tensors(sc, dev)
    params = [t.clone().requires_grad_(True) for t in (m, s, q, o, sh)]
    cam, bg = sc.camera, sc.background.to(dev)
    target = torch.rand(cam.H, cam.W, 3, generator=torch.Generator().manual_seed(5)).to(dev)
    st = DensifyStats(sc.N, dev)
    times = {False: [], True: []}
    for k in range(warmup + steps):
        for absgrad in ((False, True) if k % 2 == 0 else (True, False)):
            for t in params:
                t.grad = None
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            img, aux = ms.render_gaussians_diff(*params, cam, sh_degree=3, background_color=bg, return_aux=True,
                                                absgrad=absgrad)
            if not absgrad:
                aux["means2d"].retain_grad()
            ms.l1_dssim_loss(img, target).backward()
            st.accumulate(aux["means2d_absgrad"] if absgrad else aux["means2d"].grad, aux["radii"], cam.W, cam.H)
            b.record()
            torch.cuda.synchronize()
            if k >= warmup:
                times[absgrad].append(a.elapsed_time(b))
    plain, absg = sum(times[False]) / steps, sum(times[True]) / steps
    return dict(signed_step_ms=round(plain, 4), absgrad_step_ms=round(absg, 4),
                absgrad_over_signed=round(absg / plain, 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("absgrad_step.py needs a CUDA device")
    dev = torch.device("cuda:0")
    _lib.require_device(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    sc = synthetic.make_scene("config3_1m_1080p")
    out = dict(gpu=torch.cuda.get_device_name(dev), power_limit=power_limit(),
               workload="config3_1m_1080p, SH degree 3", N=sc.N,
               l2="512 MiB memset before every timed call / step", order="variants alternated, order swapped per round",
               reps=args.reps, steps=args.steps)
    out["pair_backward"] = backward_times(sc, dev, flush, args.reps)
    torch.cuda.empty_cache()
    out["train_step"] = dict(what="render_gaussians_diff -> l1_dssim_loss -> backward -> DensifyStats.accumulate",
                             **step_times(sc, dev, flush, args.steps, args.warmup))
    line = json.dumps(out)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
