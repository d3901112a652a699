#!/usr/bin/env python
"""bench.py -- frames/s of the forward render (projection -> binning -> rasterization).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores

Workload (BASELINE.json `metric`: frames/s, 1 M Gaussians @1920x1080): the config-3 "garden-sized"
synthetic scene of SURVEY.md 8d, seen from a 64-view orbit whose view 0 is the config-3 pose.  A step
is one frame per rank; ranks render different views (Gaussians are NCCL-broadcast once, no data-path
collective afterwards) -> weak scaling, value = frames of all ranks / max-over-ranks device time.

Prints ONE JSON line (rank 0).  Keys beyond the base contract: `roofline` (dominant kernel = the
rasterizer, bound by FP32 issue rate -- no stage of this path is HBM- or tensor-bound at this size;
SURVEY.md 8d), `roofline_hbm` (the projection kernel against the measured HBM peak), `stages` (per-stage device
times and GB/s), `parity` (the timed workload's view-0 frame against the CPU oracle, computed outside the timed
region), `latency` (single-frame figures), `backward` (training-side rasterizer at the same size), `sharded`
(BASELINE configs 4 and 5 on the same ranks: views/s and band-frame latency), `cpu_baseline`.
`config` is identical for both arms (it names the workload only; how each arm runs it is in `method`).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
_emit = print
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "frames/s, 1M Gaussians @1920x1080"
WORKLOAD = "config3_1m_1080p"
N_VIEWS = 64
DUMP_BYTES = 64_000_000  # bound on what --dump-outputs writes


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=WORKLOAD)
    ap.add_argument("--n-gaussians", type=int, default=None, help="override N (debug only; marks the line)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--semantics", default="torch", choices=["torch", "gsplat"])
    ap.add_argument("--pipeline-depth", type=int, default=2, help="frames in flight per GPU (sync pipeline)")
    ap.add_argument("--pipeline", default="overlapped", choices=["overlapped", "sync"],
                    help="overlapped: sync-free frames, binning(k+1) inside rasterization(k); sync: FramePipeline")
    ap.add_argument("--raster-mode", default="fast", choices=["fast", "fast_nocull"], help="rasterizer kernel (A/B)")
    ap.add_argument("--slots", type=int, default=3, help="workspaces cycled by the overlapped pipeline")
    ap.add_argument("--bin-streams", type=int, default=2, help="high-priority binning streams (overlapped pipeline)")
    ap.add_argument("--no-sharded", action="store_true", help="skip the config-4 / config-5 legs (key `sharded`)")
    ap.add_argument("--no-extras", action="store_true", help="skip parity / backward / sharded (quick timing runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the image of the last timed step (rank 0) to DIR/image.npy "
                         "(float32, H x W x 3; every 2nd row at 4K, to stay within 64 MB): the same arguments "
                         "render the same inputs, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the output of the b200 path only")
    return args


# --------------------------------------------------------------------------------------------
def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


RASTER_KERNEL = "raster_pair_kernel"


def ncu_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/ncu_traffic.json names the report it was read from)."""
    p = ROOT / "profiles" / "ncu_traffic.json"
    if not p.exists():
        return None, None
    d = json.loads(p.read_text()).get(key)
    if not d or d.get("dram_bytes") is None:
        return None, None
    return d["dram_bytes"], d.get("source")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def oracle_frame(sc_np, cam, background, semantics=0):
    from oracle import oracle
    return oracle.render(*sc_np, cam.view_matrix.numpy(), cam.fx, cam.fy, cam.cx, cam.cy, cam.W, cam.H,
                         cam.near, cam.far, background=background, semantics=semantics, return_all=True)


# --------------------------------------------------------------------------------------------
def workload_name(args, sc):
    s = (f"{args.workload}: {sc.N} Gaussians (garden-sized synthetic, SH0 RGB) @{sc.camera.W}x{sc.camera.H}, "
         f"{N_VIEWS}-view orbit (view 0 = config-3 pose)")
    if args.n_gaussians is not None:
        s += " [DEBUG: N overridden, not the BASELINE size]"
    return s


def config_dict(args, sc):
    """Names the workload -- the same dict for this repo's arm and for `--impl reference` (how each arm runs it is in
    `method`, what it measured besides the metric in `latency` / `stages`)."""
    return {"workload": workload_name(args, sc), "n_gaussians": sc.N, "image": f"{sc.camera.W}x{sc.camera.H}",
            "views": N_VIEWS, "channels": 3, "tile_size": 16, "semantics": args.semantics,
            "step": "one full frame (projection -> binning -> rasterization) per rank",
            "l2": "inputs larger than L2: the GPU arm rotates its frames over 3 device copies of the Gaussian arrays "
                  "(3 x 56 MB = 168 MB > 126 MB L2) and streams ~230 MB of intermediates per frame; the CPU arm "
                  "streams the same 56 MB of inputs + ~100 MB of intermediates per frame through the host caches"}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, rank, world):
    """The reference algorithm on the host cores: oracle port (C, OpenMP) of projection.py:285-346,
    binning.py:108-262 and kernels/rasterization.mojo:75-162.  The reference itself is Python + Mojo
    and has no compilable C sources (no oracle/_ref); its own torch binning is a Python loop
    (~3.5 min per frame at this size, BASELINE.md), so the port is the generous baseline.
    All host cores are used whatever the launcher put into OMP_NUM_THREADS (torchrun sets it to 1)."""
    if rank != 0:
        return
    from mojosplat_b200 import synthetic
    from oracle import oracle
    oracle.set_num_threads(host_cores())
    sc = synthetic.make_scene(args.workload, N=args.n_gaussians)
    cams = synthetic.orbit_cameras(N_VIEWS, sc.camera.W, sc.camera.H, sc.camera.fx)
    sc_np = [t.numpy() for t in sc.gaussians()]
    bg = sc.background.numpy()
    cores = oracle.num_threads()
    sem = 0 if args.semantics == "torch" else 1
    # a step = one full frame, like the GPU arm.  A CPU frame takes ~0.3-0.5 s, so the driver's K and W fit a few
    # minutes as they are; only absurd requests are bounded (and the line then says what was really run)
    t0 = time.perf_counter()
    oracle_frame(sc_np, cams[0], bg, sem)
    t_frame = time.perf_counter() - t0
    budget = max(2, int(240.0 / max(t_frame, 1e-3)))
    warm = max(0, min(args.warmup, budget // 4) - 1)   # (the probe frame above is the first warm-up frame)
    steps = max(1, min(args.steps, budget - warm - 1))
    for k in range(warm):
        oracle_frame(sc_np, cams[(k + 1) % N_VIEWS], bg, sem)
    t0 = time.perf_counter()
    for k in range(steps):
        oracle_frame(sc_np, cams[k % N_VIEWS], bg, sem)
    dt = time.perf_counter() - t0
    fps = steps / dt
    sample = (f"{steps} full frames ({sc.N} Gaussians @{sc.camera.W}x{sc.camera.H}, all three stages), "
              f"{warm + 1} warm-up frames"
              + (f"; --steps {args.steps} / --warmup {args.warmup} bounded to ~4 min of CPU time"
                 if steps != args.steps or warm + 1 != args.warmup else ""))
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm + 1, "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, sc),
        "method": {"host": f"CPU only, rank 0, {cores} OpenMP threads", "timing": "wall clock around the K frames"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(json.dumps(line))


def parity_report(img, aux, ref, sc_np, bg_np, cam):
    """View-0 frame of the timed workload against the oracle's (outside the timed region).  Image: max error,
    out-of-tolerance rate (1e-4 + 1e-4 |ref|), PSNR, and the audit of every out-of-tolerance pixel (SURVEY H4:
    reproduced by the oracle with one or two borderline alpha-threshold / saturation decisions flipped, or not)."""
    from oracle import oracle
    img = np.asarray(img); rimg = ref["image"]
    err = np.abs(img - rimg)
    bad = err > (1e-4 + 1e-4 * np.abs(rimg))
    bad_px = np.argwhere(bad.any(axis=-1))
    mse = float(np.mean((img.astype(np.float64) - rimg.astype(np.float64)) ** 2))
    out = {"against": "oracle port (C, fp32) of projection.py / binning.py / rasterization.mojo, same inputs, view 0",
           "max_abs_err": float(err.max()), "frac_bad": float(bad.mean()),
           "psnr": 99.0 if mse == 0 else 10.0 * math.log10(1.0 / mse), "n_outliers": int(bad_px.shape[0]),
           "tolerance": "1e-4 + 1e-4*|ref| (tests/test_rasterization.py:110 of the reference)"}
    if bad_px.shape[0]:
        explained, _ = oracle.raster_audit(ref["means2d"], ref["conics"], sc_np[4], sc_np[3], bg_np, ref["tile_ranges"],
                                           ref["sorted_ids"], cam.W, cam.H, 16, bad_px, img[bad_px[:, 0], bad_px[:, 1]])
        out["n_unexplained"] = int((explained == 0).sum())
        out["outliers_explained_by"] = {"one_flip": int((explained == 1).sum()), "two_flips": int((explained == 2).sum())}
    else:
        out["n_unexplained"] = 0
    out["n_isect"] = [int(aux["n_isect"]), int(ref["sorted_ids"].shape[0])]
    out["means2d_bit_exact"] = bool(np.array_equal(aux["means2d"].cpu().numpy(), ref["means2d"]))
    out["radii_differ"] = int((aux["radii"].cpu().numpy() != ref["radii"]).any(-1).sum())
    out["tile_ranges_bit_exact"] = bool(np.array_equal(aux["tile_ranges"].cpu().numpy(), ref["tile_ranges"]))
    ids = aux.get("sorted_ids")
    out["sorted_ids_bit_exact"] = bool(ids is not None and ids.numel() == ref["sorted_ids"].shape[0]
                                       and np.array_equal(ids.cpu().numpy(), ref["sorted_ids"]))
    return out


# --------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    import mojosplat_b200 as ms
    from mojosplat_b200 import _lib, rasterization, synthetic

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    L = _lib.require_device(dev)  # fails loudly without the .so / an sm_100 device
    # multi-GPU boxes: run this rank, and allocate its pinned host buffers, on the GPU's own NUMA node (best effort;
    # the outcome is reported in e2e.numa -- containers often confine every rank to node 0)
    numa = None
    if world > 1:
        from mojosplat_b200 import hostmem
        numa = hostmem.bind_to_device_node(local_rank)
    sem = _lib.SEM_TORCH if args.semantics == "torch" else _lib.SEM_GSPLAT

    # ---- scene: rank 0 draws it, everyone else receives it over NCCL (one broadcast, at load) ----
    ref_scene = synthetic.make_scene(args.workload, N=1 if rank != 0 else args.n_gaussians)
    N = synthetic.CONFIGS[args.workload][0] if args.n_gaussians is None else args.n_gaussians
    cam0 = ref_scene.camera
    W, H = cam0.W, cam0.H
    if rank == 0:
        host = [t.pin_memory() for t in ref_scene.gaussians()]
        g = [t.to(dev, non_blocking=True) for t in host]
    else:
        shapes = [(N, 3), (N, 3), (N, 4), (N,), (N, 3)]
        g = [torch.empty(s, dtype=torch.float32, device=dev) for s in shapes]
        host = None
    if world > 1:
        for t in g:
            dist.broadcast(t, src=0)
    bg = ref_scene.background.to(dev)
    cams = synthetic.orbit_cameras(N_VIEWS, W, H, cam0.fx)
    for c in cams:
        _lib.camera_struct(c)  # host-side POD cached: no device read-back inside the timed loop
    view_of = lambda k: cams[(k * world + rank) % N_VIEWS]

    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    flush_guard = None
    # Input ring: 3 device copies of the Gaussian set (3 x 56 MB = 168 MB > 126 MB L2), frame k reads copy
    # k % 3, so between two uses of one copy the other two copies (plus ~2 x 230 MB of intermediates) pass
    # through the L2: the timed frames never find their inputs cached.
    RING = 3
    g_ring = [g] + [[t.clone() for t in g] for _ in range(RING - 1)]
    scene_of = lambda k: g_ring[k % RING]

    def frame(k, **kw):
        return ms.render_fused(*g, view_of(k), bg, 16, semantics=sem, **kw)

    from mojosplat_b200.pipeline import FramePipeline, OverlappedPipeline
    if args.pipeline == "overlapped":
        pipe = OverlappedPipeline(dev, N, W, H, semantics=sem, slots=args.slots, bin_streams=args.bin_streams,
                                  raster_mode=args.raster_mode)
    else:
        pipe = FramePipeline(dev, N, W, H, semantics=sem, depth=args.pipeline_depth, raster_mode=args.raster_mode)
    ring = torch.empty((4, H, W, 3), dtype=torch.float32, device=dev)

    # clocks are sampled from the first warm-up frame to the end of the e2e loop (the GPU is under this
    # workload the whole time; the device-timed region alone lasts only tens of milliseconds)
    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- warm-up ----
    Wm = max(args.warmup, 3)
    for k in range(Wm):
        frame(k)
    pipe.render(*g, [view_of(k) for k in range(Wm)], bg, out=ring, scene_of=scene_of)
    torch.cuda.synchronize(dev)

    # ---- timed region: K frames (steps) through the 2-deep frame pipeline, one device-timed region ----
    # L2 rule: "inputs larger than L2" -- the frames rotate over RING copies of the Gaussian arrays
    # (168 MB > 126 MB L2) and every step also streams ~230 MB of intermediates + the image.
    K = args.steps
    views = [view_of(k) for k in range(K)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e_beg, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    e_beg.record()
    pipe.render(*g, views, bg, out=ring, scene_of=scene_of)
    host_enqueue = time.perf_counter() - wall0   # host time to enqueue the K frames (nothing waits for the GPU)
    e_end.record()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - wall0
    if args.pipeline == "overlapped":
        assert pipe.check() == 0, "a timed frame overflowed its pair capacity"
    if world > 1:
        dist.barrier()
    if args.dump_outputs is not None and rank == 0:
        # what the caller of the pipeline received for step K - 1 (frame k lands in ring slot k % 4); images above
        # 64 MB (4K) keep every stride-th row so that the dump stays within that size
        img = ring[(K - 1) % ring.shape[0]]
        stride = -(-img.numel() * img.element_size() // DUMP_BYTES)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "image.npy"), img[::stride].cpu().numpy())
    total_ms = float(e_beg.elapsed_time(e_end))
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * K / (total_ms_max * 1e-3)

    # ---- single-frame latency: frame-by-frame, L2 flushed (512 MiB memset) between frames ----
    Kl = min(K, 20)
    ev_s = [torch.cuda.Event(enable_timing=True) for _ in range(Kl)]
    ev_e = [torch.cuda.Event(enable_timing=True) for _ in range(Kl)]
    for k in range(Kl):
        flush.zero_()
        ev_s[k].record()
        frame(k)
        ev_e[k].record()
    torch.cuda.synchronize(dev)
    latency_ms = float(sum(s.elapsed_time(e) for s, e in zip(ev_s, ev_e))) / Kl

    # ---- the same single frame as ONE CUDA-graph launch (captured sync-free frame, indirect camera) ----
    from mojosplat_b200.pipeline import GraphRenderer
    gr = GraphRenderer(*g, view_of(0), bg, semantics=sem)
    for k in range(3):
        gr.render(view_of(k))
    for k in range(Kl):
        flush.zero_()
        ev_s[k].record()
        gr.render(view_of(k))
        ev_e[k].record()
    torch.cuda.synchronize(dev)
    gr.check()
    graph_latency_ms = float(sum(s.elapsed_time(e) for s, e in zip(ev_s, ev_e))) / Kl
    del gr

    # ---- end-to-end through the public host-buffer API (pinned host in, host image out) ----
    host_all = host if host is not None else [x.cpu().pin_memory() for x in g]
    out_img = torch.empty((H, W, 3), dtype=torch.float32, pin_memory=True)
    bg_host = ref_scene.background
    from mojosplat_b200.pipeline import HostFramePipeline
    hp = HostFramePipeline(dev, N, W, H, semantics=sem)
    Ke = 100  # long enough for the fill and the drain of the three-stage pipeline not to matter
    out_ring = torch.empty((3, H, W, 3), dtype=torch.float32, pin_memory=True)
    hp.render(lambda k: host_all, [view_of(k) for k in range(3)], bg_host, out_ring)  # warm-up
    # un-pipelined single call for reference (copy in -> render -> copy out -> sync)
    ms.render_gaussians_host(*host_all, view_of(0), background_color=bg_host, out=out_img, device=dev)
    t0 = time.perf_counter()
    for k in range(3):
        ms.render_gaussians_host(*host_all, view_of(k), background_color=bg_host, out=out_img, device=dev)
    e2e_single_call_ms = 1e3 * (time.perf_counter() - t0) / 3
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    hp.render(lambda k: host_all, [view_of(k) for k in range(Ke)], bg_host, out_ring)  # ends with a device sync
    e1.record()
    torch.cuda.synchronize(dev)
    te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * Ke / (float(te.item()) * 1e-3)
    # the same with the scene uploaded once (static scene, many poses): per frame camera up, image down
    hp.render(lambda k: host_all, [view_of(k) for k in range(3)], bg_host, out_ring, upload="once")
    torch.cuda.synchronize(dev)
    e0.record()
    hp.render(lambda k: host_all, [view_of(k) for k in range(Ke)], bg_host, out_ring, upload="once")
    e1.record()
    torch.cuda.synchronize(dev)
    te2 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te2, op=dist.ReduceOp.MAX)
    e2e_resident = world * Ke / (float(te2.item()) * 1e-3)
    del hp
    clocks = sampler.stop()
    clocks["window"] = "warm-up + timed + e2e loops"
    h2d = N * (3 + 3 + 4 + 1 + 3) * 4 + 3 * 4
    d2h = H * W * 3 * 4
    del pipe, ring, g_ring, flush_guard
    torch.cuda.empty_cache()

    # ---- BASELINE configs 4 and 5 on the same ranks (SURVEY 8e): every rank takes part ----
    sharded = None
    if not (args.no_sharded or args.no_extras or args.n_gaussians is not None):
        sys.path.insert(0, str(ROOT / "benchmarks"))
        import sharded as sharded_mod
        t0 = time.perf_counter()
        c4 = sharded_mod.run_config4(dev, rank, world, reps=2)
        c5 = sharded_mod.run_config5(dev, rank, world, steps=6)
        sharded = {"config4": c4, "config5": c5, "wall_s": time.perf_counter() - t0,
                   "note": "config 4: 3 M Gaussians x 64 views, split by view (views/s, strong scaling over the ranks); "
                           "config 5: 6 M Gaussians, one 3840x2160 frame split into tile-row bands (frame latency, ms; "
                           "band exchange by NCCL all-gather and fused into the rasterizer as peer stores)"}

    if rank != 0:
        return

    # ---- per-stage device times (view 0, L2 flushed) and the work counters of that frame ----
    stage = np.zeros(4)
    Ks = 10
    info = None
    for k in range(Ks + 2):
        flush.zero_()
        _, tinfo = ms.render_fused(*g, cams[0], bg, 16, semantics=sem, timing=True)
        if k >= 2:
            stage += np.array(tinfo["stage_ms"])
    stage /= Ks
    ms.render_fused(*g, cams[0], bg, 16, semantics=sem, return_aux=True)
    img0, info = ms.render_fused(*g, cams[0], bg, 16, semantics=sem, return_aux=True)  # (second call returns sorted_ids)
    M, P = info["n_isect"], info["sort_passes"]
    launches = K * tinfo["n_launches"]
    # the stand-alone projection kernel (the stage of SURVEY 8a-1: 72 B per Gaussian) and the training-side rasterizer
    from mojosplat_b200.projection import project_gaussians_cuda
    proj_out = project_gaussians_cuda(g[0], g[1], g[2], g[3], cams[0], semantics=sem)
    pa = [torch.cuda.Event(enable_timing=True) for _ in range(Ks)]
    pb = [torch.cuda.Event(enable_timing=True) for _ in range(Ks)]
    for k in range(Ks):
        flush.zero_()
        pa[k].record()
        project_gaussians_cuda(g[0], g[1], g[2], g[3], cams[0], semantics=sem, out=proj_out)
        pb[k].record()
    torch.cuda.synchronize(dev)
    proj_alone_ms = float(sum(a.elapsed_time(b) for a, b in zip(pa, pb))) / Ks
    # the optional fast-math build of the same kernel (not the default: radii can be one off); first call untimed:
    # the kernel's module is loaded lazily
    project_gaussians_cuda(g[0], g[1], g[2], g[3], cams[0], semantics=sem, out=proj_out, fast_math=True)
    for k in range(Ks):
        flush.zero_()
        pa[k].record()
        project_gaussians_cuda(g[0], g[1], g[2], g[3], cams[0], semantics=sem, out=proj_out, fast_math=True)
        pb[k].record()
    torch.cuda.synchronize(dev)
    proj_fast_ms = float(sum(a.elapsed_time(b) for a, b in zip(pa, pb))) / Ks
    backward = None
    if not args.no_extras:
        t = [info["means2d"].clone().requires_grad_(True), info["conics"].clone().requires_grad_(True),
             g[4].clone().requires_grad_(True), g[3].clone().requires_grad_(True)]
        gimg = torch.ones((H, W, 3), dtype=torch.float32, device=dev)
        times = {}
        for mode in ("fast", "faithful"):
            fw, bw = [], []
            for k in range(4):
                for x in t:
                    x.grad = None
                flush.zero_()
                e0, e1, e2 = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e0.record()
                out = rasterization.rasterize_gaussians_diff(*t, bg, info["tile_ranges"], info["sorted_ids"], cams[0],
                                                             16, mode=mode)
                e1.record()
                out.backward(gimg)
                e2.record()
                torch.cuda.synchronize(dev)
                if k >= 1:
                    fw.append(e0.elapsed_time(e1)); bw.append(e1.elapsed_time(e2))
            times[mode] = (float(np.mean(fw)), float(np.mean(bw)))
        backward = {"workload": "rasterization forward (training variant: final T, last index) + backward at the "
                                "timed config (view 0), gradients w.r.t. means2d, conics, colours, opacities",
                    "forward_train_ms": times["fast"][0], "backward_ms": times["fast"][1],
                    "kernels": "pair layout (raster_pair_kernel<train> / raster_bwd_pair_kernel: two pixels per lane, "
                               "packed FP32), the default for 16x16 RGB",
                    "generic_kernels": {"forward_train_ms": times["faithful"][0], "backward_ms": times["faithful"][1],
                                        "note": "raster_train_fwd_kernel / raster_bwd_kernel: any tile size, 1-4 "
                                                "channels, the reference's operation order (mode='faithful')"},
                    "note": "additive (the reference is forward-only, render.py:11); includes the autograd glue"}
        del t, out, gimg
    _, e_all, e_pass = rasterization.rasterize_gaussians_stats(
        info["means2d"], info["conics"], g[4], g[3], bg, info["tile_ranges"], info["sorted_ids"], cams[0], 16)

    # stand-in for "the reference's rasterizer on this GPU" (gsplat / MAX are not installable here): the faithful
    # kernel has the structure and operation order of kernels/rasterization.mojo -- never reported as gsplat
    fa, fb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rasterization.rasterize_gaussians_cuda(info["means2d"], info["conics"], g[4], g[3], bg, info["tile_ranges"],
                                           info["sorted_ids"], cams[0], 16, mode="faithful")
    fa.record()
    rasterization.rasterize_gaussians_cuda(info["means2d"], info["conics"], g[4], g[3], bg, info["tile_ranges"],
                                           info["sorted_ids"], cams[0], 16, mode="faithful")
    fb.record()
    torch.cuda.synchronize(dev)
    faithful_ms = float(fa.elapsed_time(fb))

    # measured FP32 / SFU issue peaks (roofline denominators of the rasterizer)
    def micro(kind):
        out = torch.empty(1, dtype=torch.float32, device=dev)
        blocks, iters = 148 * 8, 8192
        best = 1e9
        for _ in range(4):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            _lib.check(L.bsplat_microbench(kind, blocks, iters, _lib.ptr(out), _lib.stream_ptr(dev)), "microbench")
            b.record()
            torch.cuda.synchronize(dev)
            best = min(best, a.elapsed_time(b))
        return blocks * 256 * 8 * iters / (best * 1e-3)
    ffma_per_s, ex2_per_s = micro(0), micro(1)
    fp32_peak_tflops = 2 * ffma_per_s / 1e12

    hbm_peak, hbm_src = measured_peaks()
    raster_s = stage[3] * 1e-3
    flops = 14 * e_all + 10 * e_pass
    achieved = flops / raster_s / 1e12
    n_tiles = math.ceil(H / 16) * math.ceil(W / 16)
    proj_bytes = 72 * N
    # the fused kernel reads colours + opacity too (56 B) and writes the tile rectangle, the depth key and the 48-byte
    # raster record instead of the four stage outputs (60 B): work the separate record / depth-key passes used to do
    proj_fused_bytes = (56 + 60) * N
    bin_bytes = 52 * N + (28 + 24 * P) * M + 8 * n_tiles
    bin_traffic, bin_traffic_src = ncu_traffic("binning")
    stages = {
        "projection": {"ms": proj_alone_ms, "GB/s": proj_bytes / (proj_alone_ms * 1e-3) / 1e9,
                       "frac_hbm": proj_bytes / (proj_alone_ms * 1e-3) / 1e9 / hbm_peak, "bytes": proj_bytes,
                       "kernel": "project_kernel alone (bsplat_project_fwd: the four stage outputs)"},
        "projection_fast_math": {"ms": proj_fast_ms, "GB/s": proj_bytes / (proj_fast_ms * 1e-3) / 1e9,
                                 "frac_hbm": proj_bytes / (proj_fast_ms * 1e-3) / 1e9 / hbm_peak, "bytes": proj_bytes,
                                 "kernel": "project_kernel, BSPLAT_PROJ_FAST_MATH build (MUFU exp / rcp / sqrt, free "
                                           "contraction): an option, not what the frames above run -- values within "
                                           "1e-4, but a radius next to an integer boundary can be one off"},
        "projection_fused": {"ms": stage[0], "GB/s": proj_fused_bytes / (stage[0] * 1e-3) / 1e9,
                             "frac_hbm": proj_fused_bytes / (stage[0] * 1e-3) / 1e9 / hbm_peak,
                             "bytes": proj_fused_bytes,
                             "kernel": "project_kernel inside a frame: epilogue writes tile rectangles, depth keys + "
                                       "digit histograms and raster records (116 B per Gaussian) instead of the stage "
                                       "outputs"},
        "binning": {"ms": stage[1] + stage[2], "depth_sort_count_scan_ms": stage[1], "emit_tile_sort_ranges_ms": stage[2],
                    "GB/s": bin_bytes / ((stage[1] + stage[2]) * 1e-3) / 1e9,
                    "frac_hbm": bin_bytes / ((stage[1] + stage[2]) * 1e-3) / 1e9 / hbm_peak,
                    "bytes": bin_bytes, "bytes_note": "SURVEY 8d single-level formula 52 N + (28 + 24 P) M + 8 T; the "
                    "two-level path moves far fewer bytes (dram_bytes_ncu) -- it is latency / issue bound, not HBM bound",
                    "dram_bytes_ncu": bin_traffic, "dram_bytes_source": bin_traffic_src,
                    "GB/s_real": (bin_traffic / ((stage[1] + stage[2]) * 1e-3) / 1e9) if bin_traffic else None,
                    "M": M, "sort_passes": P, "key_bits": info["key_bits"]},
        "raster": {"ms": stage[3], "E_all": e_all, "E_pass": e_pass, "nominal_256M": 256 * M,
                   "G_splat_px_per_s": e_all / raster_s / 1e9,
                   "sfu_frac": (e_all / raster_s) / ex2_per_s,
                   "reference_structure_kernel_ms": faithful_ms,
                   "reference_structure_kernel": "raster_faithful_kernel (1 thread/pixel, 256-batch staging, operation "
                                                 "order of kernels/rasterization.mojo; stand-in, NOT gsplat)"},
        "hbm_peak_GB/s": hbm_peak, "hbm_peak_source": hbm_src,
        "ffma_peak_T/s": ffma_per_s / 1e12, "ex2_peak_T/s": ex2_per_s / 1e12,
    }
    traffic, traffic_src = ncu_traffic("raster")
    roofline = {"kernel": RASTER_KERNEL, "bound": "fp32", "achieved": achieved, "peak": fp32_peak_tflops,
                "unit": "TFLOP/s", "frac": achieved / fp32_peak_tflops, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": "measured in this run (FFMA chain micro-benchmark, bsplat_microbench)",
                "work": "14*E_all + 10*E_pass flop per launch (SURVEY.md 8d)", "share_of_step": stage[3] / stage.sum(),
                "ms": stage[3], "includes": "raster_long_compact_kernel (long-list pre-pass) + raster_pair_kernel"}

    # the HBM-bound kernel of the path, for reference next to the (FP32-bound) dominant one
    ptraffic, ptraffic_src = ncu_traffic("projection")
    roofline_hbm = {"kernel": "project_kernel", "bound": "hbm", "achieved": proj_bytes / (proj_alone_ms * 1e-3) / 1e9,
                    "peak": hbm_peak, "unit": "GB/s", "frac": proj_bytes / (proj_alone_ms * 1e-3) / 1e9 / hbm_peak,
                    "traffic": ptraffic, "traffic_source": ptraffic_src, "peak_source": hbm_src,
                    "work": "72 B per Gaussian (SURVEY.md 8d): 40 B read + 32 B written"}

    cpu_baseline, parity = None, None
    sc_np = [x.numpy() for x in ref_scene.gaussians()]
    semv = 0 if args.semantics == "torch" else 1
    if not args.no_extras:
        from oracle import oracle
        oracle.set_num_threads(host_cores())
        ref0 = oracle_frame(sc_np, cams[0], bg_host.numpy(), semv)
        parity = parity_report(img0.cpu().numpy(), info, ref0, sc_np, bg_host.numpy(), cams[0])
    if not args.no_cpu_baseline and world == 1:
        from oracle import oracle
        oracle.set_num_threads(host_cores())
        t0 = time.perf_counter()
        reps = 20  # ~10 s of CPU work on 16 cores (bounded sample of the same workload)
        for k in range(reps):
            oracle_frame(sc_np, cams[k], bg_host.numpy(), semv)
        dt = (time.perf_counter() - t0) / reps
        cpu_baseline = {"value": 1.0 / dt, "unit": "frames/s", "cores": oracle.num_threads(), "kind": "port",
                        "sample": f"{reps} full frames of the same workload (oracle C port, all three stages)"}

    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K,
        "warmup": max(args.warmup, 3), "ms_per_step": total_ms_max / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, ref_scene),
        "method": {"parallelism": f"views split across {world} rank(s); Gaussians NCCL-broadcast once at load; "
                                  + ("sync-free frames (device-side M); projection+binning on a high-priority stream, "
                                     f"rasterizer on a second stream, {args.slots} workspaces / {args.bin_streams} binning streams: binning(k+1) runs inside "
                                     "rasterization(k) (OverlappedPipeline)" if args.pipeline == "overlapped" else
                                     f"{args.pipeline_depth} frames in flight per GPU (begin(k+1) overlaps end(k), FramePipeline)"),
                   "timing": "one CUDA-event pair around the K steps, max over ranks",
                   "l2": "single_frame_ms / graph_frame_ms and the per-stage times use a 512 MiB flush between frames"},
        "latency": {"wall_ms_per_step": 1e3 * wall / K, "host_enqueue_ms_per_step": 1e3 * host_enqueue / K,
                    "single_frame_ms": latency_ms, "graph_frame_ms": graph_latency_ms},
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": Ke, "api": "mojosplat_b200.pipeline.HostFramePipeline.render (pinned host Gaussians in and host image "
                                     "out EVERY frame; H2D(k+1) | render(k) | D2H(k-1) overlapped)",
                "resident_scene_value": e2e_resident,
                "resident_scene_note": "same pipeline with the Gaussians uploaded once per batch (static scene): per frame "
                                       "only the camera goes up and the image (d2h_bytes_per_step) comes down",
                "numa": numa, "host_cores_visible": host_cores(),
                "single_call_ms": e2e_single_call_ms,
                "single_call_api": "mojosplat_b200.render_gaussians_host (copy in -> render -> copy out -> sync)"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_hbm": roofline_hbm,
        "stages": stages, "parity": parity, "backward": backward, "sharded": sharded,
        "cpu_baseline": cpu_baseline,
    }
    _emit(json.dumps(line, default=float))


def main():
    # The contract is ONE JSON line on stdout: NCCL and friends print banners there ("NCCL version ..."), so
    # everything written to fd 1 during the run goes to stderr and the line is written to the real stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    global _emit
    def _emit(text):
        os.write(real_stdout, (text + "\n").encode())
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG=VERSION/INFO makes NCCL print a banner on stdout; the contract is one JSON line there
        # (the version banner is printed at every level but NONE: send NCCL's log to stderr instead)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
