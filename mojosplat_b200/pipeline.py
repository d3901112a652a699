"""Software-pipelined multi-view rendering on one GPU (additive; BASELINE.json configs 3-4).

A frame has two halves with opposite characters: ``begin`` (projection, depth sort of the N
Gaussians, count + scan: ~10 small latency-bound kernels that leave most of the chip idle) and
``end`` (emission, tile sort, tile ranges, rasterization: the rasterizer fills every SM).  Between
them sits the frame's only host read-back (M).  ``FramePipeline`` keeps ``depth`` frames in flight on
``depth`` CUDA streams with one workspace each, so that begin(k+1) runs on the GPU while end(k) is
executing and the host wait for M(k+1) is hidden behind end(k).  Results are identical to
frame-by-frame rendering (same kernels, same order inside a frame).
"""
from __future__ import annotations

import ctypes
from ctypes import byref, c_size_t
from typing import Sequence

import torch

from . import _lib
from .binning import read_bin_info
from .rasterization import RASTER_MODES
from .utils import Camera


def _gaussians(t, N: int, C: int) -> list:
    """The five Gaussian arrays (means3d, scales, quats, opacities, features) as contiguous float32, opacities flat."""
    q = [_lib.as_f32(t[0], "means3d"), _lib.as_f32(t[1], "scales"), _lib.as_f32(t[2], "quats"),
         _lib.as_f32(t[3], "opacities").reshape(-1), _lib.as_f32(t[4], "features")]
    assert q[0].shape[0] == N and q[4].shape == (N, C)
    return q


class FramePipeline:
    def __init__(self, device, N: int, W: int, H: int, channels: int = 3, tile_size: int = 16,
                 semantics: int = _lib.SEM_TORCH, depth: int = 2, m_capacity: int | None = None,
                 raster_mode: str = "fast"):
        self.dev = torch.device(device)
        self.L = _lib.require_device(self.dev)
        self.N, self.W, self.H, self.C, self.ts = int(N), int(W), int(H), int(channels), int(tile_size)
        self.semantics, self.flags = semantics, RASTER_MODES[raster_mode]
        self.depth = depth
        self.m_cap = int(m_capacity) if m_capacity else 8 * self.N + 4096
        with torch.cuda.device(self.dev):
            self.streams = [torch.cuda.Stream(self.dev) for _ in range(depth)]
            self.events = [torch.cuda.Event() for _ in range(depth)]
            self.info = [torch.zeros(32, dtype=torch.uint8).pin_memory() for _ in range(depth)]
            self.ws = [self._alloc(self.m_cap) for _ in range(depth)]
        self.last_M = 0

    def _alloc(self, m_cap: int) -> torch.Tensor:
        nbytes = self.L.bsplat_render_workspace_bytes(self.N, m_cap, self.W, self.H, self.ts)
        return torch.empty(nbytes, dtype=torch.uint8, device=self.dev)

    # -- the two halves ---------------------------------------------------------------------
    def _begin(self, slot: int, g, cam_struct) -> None:
        s = self.streams[slot]
        rc = self.L.bsplat_render_begin(self.N, _lib.ptr(g[0]), _lib.ptr(g[1]), _lib.ptr(g[2]), _lib.ptr(g[3]),
                                        byref(cam_struct), self.ts, self.semantics, _lib.ptr(self.ws[slot]),
                                        self.ws[slot].numel(), self.info[slot].data_ptr(), s.cuda_stream)
        _lib.check(rc, "bsplat_render_begin")
        self.events[slot].record(s)

    def _end(self, slot: int, g, cam_struct, background, image) -> int:
        self.events[slot].synchronize()  # host waits for begin(k) only; the other stream keeps the GPU busy
        M = int(read_bin_info(self.info[slot]).n_isect)
        s = self.streams[slot]
        needed = c_size_t(0)
        for attempt in range(2):
            rc = self.L.bsplat_render_end(self.N, M, _lib.ptr(g[4]), _lib.ptr(g[3]), self.C, byref(cam_struct),
                                          _lib.ptr(background), self.ts, self.semantics, self.flags,
                                          _lib.ptr(image), _lib.ptr(self.ws[slot]), self.ws[slot].numel(),
                                          byref(needed), s.cuda_stream)
            if rc == _lib.E_WORKSPACE and attempt == 0:
                # rare: this view produced more intersections than the workspace was sized for.
                # Grow the slot and redo its begin half (the N-part lives in the old buffer).
                s.synchronize()
                self.m_cap = int(M * 1.3) + 4096
                self.ws[slot] = self._alloc(self.m_cap)
                self._begin(slot, g, cam_struct)
                self.events[slot].synchronize()
                continue
            break
        _lib.check(rc, "bsplat_render_end")
        self.last_M = M
        return M

    # -- driver -----------------------------------------------------------------------------
    @torch.no_grad()
    def render(self, means3d, scales, quats, opacities, features, cameras: Sequence[Camera], background,
               out: torch.Tensor | None = None, scene_of=None) -> torch.Tensor:
        """Render all cameras; returns images [n, H, W, C] (valid on the current stream on return).
        If ``out`` has fewer than n slots it is used as a ring (frame k -> out[k % len(out)]).
        ``scene_of`` (optional): callable k -> (means3d, scales, quats, opacities, features) giving frame k
        its own Gaussian set of the same N (dynamic scenes; bench.py rotates copies so that the inputs
        touched between two uses of one copy exceed the L2)."""
        g0 = _gaussians((means3d, scales, quats, opacities, features), self.N, self.C)
        n = len(cameras)
        gs = [g0] * n if scene_of is None else [_gaussians(scene_of(k), self.N, self.C) for k in range(n)]
        bg = _lib.as_f32(background, "background").to(self.dev)
        if out is None:
            out = torch.empty((n, self.H, self.W, self.C), dtype=torch.float32, device=self.dev)
        cams = [_lib.camera_struct(c) for c in cameras]
        cur = torch.cuda.current_stream(self.dev)
        with torch.cuda.device(self.dev):
            for s in self.streams:
                s.wait_stream(cur)  # inputs were produced on the caller's stream
            if n > 0:
                self._begin(0, gs[0], cams[0])
            for k in range(n):
                slot = k % self.depth
                self._end(slot, gs[k], cams[k], bg, out[k % out.shape[0]])
                # enqueue the next frame's first half right behind: it overlaps end(k) on the GPU.
                # With depth 2 the slot of frame k+1 finished end(k-1) long ago in stream order.
                if k + 1 < n:
                    self._begin((k + 1) % self.depth, gs[k + 1], cams[k + 1])
            for s in self.streams:
                cur.wait_stream(s)
        return out


class OverlappedPipeline:
    """Sync-free multi-view rendering with binning/rasterization overlap (bsplat_render_enqueue).

    Two CUDA streams: a HIGH-priority one for projection + binning (about ten latency-bound kernels that
    leave most of the chip idle) and a LOW-priority one for the rasterizer (fills every SM, bound by
    instruction issue).  Nothing on the host waits for the GPU: M stays on the device, the pair buffers are
    sized by a capacity.  The block scheduler serves the high-priority stream first whenever rasterizer
    CTAs retire, so binning(k+1) runs inside rasterization(k) and the frame rate approaches the
    rasterizer's alone.  ``slots`` workspaces are cycled; binning of frame k waits (on the device) for the
    rasterizer of frame k - slots.  After the batch the per-frame bin infos are checked; a frame whose M
    exceeded the capacity is re-rendered synchronously with a larger workspace (rare: capacity adapts).
    Results are identical to frame-by-frame rendering.
    """

    def __init__(self, device, N: int, W: int, H: int, channels: int = 3, tile_size: int = 16,
                 semantics: int = _lib.SEM_TORCH, slots: int = 3, m_capacity: int | None = None,
                 raster_mode: str = "fast", bin_streams: int = 2, packed: bool = False):
        self.dev = torch.device(device)
        self.L = _lib.require_device(self.dev)
        self.N, self.W, self.H, self.C, self.ts = int(N), int(W), int(H), int(channels), int(tile_size)
        self.semantics, self.flags = semantics, RASTER_MODES[raster_mode] | (_lib.FLAG_PACKED if packed else 0)
        self.slots = slots
        self.n_bin = max(1, min(bin_streams, slots))
        self.m_cap = int(m_capacity) if m_capacity else 8 * self.N + 4096
        with torch.cuda.device(self.dev):
            # binning chains of consecutive frames alternate between high-priority streams: two chains in
            # flight keep the rasterizer stream fed (one chain under contention is slower than a rasterization)
            self.s_bins = [torch.cuda.Stream(self.dev, priority=-1) for _ in range(self.n_bin)]
            self.s_bin = self.s_bins[0]
            self.s_ras = torch.cuda.Stream(self.dev, priority=0)
            self.ev_bin = [torch.cuda.Event() for _ in range(slots)]
            self.ev_ras = [torch.cuda.Event() for _ in range(slots)]
            self._alloc_all()
        self.last_M = 0

    def _alloc_all(self):
        nbytes = self.L.bsplat_render_workspace_bytes(self.N, self.m_cap, self.W, self.H, self.ts)
        self.ws = [torch.empty(nbytes, dtype=torch.uint8, device=self.dev) for _ in range(self.slots)]

    def _enqueue(self, slot, g, cam_struct, bg, image, info_host, s_bin=None):
        s_bin = s_bin or self.s_bin
        needed = c_size_t(0)
        rc = self.L.bsplat_render_enqueue(
            self.N, _lib.ptr(g[0]), _lib.ptr(g[1]), _lib.ptr(g[2]), _lib.ptr(g[3]), _lib.ptr(g[4]), self.C,
            ctypes.addressof(cam_struct), _lib.ptr(bg), self.ts, self.semantics, self.flags, _lib.ptr(image),
            _lib.ptr(self.ws[slot]), self.ws[slot].numel(), self.m_cap, byref(needed), info_host.data_ptr(),
            s_bin.cuda_stream, self.s_ras.cuda_stream, self.ev_bin[slot].cuda_event)
        _lib.check(rc, "bsplat_render_enqueue")

    @torch.no_grad()
    def render(self, means3d, scales, quats, opacities, features, cameras: Sequence[Camera], background,
               out: torch.Tensor | None = None, scene_of=None) -> torch.Tensor:
        """Render all cameras; images [n, H, W, C] (or a ring, see FramePipeline.render)."""
        g0 = _gaussians((means3d, scales, quats, opacities, features), self.N, self.C)
        n = len(cameras)
        gs = [g0] * n if scene_of is None else [_gaussians(scene_of(k), self.N, self.C) for k in range(n)]
        bg = _lib.as_f32(background, "background").to(self.dev)
        if out is None:
            out = torch.empty((n, self.H, self.W, self.C), dtype=torch.float32, device=self.dev)
        cams = [_lib.camera_struct(c) for c in cameras]
        infos = torch.zeros((max(n, 1), 32), dtype=torch.uint8).pin_memory()
        cur = torch.cuda.current_stream(self.dev)
        with torch.cuda.device(self.dev):
            for sb in self.s_bins:
                sb.wait_stream(cur)
            self.s_ras.wait_stream(cur)
            for k in range(n):
                slot = k % self.slots
                sb = self.s_bins[k % self.n_bin]
                if k >= self.slots:
                    sb.wait_event(self.ev_ras[slot])  # workspace of frame k - slots is free again
                # (ring output: frame k - len(out) was rasterized earlier on the same in-order stream)
                self.ev_bin[slot].record(sb)  # materialise the handle; re-recorded inside the call
                self._enqueue(slot, gs[k], cams[k], bg, out[k % out.shape[0]], infos[k], sb)
                self.ev_ras[slot].record(self.s_ras)
            cur.wait_stream(self.s_ras)
            for sb in self.s_bins:
                cur.wait_stream(sb)
        self._pending = (infos, gs, cams, bg, out, n)
        return out

    def check(self) -> int:
        """Synchronise and verify the last batch: re-render frames whose M exceeded the capacity.
        Returns the number of frames that had to be redone."""
        infos, gs, cams, bg, out, n = self._pending
        torch.cuda.synchronize(self.dev)
        redone = 0
        max_m = 0
        for k in range(n):
            info = read_bin_info(infos[k])
            max_m = max(max_m, int(info.n_isect))
            if info.reserved[1]:
                redone += 1
        self.last_M = max_m
        if redone:
            self.m_cap = int(max_m * 1.25) + 4096
            self._alloc_all()
            for k in range(n):
                info = read_bin_info(infos[k])
                if info.reserved[1]:
                    with torch.cuda.device(self.dev):
                        self.ev_bin[0].record(self.s_bin)
                        self._enqueue(0, gs[k], cams[k], bg, out[k % out.shape[0]], infos[k])
                    torch.cuda.synchronize(self.dev)
        return redone


class GraphRenderer:
    """One frame captured into a CUDA graph and replayed per view (SURVEY.md 8f rank 2).

    The sync-free frame (bsplat_render_enqueue) is captured once with BSPLAT_FLAG_CAMERA_INDIRECT: the
    graph starts by copying the camera POD from a pinned host struct, so ``render(camera)`` only rewrites
    that struct and launches the graph -- one driver call instead of ~15 kernel/memset launches, no host
    read-back.  Gaussians, background and the output image are fixed device buffers owned by the renderer
    (``update_gaussians`` copies new values in place; N, image size and channel count are fixed).
    The pair capacity is fixed at capture time; ``check()`` reports an overflow of the last frame (the
    caller then rebuilds the renderer with a larger ``m_capacity``).
    """

    def __init__(self, means3d, scales, quats, opacities, features, camera: Camera, background,
                 tile_size: int = 16, semantics: int = _lib.SEM_TORCH, m_capacity: int | None = None,
                 raster_mode: str = "fast"):
        self.dev = means3d.device
        self.L = _lib.require_device(self.dev)
        self.N, self.C = features.shape
        self.g = [t.clone() for t in _gaussians((means3d, scales, quats, opacities, features), self.N, self.C)]
        self.W, self.H, self.ts = int(camera.W), int(camera.H), int(tile_size)
        self.bg = _lib.as_f32(background, "background").to(self.dev).clone()
        self.image = torch.empty((self.H, self.W, self.C), dtype=torch.float32, device=self.dev)
        self.m_cap = int(m_capacity) if m_capacity else 8 * self.N + 4096
        nbytes = self.L.bsplat_render_workspace_bytes(self.N, self.m_cap, self.W, self.H, self.ts)
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=self.dev)
        # pinned host blocks the graph reads / writes at replay time
        self.cam_host = torch.zeros(ctypes.sizeof(_lib.BsplatCamera), dtype=torch.uint8).pin_memory()
        self.info_host = torch.zeros(32, dtype=torch.uint8).pin_memory()
        self._write_camera(camera)
        flags = RASTER_MODES[raster_mode] | _lib.FLAG_CAMERA_INDIRECT
        self.stream = torch.cuda.Stream(self.dev)
        self.graph = torch.cuda.CUDAGraph()

        def enqueue():
            needed = c_size_t(0)
            rc = self.L.bsplat_render_enqueue(
                self.N, _lib.ptr(self.g[0]), _lib.ptr(self.g[1]), _lib.ptr(self.g[2]), _lib.ptr(self.g[3]),
                _lib.ptr(self.g[4]), self.C, self.cam_host.data_ptr(), _lib.ptr(self.bg), self.ts, semantics, flags,
                _lib.ptr(self.image), _lib.ptr(self.ws), self.ws.numel(), self.m_cap, byref(needed),
                self.info_host.data_ptr(), torch.cuda.current_stream(self.dev).cuda_stream, None, None)
            _lib.check(rc, "bsplat_render_enqueue")

        with torch.cuda.device(self.dev):
            self.stream.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(self.stream):
                enqueue()  # warm-up outside the capture (module loading, lazy allocations)
            self.stream.synchronize()
            with torch.cuda.graph(self.graph, stream=self.stream):
                enqueue()

    def _write_camera(self, camera: Camera) -> None:
        if int(camera.W) != self.W or int(camera.H) != self.H:
            raise ValueError("GraphRenderer: the image size is fixed at capture time")
        cs = _lib.camera_struct(camera)
        ctypes.memmove(self.cam_host.data_ptr(), ctypes.addressof(cs), ctypes.sizeof(cs))

    def update_gaussians(self, means3d=None, scales=None, quats=None, opacities=None, features=None) -> None:
        for dst, src in zip(self.g, (means3d, scales, quats, opacities, features)):
            if src is not None:
                dst.copy_(src.reshape(dst.shape))

    @torch.no_grad()
    def render(self, camera: Camera) -> torch.Tensor:
        """Replays the frame for ``camera``; returns the renderer's image buffer (valid on the current
        stream; overwritten by the next call)."""
        # the previous replay must have consumed the pinned camera before it is rewritten
        self.stream.synchronize()
        self._write_camera(camera)
        cur = torch.cuda.current_stream(self.dev)
        self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            self.graph.replay()
        cur.wait_stream(self.stream)
        return self.image

    def check(self) -> int:
        """Synchronise; returns M of the last frame, raises if it exceeded the captured capacity."""
        self.stream.synchronize()
        info = read_bin_info(self.info_host)
        if info.reserved[1]:
            raise RuntimeError(f"GraphRenderer: {int(info.n_isect)} intersections exceed the captured capacity "
                               f"{self.m_cap}; rebuild with a larger m_capacity")
        return int(info.n_isect)


class HostFramePipeline:
    """End-to-end frames from HOST buffers: every frame uploads its Gaussians (pinned host -> device),
    renders (sync-free frame, binning / rasterizer streams as in OverlappedPipeline) and downloads its image
    (device -> pinned host), with the three phases of consecutive frames overlapped on separate streams:
    H2D(k+1) | render(k) | D2H(k-1).  PCIe is full duplex, so the frame period approaches the larger of the
    upload time and the render time instead of their sum.  This is the path bench.py's `e2e` figure times.
    """

    def __init__(self, device, N: int, W: int, H: int, channels: int = 3, tile_size: int = 16,
                 semantics: int = _lib.SEM_TORCH, m_capacity: int | None = None, raster_mode: str = "fast",
                 in_slots: int = 3, out_slots: int = 3):
        self.dev = torch.device(device)
        self.N, self.W, self.H, self.C = int(N), int(W), int(H), int(channels)
        self.in_slots, self.out_slots = in_slots, out_slots
        self.core = OverlappedPipeline(device, N, W, H, channels, tile_size, semantics, slots=out_slots,
                                       m_capacity=m_capacity, raster_mode=raster_mode, bin_streams=2)
        with torch.cuda.device(self.dev):
            self.s_in = torch.cuda.Stream(self.dev)
            self.s_out = torch.cuda.Stream(self.dev)
            shapes = [(N, 3), (N, 3), (N, 4), (N,), (N, channels)]
            self.g_dev = [[torch.empty(sh, dtype=torch.float32, device=self.dev) for sh in shapes]
                          for _ in range(in_slots)]
            self.img_dev = torch.empty((out_slots, H, W, channels), dtype=torch.float32, device=self.dev)
            self.bg_dev = torch.empty((channels,), dtype=torch.float32, device=self.dev)

    @torch.no_grad()
    def render(self, host_scenes, cameras: Sequence[Camera], background_host: torch.Tensor,
               out_host: torch.Tensor, upload: str = "every_frame", timeline: bool = False) -> torch.Tensor:
        """host_scenes: callable k -> 5 contiguous float32 CPU tensors (pinned for full speed);
        out_host: pinned [n or ring, H, W, C].  Returns out_host after a final synchronisation.
        upload="once": the scene of frame 0 is uploaded once and stays resident (a static scene seen from many
        poses); every frame still sends its camera and downloads its image.
        timeline=True: per-frame device times (ms since the first enqueue) of (rasterizer end, download start,
        download end) in ``self.last_timeline``; ``self.last_host_enqueue_s`` is the host time spent enqueueing."""
        import time
        core = self.core
        n = len(cameras)
        cams = [_lib.camera_struct(c) for c in cameras]
        infos = torch.zeros((max(n, 1), 32), dtype=torch.uint8).pin_memory()
        mk = (lambda: torch.cuda.Event(enable_timing=True)) if timeline else torch.cuda.Event
        ev_in = [torch.cuda.Event() for _ in range(n)]
        ev_used = [None] * n                               # frame k no longer reads its input slot
        ev_ras = [mk() for _ in range(n)]
        ev_dl = [mk() for _ in range(n)] if timeline else None
        ev_out = [mk() for _ in range(n)]
        t_host = time.perf_counter()
        with torch.cuda.device(self.dev):
            ev0 = None
            if timeline:
                ev0 = torch.cuda.Event(enable_timing=True)
                ev0.record(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(self.s_in):
                self.bg_dev.copy_(background_host.reshape(-1), non_blocking=True)
            for k in range(n):
                islot, oslot = k % self.in_slots, k % self.out_slots
                if upload == "once":
                    islot = 0
                if upload != "once" or k == 0:
                    src = host_scenes(k)
                    with torch.cuda.stream(self.s_in):
                        if k >= self.in_slots:
                            self.s_in.wait_event(ev_used[k - self.in_slots])
                        for d, h in zip(self.g_dev[islot], src):
                            d.copy_(h.reshape(d.shape), non_blocking=True)
                        ev_in[k].record(self.s_in)
                else:
                    ev_in[k] = ev_in[0]
                sb = core.s_bins[k % core.n_bin]
                sb.wait_event(ev_in[k])
                if k >= self.out_slots:
                    sb.wait_event(ev_ras[k - self.out_slots])    # workspace slot free
                    core.s_ras.wait_event(ev_out[k - self.out_slots])  # image slot downloaded
                core.ev_bin[oslot].record(sb)
                core._enqueue(oslot, self.g_dev[islot], cams[k], self.bg_dev, self.img_dev[oslot], infos[k], sb)
                ev_ras[k].record(core.s_ras)   # rasterizer read colours/opacities: inputs are free after it
                ev_used[k] = ev_ras[k]
                # download on its own stream (plain stream calls: no context-manager overhead per frame)
                self.s_out.wait_event(ev_ras[k])
                if timeline:
                    ev_dl[k].record(self.s_out)
                with torch.cuda.stream(self.s_out):
                    out_host[k % out_host.shape[0]].copy_(self.img_dev[oslot], non_blocking=True)
                ev_out[k].record(self.s_out)
        self.last_host_enqueue_s = time.perf_counter() - t_host
        torch.cuda.synchronize(self.dev)
        self.last_timeline = None
        if timeline:
            self.last_timeline = [(ev0.elapsed_time(ev_ras[k]), ev0.elapsed_time(ev_dl[k]), ev0.elapsed_time(ev_out[k]))
                                  for k in range(n)]
        for k in range(n):
            info = read_bin_info(infos[k])
            if info.reserved[1]:
                raise RuntimeError(f"frame {k}: {int(info.n_isect)} intersections exceed the pair capacity "
                                   f"{core.m_cap}; construct HostFramePipeline with a larger m_capacity")
        return out_host
