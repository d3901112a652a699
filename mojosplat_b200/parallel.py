"""Multi-camera and multi-GPU entry points (additive; the reference is single-camera, single-GPU:
``"C": 1`` at mojosplat/projection.py:431 and rasterization.py:175, ``I = 1`` at binning.py:72).

The forward path shards in exactly two ways (SURVEY.md section 8e):

* **by view** -- every rank holds the whole Gaussian set (one NCCL broadcast at load), ranks render
  disjoint subsets of the cameras, no data-path collective (``render_views``); images are only
  gathered if a consumer asks for them.
* **by tile-row band** -- one very large frame: every rank projects all Gaussians (HBM-bound, cheap),
  bins and rasterizes only its band of tile rows (bands balanced by intersection count), then one
  all-gather of the bands (``render_frame_row_split``).  Per-tile lists are those of the
  single-GPU run, so the assembled image is bit-identical to it.

One process per GPU (torchrun); ``torch.distributed`` is plumbing (NCCL on GPUs, gloo in the CPU
tests of this host logic).
"""
from __future__ import annotations

import math
from typing import Callable, Sequence

import torch
import torch.distributed as dist

from . import _lib
from .binning import bin_gaussians_to_tiles_cuda, read_bin_info
from .projection import project_gaussians_cuda
from .rasterization import rasterize_gaussians_cuda
from .render import TILE_SIZE, render_fused
from .utils import Camera


# ----------------------------------------------------------------------------------------------
# partitioning (pure host logic, tested on CPU with gloo)
# ----------------------------------------------------------------------------------------------
def split_views(n_views: int, rank: int, world: int) -> list:
    """Round-robin view assignment: rank r renders views r, r+world, ... (orbit neighbours have similar
    cost, so round-robin balances better than contiguous blocks)."""
    return list(range(rank, n_views, world))


def balanced_row_bands(row_cost: Sequence[float], world: int) -> list:
    """Split tile rows 0..R-1 into ``world`` contiguous bands with near-equal summed cost.
    Returns [(begin, end)] * world; bands may be empty (when world > R or the cost is concentrated)."""
    import bisect
    R = len(row_cost)
    cum = [0.0]
    for c in row_cost:
        cum.append(cum[-1] + float(c))
    total = cum[-1]
    cuts = [0]
    for r in range(1, world):
        target = total * r / world
        e = bisect.bisect_left(cum, target)          # first e with cost(rows[0:e]) >= target
        if e > 0 and abs(cum[e - 1] - target) <= abs(cum[min(e, R)] - target):
            e -= 1                                     # the cut just before is at least as close
        cuts.append(min(max(e, cuts[-1]), R))
    cuts.append(R)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def tile_row_cost(means2d: torch.Tensor, radii: torch.Tensor, H: int, W: int, tile_size: int) -> torch.Tensor:
    """Approximate number of (gaussian, tile) intersections per tile row -- only used to balance the
    bands, never to decide what is rendered."""
    ts = float(tile_size)
    th, tw = math.ceil(H / tile_size), math.ceil(W / tile_size)
    r = radii.to(torch.float32)
    x0 = ((means2d[:, 0] - r[:, 0]).clamp(0, W - 1) / ts).floor()
    x1 = ((means2d[:, 0] + r[:, 0]).clamp(0, W - 1) / ts).floor()
    y0 = ((means2d[:, 1] - r[:, 1]).clamp(0, H - 1) / ts).floor().long().clamp(0, th - 1)
    y1 = ((means2d[:, 1] + r[:, 1]).clamp(0, H - 1) / ts).floor().long().clamp(0, th - 1)
    width = (x1 - x0 + 1).clamp(min=0)
    # difference array over rows: +width at y0, -width after y1
    diff = torch.zeros(th + 1, dtype=torch.float32, device=means2d.device)
    diff.index_add_(0, y0, width)
    diff.index_add_(0, y1 + 1, -width)
    return diff.cumsum(0)[:th]


def broadcast_gaussians(tensors: Sequence[torch.Tensor], src: int = 0, group=None) -> None:
    """The one exchange of the view-split path: rank ``src``'s Gaussian arrays to everyone
    (56 B per Gaussian for RGB: 168 MB at 3 M).  In place."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    for t in tensors:
        dist.broadcast(t, src=src, group=group)


# ----------------------------------------------------------------------------------------------
# rendering
# ----------------------------------------------------------------------------------------------
def render_gaussians_batched(means3d, scales, quats, opacities, features, cameras: Sequence[Camera],
                             background_color=None, tile_size: int = TILE_SIZE, backend: str = "cuda",
                             out: torch.Tensor | None = None) -> torch.Tensor:
    """All cameras on this GPU: images [C, H, W, 3].  Views are independent.  Batches of equal-size views
    go through the sync-free overlapped pipeline (pipeline.OverlappedPipeline: no host read-back, binning
    of view k+1 inside the rasterization of view k); a frame whose pair count outgrows the workspace is redone
    after the batch.  Results are identical to one render_gaussians call per view."""
    from .projection import CUDA_BACKENDS
    from .render import _background_tensor
    if backend not in CUDA_BACKENDS:
        raise ValueError(f"Invalid backend: {backend}")
    C = features.shape[-1]
    dev = means3d.device
    bg = _background_tensor(background_color, C, dev, torch.float32)
    cam0 = cameras[0]
    if out is None:
        out = torch.empty((len(cameras), cam0.H, cam0.W, C), dtype=torch.float32, device=dev)
    same_size = all(c.H == cam0.H and c.W == cam0.W for c in cameras)
    N = means3d.shape[0]
    if len(cameras) >= 3 and same_size and N > 0 and out.shape[0] == len(cameras):
        from .pipeline import OverlappedPipeline
        key = (dev.index, N, int(cam0.W), int(cam0.H), C, int(tile_size), CUDA_BACKENDS[backend])
        pipe = _pipelines.get(key)
        if pipe is None:
            _pipelines.clear()  # one cached pipeline (three workspaces) at a time
            pipe = _pipelines[key] = OverlappedPipeline(dev, N, cam0.W, cam0.H, C, tile_size, CUDA_BACKENDS[backend])
        pipe.render(means3d, scales, quats, opacities, features, cameras, bg, out=out)
        pipe.check()
        return out
    for k, cam in enumerate(cameras):
        out[k] = render_fused(means3d, scales, quats, opacities, features, cam, bg, tile_size,
                              semantics=CUDA_BACKENDS[backend])
    return out


_pipelines: dict = {}


def render_views(means3d, scales, quats, opacities, features, cameras: Sequence[Camera], background_color=None,
                 tile_size: int = TILE_SIZE, backend: str = "cuda", gather: bool = False, group=None,
                 render_fn: Callable | None = None):
    """View-split multi-GPU render.  Returns ``(view_ids, images)`` of this rank, or -- with
    ``gather=True`` -- all images ``[n_views, H, W, C]`` on every rank (one all_gather)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    mine = split_views(len(cameras), rank, world)
    fn = render_fn or (lambda cams: render_gaussians_batched(means3d, scales, quats, opacities, features, cams,
                                                             background_color, tile_size, backend))
    images = fn([cameras[v] for v in mine]) if mine else None
    if not gather or world == 1:
        return mine, images
    n_max = math.ceil(len(cameras) / world)
    cam0 = cameras[0]
    C = features.shape[-1]
    dev = features.device
    pad = torch.zeros((n_max, cam0.H, cam0.W, C), dtype=torch.float32, device=dev)
    if images is not None:
        pad[: images.shape[0]] = images
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    full = torch.empty((len(cameras), cam0.H, cam0.W, C), dtype=torch.float32, device=dev)
    for r in range(world):
        ids = split_views(len(cameras), r, world)
        if ids:
            full[ids] = parts[r][: len(ids)]
    return list(range(len(cameras))), full


def render_band(means3d, scales, quats, opacities, features, camera: Camera, background, band, tile_size=TILE_SIZE,
                semantics=_lib.SEM_TORCH, out: torch.Tensor | None = None, projected=None):
    """Project everything, bin + rasterize only tile rows [band[0], band[1]).  Returns the full-size image
    buffer with only the band rows written."""
    H, W = camera.H, camera.W
    if projected is None:
        projected = project_gaussians_cuda(means3d, scales, quats, opacities, camera, semantics=semantics)
    means2d, conics, depths, radii = projected
    ids, ranges = bin_gaussians_to_tiles_cuda(means2d, radii, depths, H, W, tile_size, semantics=semantics,
                                              tile_rows=band)
    if out is None:
        out = torch.zeros((H, W, features.shape[-1]), dtype=torch.float32, device=means3d.device)
    rasterize_gaussians_cuda(means2d, conics, features, opacities, background, ranges, ids, camera, tile_size,
                             tile_rows=band, out=out)
    return out


def render_frame_row_split(means3d, scales, quats, opacities, features, camera: Camera, background_color=None,
                           tile_size: int = TILE_SIZE, semantics=_lib.SEM_TORCH, group=None, bands=None):
    """One frame split into tile-row bands across the ranks, then one all-gather of the bands.
    The result equals the single-GPU image bit for bit (per-tile lists are unchanged)."""
    from .render import _background_tensor
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    H, W = camera.H, camera.W
    C = features.shape[-1]
    th = math.ceil(H / tile_size)
    bg = _background_tensor(background_color, C, means3d.device, torch.float32)
    projected = project_gaussians_cuda(means3d, scales, quats, opacities, camera, semantics=semantics)
    if bands is None:
        cost = tile_row_cost(projected[0], projected[3], H, W, tile_size)
        if world > 1:
            dist.broadcast(cost, src=0, group=group)  # identical inputs give identical costs; be explicit
        bands = balanced_row_bands(cost.tolist(), world)
    image = torch.zeros((H, W, C), dtype=torch.float32, device=means3d.device)
    render_band(means3d, scales, quats, opacities, features, camera, bg, bands[rank], tile_size, semantics,
                out=image, projected=projected)
    if world == 1:
        return image
    return assemble_bands(image, bands, tile_size, rank, world, group)


def assemble_bands(image: torch.Tensor, bands, tile_size: int, rank: int, world: int, group=None) -> torch.Tensor:
    """All-gather of the row bands (each rank contributes rows [b0*ts, min(b1*ts, H)) of its buffer)."""
    H = image.shape[0]
    rows = [(min(b0 * tile_size, H), min(b1 * tile_size, H)) for b0, b1 in bands]
    n_max = max(e - s for s, e in rows)
    pad = torch.zeros((n_max,) + tuple(image.shape[1:]), dtype=image.dtype, device=image.device)
    s, e = rows[rank]
    pad[: e - s] = image[s:e]
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    full = torch.empty_like(image)
    for r, (s, e) in enumerate(rows):
        full[s:e] = parts[r][: e - s]
    return full


class RowBandRenderer:
    """One huge frame per step, split into tile-row bands across the ranks (BASELINE.json config 5).

    Per frame and rank: ONE sync-free C call (bsplat_render_enqueue_band: list the Gaussians that can reach the band
    with a conservative pre-test, project those, bin + rasterize the band only, write the band rows) followed by the
    exchange of the bands.  pretest=False projects all N instead (A/B; bit-identical result).  Bands are balanced by
    intersection count; they are computed once (``rebalance``) and reused -- consecutive frames of a
    sequence have near-identical row costs -- instead of per frame.  The assembled image equals the
    single-GPU image bit for bit (per-tile lists do not depend on the split).

    exchange="nccl": bands padded to equal height, one all_gather_into_tensor, rows copied into place.
    exchange="p2p" : the rasterizer itself stores every finished tile into the image buffer of EVERY rank
                     (symmetric memory over NVLink / NVSwitch peer mappings) -- compute and gather are one
                     kernel, followed only by a device-side barrier.
    """

    def __init__(self, N: int, camera: Camera, channels: int = 3, tile_size: int = TILE_SIZE,
                 semantics=_lib.SEM_TORCH, group=None, m_capacity: int | None = None, exchange: str = "nccl",
                 pretest: bool = True):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.L = _lib.require_device(self.dev)
        self.N, self.C, self.ts, self.semantics = int(N), int(channels), int(tile_size), semantics
        self.raster_flags = _lib.RASTER_FAST | (0 if pretest else _lib.FLAG_NO_BAND_PRETEST)
        self.H, self.W = int(camera.H), int(camera.W)
        self.th = math.ceil(self.H / self.ts)
        self.m_cap = int(m_capacity) if m_capacity else 4 * self.N + 4096
        nbytes = self.L.bsplat_render_workspace_bytes(self.N, self.m_cap, self.W, self.H, self.ts)
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=self.dev)
        self.info = torch.zeros(32, dtype=torch.uint8).pin_memory()
        self.exchange = exchange if self.world > 1 else "none"
        self.bands = [(r * self.th // self.world, (r + 1) * self.th // self.world) for r in range(self.world)]
        self._pad = None
        self._hdl, self._peer_arr = None, None
        if self.exchange == "p2p":
            # symmetric memory: every rank maps every rank's image buffer (NVLink / NVSwitch peer access)
            import ctypes
            import torch.distributed._symmetric_memory as symm_mem
            pg = group if group is not None else dist.group.WORLD
            self.image = symm_mem.empty((self.H, self.W, self.C), dtype=torch.float32, device=self.dev)
            self.image.zero_()
            self._hdl = symm_mem.rendezvous(self.image, pg)
            ptrs = [int(p) for r, p in enumerate(self._hdl.buffer_ptrs) if r != self.rank]
            if len(ptrs) > 7:
                raise ValueError("fused band exchange supports up to 8 ranks")
            self._peer_arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
        else:
            self.image = torch.zeros((self.H, self.W, self.C), dtype=torch.float32, device=self.dev)

    def rebalance(self, means3d, scales, quats, opacities, camera: Camera) -> list:
        """Bands with equal intersection counts for this pose (projection + a row histogram; one host sync)."""
        proj = project_gaussians_cuda(means3d, scales, quats, opacities, camera, semantics=self.semantics)
        cost = tile_row_cost(proj[0], proj[3], self.H, self.W, self.ts)
        if self.world > 1:
            dist.broadcast(cost, src=0, group=self.group)
        cost_list = cost.tolist()
        self._row_cost = cost_list
        self.bands = balanced_row_bands(cost_list, self.world)
        self._pad = None
        # size the pair buffers for this rank's band (the cost is the torch-rule intersection count per row)
        b0, b1 = self.bands[self.rank]
        self._resize(int(1.25 * sum(cost_list[b0:b1])) + 65536)
        return self.bands

    def tune_bands(self, means3d, scales, quats, opacities, features, camera: Camera, background,
                   iters: int = 3) -> list:
        """Refine the bands of ``rebalance`` with measured times (once per sequence): the intersection count is a good
        cost model for the inner bands but not for the first and last one, whose corner tiles hold the Gaussians the
        torch rules clamp into them (cheap per pair, plus a pre-pass).  Each round renders one frame, all-gathers the
        ranks' device times of the band call, spreads every band's time over its rows in proportion to their pair
        counts and re-cuts the rows into bands of equal time."""
        if self.world == 1 or not hasattr(self, "_row_cost"):
            return self.bands
        cost = self._row_cost
        for _ in range(iters):
            self._time_band = True
            self.render(means3d, scales, quats, opacities, features, camera, background)
            self._time_band = False
            try:
                self.check()
            except RuntimeError:
                continue  # (capacity grown; measure again)
            t = torch.tensor([self._ev[0].elapsed_time(self._ev[1])], dtype=torch.float32, device=self.dev)
            ts = torch.empty(self.world, dtype=torch.float32, device=self.dev)
            dist.all_gather_into_tensor(ts, t, group=self.group)
            ts = ts.tolist()
            dens = [0.0] * len(cost)
            mean_rate = sum(ts) / max(sum(cost), 1.0)
            for r, (b0, b1) in enumerate(self.bands):
                c = sum(cost[b0:b1])
                rate = ts[r] / c if c > 0 else mean_rate
                for row in range(b0, b1):
                    dens[row] = cost[row] * rate
            self.bands = balanced_row_bands(dens, self.world)
            self._pad = None
            b0, b1 = self.bands[self.rank]
            self._resize(int(1.25 * sum(cost[b0:b1])) + 65536)
        return self.bands

    def _resize(self, m_cap: int) -> None:
        self.m_cap = int(m_cap)
        nbytes = self.L.bsplat_render_workspace_bytes(self.N, self.m_cap, self.W, self.H, self.ts)
        if nbytes > self.ws.numel():
            self.ws = torch.empty(nbytes, dtype=torch.uint8, device=self.dev)

    @torch.no_grad()
    def render(self, means3d, scales, quats, opacities, features, camera: Camera, background) -> torch.Tensor:
        from ctypes import byref, c_size_t
        b0, b1 = self.bands[self.rank]
        cam = _lib.camera_struct(camera)
        stream = torch.cuda.current_stream(self.dev).cuda_stream
        needed = c_size_t(0)
        import ctypes
        timed = getattr(self, "_time_band", False)
        if timed:
            self._ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        if self.exchange == "p2p":
            # nobody may still be reading the previous frame out of a buffer this frame writes into
            self._hdl.barrier(channel=0)
            if timed:
                self._ev[0].record()
            rc = self.L.bsplat_render_enqueue_band_p2p(
                self.N, _lib.ptr(means3d), _lib.ptr(scales), _lib.ptr(quats), _lib.ptr(opacities),
                _lib.ptr(features), self.C, ctypes.addressof(cam), _lib.ptr(background), self.ts, self.semantics,
                self.raster_flags, b0, b1, _lib.ptr(self.image), self._peer_arr, len(self._peer_arr),
                _lib.ptr(self.ws), self.ws.numel(), self.m_cap, byref(needed), self.info.data_ptr(), stream,
                None, None)
            _lib.check(rc, "bsplat_render_enqueue_band_p2p")
            if timed:
                self._ev[1].record()
            self._hdl.barrier(channel=1)  # every rank's tiles have landed everywhere
            return self.image
        if timed:
            self._ev[0].record()
        rc = self.L.bsplat_render_enqueue_band(
            self.N, _lib.ptr(means3d), _lib.ptr(scales), _lib.ptr(quats), _lib.ptr(opacities), _lib.ptr(features),
            self.C, ctypes.addressof(cam), _lib.ptr(background), self.ts, self.semantics, self.raster_flags, b0, b1,
            _lib.ptr(self.image), _lib.ptr(self.ws), self.ws.numel(), self.m_cap, byref(needed),
            self.info.data_ptr(), stream, None, None)
        _lib.check(rc, "bsplat_render_enqueue_band")
        if timed:
            self._ev[1].record()
        if self.exchange == "nccl":
            rows = [(min(a * self.ts, self.H), min(b * self.ts, self.H)) for a, b in self.bands]
            n_max = max(e - s for s, e in rows)
            if self._pad is None or self._pad.shape[1] != n_max:
                self._pad = torch.empty((self.world, n_max, self.W, self.C), dtype=torch.float32, device=self.dev)
            s, e = rows[self.rank]
            mine = self._pad[self.rank]
            mine[: e - s].copy_(self.image[s:e])
            dist.all_gather_into_tensor(self._pad.view(-1), mine.reshape(-1), group=self.group)
            for r, (s, e) in enumerate(rows):
                if r != self.rank:
                    self.image[s:e].copy_(self._pad[r, : e - s])
        return self.image

    def check(self) -> int:
        torch.cuda.synchronize(self.dev)
        info = read_bin_info(self.info)
        if info.reserved[1]:
            need = int(info.n_isect)
            self._resize(int(1.25 * need) + 65536)  # the next render() fits; this frame must be redone
            raise RuntimeError(f"band produced {need} intersections > capacity; workspace grown, render again")
        return int(info.n_isect)
