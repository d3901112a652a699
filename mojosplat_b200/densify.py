"""Adaptive density control: 3DGS's ``densify_and_prune`` on sm_100a kernels (include/bsplat.h: bsplat_densify_*).

``DensifyStats`` accumulates the screen-space statistics after every backward pass (one kernel, no host
synchronisation); ``densify_and_prune`` then clones, splits and prunes the Gaussians in one planning kernel, one
read-back of four counts and one gather kernel that writes every parameter and, with ``optimizer``, every Adam moment
of the new set.  ``scene_extent`` is 3DGS's camera-extent helper.

Out of scope: the opacity reset (two torch lines, see ``densify_and_prune``), AbsGS gradients, MCMC relocation, fused
optimizers and multi-GPU densification.
"""
from __future__ import annotations

import ctypes
import math

import torch

from . import _lib

REQUIRED = ("means3d", "scales", "quats")
MAX_TENSORS = 32
MAX_WIDTH = 256


def _check_cuda_f32(name: str, t) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if t.device.type != "cuda":
        raise RuntimeError(f"{name}: the densification kernels need CUDA tensors; there is no CPU fallback "
                           f"(got device '{t.device}')")
    if t.dtype != torch.float32:
        raise ValueError(f"{name} must be float32, got {t.dtype}")


class DensifyStats:
    """Per-Gaussian screen-space statistics of 3DGS's densification: ``grad2d`` (f32, sum of the NDC-scaled norms of
    d loss / d means2d over the views where the Gaussian was visible), ``count`` (i32, those views) and ``max_radius``
    (i32, the largest screen radius in pixels seen)."""

    def __init__(self, N: int, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError(f"DensifyStats needs a CUDA device; there is no CPU fallback (got '{device}')")
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        self.reset(N)

    @property
    def N(self) -> int:
        return self.grad2d.shape[0]

    def reset(self, N: int) -> None:
        """Zero the three arrays and resize them to N rows."""
        self.grad2d = torch.zeros(N, dtype=torch.float32, device=self.device)
        self.count = torch.zeros(N, dtype=torch.int32, device=self.device)
        self.max_radius = torch.zeros(N, dtype=torch.int32, device=self.device)

    def accumulate(self, means2d_grad: torch.Tensor, radii: torch.Tensor, width: int, height: int) -> None:
        """Add one view: ``means2d_grad`` (N, 2) is d loss / d means2d in pixels (``aux["means2d"].grad`` after
        ``retain_grad()``), ``radii`` (N, 2) int32 the projection's radii; rows with ``max(radii) == 0`` are skipped."""
        _check_cuda_f32("means2d_grad", means2d_grad)
        if means2d_grad.shape != (self.N, 2) or not isinstance(radii, torch.Tensor) or radii.shape != (self.N, 2):
            raise ValueError(f"expected means2d_grad and radii of shape ({self.N}, 2), got "
                             f"{tuple(means2d_grad.shape)} and {tuple(getattr(radii, 'shape', ()))}")
        if radii.dtype != torch.int32 or radii.device != self.device or means2d_grad.device != self.device:
            raise ValueError("radii must be int32 and both tensors on the stats' device")
        if int(width) < 1 or int(height) < 1:
            raise ValueError(f"image size must be positive, got {width} x {height}")
        L = _lib.require_device(self.device)
        g, r = means2d_grad.contiguous(), radii.contiguous()
        with torch.cuda.device(self.device):
            rc = L.bsplat_densify_stats(self.N, _lib.ptr(g), _lib.ptr(r), int(width), int(height),
                                        _lib.ptr(self.grad2d), _lib.ptr(self.count), _lib.ptr(self.max_radius),
                                        _lib.stream_ptr(self.device))
        _lib.check(rc, "bsplat_densify_stats")


def scene_extent(cameras) -> float:
    """3DGS's ``cameras_extent``: 1.1 x the largest distance of a camera centre from the mean of the centres."""
    centres = torch.stack([torch.linalg.inv(c.view_matrix.detach().double().cpu())[:3, 3] for c in cameras])
    return 1.1 * float((centres - centres.mean(dim=0)).norm(dim=1).max())


def _log_f32(x: float) -> float:
    """log(x) in double, rounded once to fp32 (-inf for 0)."""
    return float(torch.tensor(math.log(x) if x > 0 else -math.inf, dtype=torch.float64).float())


def densify_and_prune(params: dict, stats: DensifyStats, scene_extent: float, *, opacities=None,
                      grad_threshold: float = 2e-4, percent_dense: float = 0.01, min_opacity: float = 0.005,
                      max_screen_radius=None, max_world_scale=None, optimizer=None, generator=None):
    """3DGS's ``densify_and_prune`` on the GPU; returns ``(new_params, counts)``.

    ``params`` holds ``"means3d"`` (N, 3), ``"scales"`` (N, 3, log-scales) and ``"quats"`` (N, 4); any other entry is
    an (N, ...) float32 CUDA tensor copied row-wise (opacities, colours, (N, K, 3) SH, ...).  With ``avg = grad2d /
    count`` of ``stats``:

    - ``count > 0`` and ``avg >= grad_threshold``: a Gaussian whose largest log-scale is ``<= log(percent_dense *
      scene_extent)`` is cloned (the row, then an identical copy), any other is split into two children at
      ``mu + R(q / |q|) (exp(s) * n)``, ``n`` from ``torch.randn((n_split, 2, 3), generator=generator)``, with
      log-scales ``s - ln 1.6``;
    - the output rows are then pruned where the opacity the renderer sees (``opacities``, default
      ``params["opacities"]``) is ``< min_opacity``, where ``max_world_scale`` is given and the row's largest log-scale
      is ``> log(max_world_scale)`` (split children with their reduced scales), and where ``max_screen_radius`` is given
      and ``stats.max_radius > max_screen_radius``.  The two rows of a clone or a split share their fate.

    Thresholds are computed in double and rounded once to fp32; every comparison is made in fp32 in log space.  The
    output keeps the input order, each Gaussian replaced in place by its 0, 1 or 2 rows.  The new tensors are fresh
    leaves with ``requires_grad=True``.  Difference from the 3DGS reference: its screen-size prune reads radii it has
    just reset to zero, so there it never fires in the same call; here ``max_screen_radius`` prunes on the statistics
    accumulated since the last reset.

    ``optimizer`` (e.g. ``torch.optim.Adam``): every param of its groups must be one of ``params``' tensors; each of
    their state tensors with N leading rows (``exp_avg``, ``exp_avg_sq``, ``max_exp_avg_sq``) is remapped -- kept rows
    and the original row of a clone keep their moments, clone copies and split children start at zero -- and the
    groups and state are rebound to the new tensors in place.  Scalar state (``step``) is left as it is.  ``stats`` is
    reset to the new size.  ``counts`` = ``dict(n_out, n_clone, n_split, n_pruned)``: ``n_split`` counts split
    decisions (the noise rows), ``n_pruned`` output rows dropped, ``n_out = N + n_clone + n_split - n_pruned``.

    The opacity reset of 3DGS is not part of this call.  With opacities stored as the renderer sees them it is::

        params["opacities"].data.clamp_(max=0.01)
        st = optimizer.state[params["opacities"]]; st["exp_avg"].zero_(); st["exp_avg_sq"].zero_()
    """
    if not isinstance(params, dict):
        raise TypeError("params must be a dict of tensors")
    for k in REQUIRED:
        if k not in params:
            raise ValueError(f"params must hold '{k}'")
    for k, t in params.items():
        _check_cuda_f32(f"params['{k}']", t)
    N, dev = params["means3d"].shape[0], params["means3d"].device
    for k, t in params.items():
        if t.dim() < 1 or t.shape[0] != N or t.device != dev:
            raise ValueError(f"params['{k}'] must have N = {N} leading rows on {dev}, got {tuple(t.shape)} on "
                             f"{t.device}")
    if not isinstance(stats, DensifyStats):
        raise TypeError("stats must be a DensifyStats")
    if stats.N != N or stats.device != dev:
        raise ValueError(f"stats hold {stats.N} rows on {stats.device}; params have {N} on {dev}")
    for k, w in (("means3d", (3,)), ("scales", (3,)), ("quats", (4,))):
        if tuple(params[k].shape[1:]) != w:
            raise ValueError(f"params['{k}'] must be (N, {w[0]}), got {tuple(params[k].shape)}")
    if opacities is None:
        if "opacities" not in params:
            raise ValueError("pass opacities= (the values the renderer sees) or a params['opacities'] entry")
        opacities = params["opacities"]
    _check_cuda_f32("opacities", opacities)
    if opacities.numel() != N or opacities.device != dev:
        raise ValueError(f"opacities must hold N = {N} values on the params' device")

    # every tensor the gather writes: the params, then the optimizer state with N leading rows
    jobs = [(k, None, t) for k, t in params.items()]
    owner = {id(t): k for k, t in params.items()}
    if optimizer is not None:
        for group in optimizer.param_groups:
            for p in group["params"]:
                if id(p) not in owner:
                    raise ValueError("the optimizer holds a parameter that is not in params")
                for sk, sv in optimizer.state.get(p, {}).items():
                    if isinstance(sv, torch.Tensor) and sv.dim() >= 1 and sv.shape[0] == N:
                        _check_cuda_f32(f"optimizer state '{sk}' of params['{owner[id(p)]}']", sv)
                        jobs.append((owner[id(p)], sk, sv))
    if len(jobs) > MAX_TENSORS:
        raise ValueError(f"{len(jobs)} tensors to remap (params + optimizer state); at most {MAX_TENSORS}")
    for k, sk, t in jobs:
        w = math.prod(t.shape[1:])
        if not 1 <= w <= MAX_WIDTH:
            raise ValueError(f"params['{k}']{'' if sk is None else ' state ' + sk}: {w} values per row; "
                             f"the gather takes 1..{MAX_WIDTH}")

    L = _lib.require_device(dev)
    p = _lib.BsplatDensifyParams()
    p.grad_threshold = float(torch.tensor(grad_threshold, dtype=torch.float64).float())
    p.log_clone_max_scale = _log_f32(percent_dense * scene_extent)
    p.min_opacity = float(torch.tensor(min_opacity, dtype=torch.float64).float())
    p.log_max_world_scale = math.inf if max_world_scale is None else _log_f32(max_world_scale)
    p.max_screen_radius = 0x7fffffff if max_screen_radius is None else int(max_screen_radius)
    counts_host = torch.zeros(4, dtype=torch.int64).pin_memory()
    src = {id(t): t.detach().contiguous() for _, _, t in jobs}
    means, scales, quats = src[id(params["means3d"])], src[id(params["scales"])], src[id(params["quats"])]
    opac = opacities.detach().reshape(N).contiguous()
    ws = _lib.workspace.get(dev, "densify", L.bsplat_densify_workspace_bytes(N))
    stream = _lib.stream_ptr(dev)
    with torch.cuda.device(dev):
        rc = L.bsplat_densify_plan(N, _lib.ptr(stats.grad2d), _lib.ptr(stats.count), _lib.ptr(stats.max_radius),
                                   _lib.ptr(scales), _lib.ptr(opac), ctypes.byref(p), _lib.ptr(ws), ws.numel(), None,
                                   ctypes.c_void_p(counts_host.data_ptr()), stream)
        _lib.check(rc, "bsplat_densify_plan")
        torch.cuda.current_stream(dev).synchronize()
        n_out, n_clone, n_split, n_pruned = (int(v) for v in counts_host.tolist())
        noise = torch.randn((n_split, 2, 3), generator=generator, device=dev)
        outs = [torch.empty((n_out, *t.shape[1:]), dtype=torch.float32, device=dev) for _, _, t in jobs]
        if n_out > 0:
            desc = (_lib.BsplatDensifyTensor * len(jobs))()
            for d, (k, sk, t), o in zip(desc, jobs, outs):
                d.src, d.dst, d.width = src[id(t)].data_ptr(), o.data_ptr(), math.prod(t.shape[1:])
                d.role = (_lib.DENSIFY_STATE if sk is not None else _lib.DENSIFY_MEANS if k == "means3d"
                          else _lib.DENSIFY_LOG_SCALES if k == "scales" else _lib.DENSIFY_COPY)
            rc = L.bsplat_densify_apply(N, _lib.ptr(ws), _lib.ptr(means), _lib.ptr(scales), _lib.ptr(quats),
                                        _lib.ptr(noise), len(jobs), desc, stream)
            _lib.check(rc, "bsplat_densify_apply")
    new_params = {}
    new_state = {}
    for (k, sk, t), o in zip(jobs, outs):
        if sk is None:
            new_params[k] = o.requires_grad_(True)
        else:
            new_state.setdefault(k, {})[sk] = o
    if optimizer is not None:
        for group in optimizer.param_groups:
            for i, old in enumerate(group["params"]):
                k = owner[id(old)]
                new = new_params[k]
                group["params"][i] = new
                st = optimizer.state.pop(old, None)
                if st is not None:
                    st = dict(st)
                    st.update(new_state.get(k, {}))
                    optimizer.state[new] = st
    stats.reset(n_out)
    return new_params, dict(n_out=n_out, n_clone=n_clone, n_split=n_split, n_pruned=n_pruned)
