"""3DGS-MCMC densification (Kheradmand et al. 2024; gsplat's ``MCMCStrategy``) on sm_100a kernels
(include/bsplat.h: bsplat_mcmc_*).

The scene keeps a hard budget ``cap_max``.  ``mcmc_refine`` relocates the dead Gaussians onto live ones and grows the
set by 5 % per call until it reaches the cap; ``mcmc_inject_noise`` adds opacity-gated noise to the positions every
step.  gsplat's schedule is three ``if``s in the training loop (defaults: refine every 100 steps from step 500 to step
25 000, noise every step, ``noise_lr`` 5e5, both regularisers 0.01)::

    for step in range(max_steps):
        img = render_gaussians_diff(...)
        loss = l1_dssim_loss(img, target)
        o = params["opacities"]                     # torch.sigmoid(params["opacities"]) with opacity_logits=True
        loss = loss + 0.01 * o.abs().mean() + 0.01 * torch.exp(params["scales"]).abs().mean()
        loss.backward()
        optimizer.step()
        optimizer.zero_grad()
        if 500 < step < 25_000 and step % 100 == 0:
            params, counts = mcmc_refine(params, cap_max=cap_max, optimizer=optimizer, generator=cpu_gen)
        mcmc_inject_noise(params, means_lr * 5e5, generator=cuda_gen)

The draws stay in torch in the ``_*_draws`` helpers and the kernels turn them into rows: ``torch.multinomial`` on
the host from a CPU generator (deterministic, unlike its CUDA version) and ``torch.randn`` on the device.  ``torch.multinomial`` takes at most 2^24 categories, so N is limited to
2^24 Gaussians.  Out of scope: a GPU sampler, noise drawn inside the kernel, a strategy class and multi-GPU MCMC.
"""
from __future__ import annotations

import ctypes
import math

import torch

from . import _lib
from .densify import _check_cuda_f32, _rebind, _row_jobs

REQUIRED = ("means3d", "scales", "quats", "opacities")
MAX_ROWS = 1 << 24  # torch.multinomial's limit on the number of categories


def _f32(x: float) -> float:
    return float(torch.tensor(x, dtype=torch.float64).float())


def _host_opacity(params: dict, opacity_logits: bool) -> torch.Tensor:
    """The opacities the renderer sees, (N,) fp32, copied to the host (a host synchronise, 4 B per Gaussian).  The
    index draws run there because ``torch.multinomial`` on CUDA builds its distribution with a floating-point
    ``cumsum``, which is not deterministic: two runs with one seed would relocate different Gaussians."""
    o = params["opacities"].detach().reshape(-1)
    return (torch.sigmoid(o) if opacity_logits else o).cpu()


def _relocate_draws(params: dict, min_opacity: float, opacity_logits: bool, generator):
    """``(dead, sampled)`` on the params' device: the indices of the dead rows (``o <= min_opacity``, or NaN) in index
    order, and as many indices drawn with replacement in proportion to the opacity of the alive rows (None when no row
    is dead or none is alive).  The opacities are copied to the host and drawn from there (see ``_host_opacity``)."""
    o = _host_opacity(params, opacity_logits)
    dev = params["opacities"].device
    alive = o > _f32(min_opacity)
    dead = torch.nonzero(~alive).flatten()
    if dead.numel() == 0 or dead.numel() == o.numel():
        return dead.to(dev), None
    w = torch.where(alive, o, torch.zeros(()))
    return dead.to(dev), torch.multinomial(w, dead.numel(), replacement=True, generator=generator).to(dev)


def _n_add(N: int, cap_max: int, growth: float) -> int:
    return max(0, min(int(cap_max), int(growth * N)) - N)


def _add_draws(params: dict, n_add: int, opacity_logits: bool, generator):
    """``n_add`` indices, on the params' device, drawn with replacement in proportion to the (updated) opacities, or
    None when ``n_add == 0`` or every weight is 0.  Non-positive (and NaN) opacities weigh 0; after a relocation every
    opacity is positive."""
    if n_add == 0:
        return None
    o = _host_opacity(params, opacity_logits)
    o = torch.where(o > 0, o, torch.zeros(()))
    if not bool((o > 0).any()):
        return None
    return torch.multinomial(o, n_add, replacement=True, generator=generator).to(params["opacities"].device)


def _noise_draw(N: int, device, generator) -> torch.Tensor:
    return torch.randn((N, 3), generator=generator, device=device)


def _check_params(params: dict):
    """(N, device) of a valid ``params``; the row limit is checked before anything touches a device."""
    if not isinstance(params, dict):
        raise TypeError("params must be a dict of tensors")
    for k in REQUIRED:
        if k not in params:
            raise ValueError(f"params must hold '{k}'")
        if not isinstance(params[k], torch.Tensor):
            raise TypeError(f"params['{k}'] must be a torch.Tensor")
    N = params["means3d"].shape[0]
    if N > MAX_ROWS:
        raise ValueError(f"{N} Gaussians: the MCMC draws use torch.multinomial, which takes at most 2^24 = {MAX_ROWS} "
                         "categories")
    for k, t in params.items():
        _check_cuda_f32(f"params['{k}']", t)
    dev = params["means3d"].device
    for k, t in params.items():
        if t.dim() < 1 or t.shape[0] != N or t.device != dev:
            raise ValueError(f"params['{k}'] must have N = {N} leading rows on {dev}, got {tuple(t.shape)} on "
                             f"{t.device}")
        if not t.is_contiguous():
            raise ValueError(f"params['{k}'] must be contiguous (the MCMC kernels write it in place)")
    for k, w in (("means3d", (3,)), ("scales", (3,)), ("quats", (4,))):
        if tuple(params[k].shape[1:]) != w:
            raise ValueError(f"params['{k}'] must be (N, {w[0]}), got {tuple(params[k].shape)}")
    if params["opacities"].numel() != N:
        raise ValueError(f"params['opacities'] must hold N = {N} values, got {tuple(params['opacities'].shape)}")
    return N, dev


def _mcmc_params(min_opacity: float, opacity_logits: bool) -> _lib.BsplatMcmcParams:
    p = _lib.BsplatMcmcParams()
    p.min_opacity = _f32(min_opacity)
    p.opacity_logits = 1 if opacity_logits else 0
    return p


def mcmc_refine(params: dict, *, cap_max: int, min_opacity: float = 0.005, growth: float = 1.05,
                opacity_logits: bool = False, optimizer=None, generator=None):
    """One 3DGS-MCMC refinement: relocate, then add.  Returns ``(params, counts)``.

    ``params`` holds ``"means3d"`` (N, 3), ``"scales"`` (N, 3, log-scales), ``"quats"`` (N, 4) and ``"opacities"``
    (N or N x 1: the value the renderer sees, or its logit with ``opacity_logits=True``); any other entry is an (N, ...)
    contiguous float32 CUDA tensor copied row-wise (colours, (N, K, 3) SH, ...).  ``o`` below is the opacity the renderer
    sees.  A row sampled ``c`` times, ``n = min(c + 1, 51)``, gets ``o' = clamp(1 - (1 - o)^(1/n), min_opacity,
    1 - 2^-23)`` (``o`` taken as at most 1) and log-scales ``s + log(o / D)``, ``D = sum_{k<n} C(n, k+1) (-1)^k
    o'^(k+1) / sqrt(k+1)``, evaluated in double and rounded once (in logit mode ``sigmoid`` and the stored
    ``log(o' / (1 - o'))`` too).

    - Relocate, in place: the dead rows (``o <= min_opacity``; a NaN opacity counts as dead) draw as many rows by
      ``torch.multinomial(o * alive, n_dead, replacement=True, generator=generator)``; every sampled row is updated and
      dead row ``k`` becomes a copy of updated sampled row ``k``.  Nothing happens when no row is alive.
    - Add: ``n_add = max(0, min(cap_max, int(growth * N)) - N)`` rows drawn by multinomial over the updated opacities;
      the sampled rows are updated and rows ``N + k`` are copies of the updated sampled rows.  Nothing is added when
      every weight is 0.

    ``optimizer`` (e.g. ``torch.optim.Adam``): every param of its groups must be one of ``params``' tensors.  Its state
    tensors with N rows are zeroed, in place, at the sampled and the dead rows of the relocation; one difference from
    gsplat, which zeroes only the sampled rows, so a relocated row keeps the stale moments of the Gaussian it replaces.
    The add keeps the existing rows' moments and starts the appended rows at zero (gsplat's rule).  Scalar state
    (``step``) is left as it is.

    When nothing is added the same tensor objects come back, modified in place.  Otherwise they are fresh leaves with
    ``requires_grad=True`` and the optimizer's groups and state are rebound to them in place.  ``counts`` =
    ``dict(n_dead, n_relocated, n_added, n_out)``.  Each of the two draws copies the N opacities to the host and runs
    ``torch.multinomial`` there, with ``generator`` a CPU ``torch.Generator``: on CUDA it builds its distribution with
    a floating-point ``cumsum``, which is not deterministic.  N is at most 2^24 (``torch.multinomial``'s limit).
    """
    if not 1e-30 <= float(min_opacity) < 1.0:  # (sigmoid of its logit stays positive in fp32: some weight is > 0)
        raise ValueError(f"min_opacity must be in [1e-30, 1), got {min_opacity}")
    if int(cap_max) < 0 or not math.isfinite(float(growth)):
        raise ValueError(f"cap_max must be >= 0 and growth finite, got {cap_max}, {growth}")
    if generator is not None and generator.device.type != "cpu":
        raise ValueError("mcmc_refine draws its indices on the host: pass a CPU torch.Generator "
                         f"(got one on '{generator.device}')")
    N, dev = _check_params(params)
    jobs, owner = _row_jobs(params, optimizer, N)
    for k, sk, t in jobs:
        if sk is not None and not t.is_contiguous():
            raise ValueError(f"optimizer state '{sk}' of params['{k}'] must be contiguous")
    n_add = _n_add(N, cap_max, growth)
    counts = dict(n_dead=0, n_relocated=0, n_added=0, n_out=N)
    if N == 0:
        return dict(params), counts
    L = _lib.require_device(dev)
    prm = _mcmc_params(min_opacity, opacity_logits)
    stream = _lib.stream_ptr(dev)
    ws = _lib.workspace.get(dev, "mcmc", L.bsplat_mcmc_workspace_bytes(N))

    def descriptors(outs):
        desc = (_lib.BsplatMcmcTensor * len(jobs))()
        for d, (k, sk, t), o in zip(desc, jobs, outs):
            d.src, d.dst, d.width = t.data_ptr(), o.data_ptr(), math.prod(t.shape[1:])
            d.role = (_lib.MCMC_STATE if sk is not None else _lib.MCMC_OPACITY if k == "opacities"
                      else _lib.MCMC_LOG_SCALES if k == "scales" else _lib.MCMC_COPY)
        return desc

    with torch.no_grad(), torch.cuda.device(dev):
        dead, sampled = _relocate_draws(params, min_opacity, opacity_logits, generator)
        counts["n_dead"] = dead.numel()
        if sampled is not None:
            rc = L.bsplat_mcmc_relocate(N, dead.numel(), _lib.ptr(dead), _lib.ptr(sampled), ctypes.byref(prm),
                                        len(jobs), descriptors([t for _, _, t in jobs]), _lib.ptr(ws), ws.numel(),
                                        None, stream)
            _lib.check(rc, "bsplat_mcmc_relocate")
            counts["n_relocated"] = dead.numel()
        added = _add_draws(params, n_add, opacity_logits, generator)
        if added is None:
            return dict(params), counts
        outs = [torch.empty((N + n_add, *t.shape[1:]), dtype=torch.float32, device=dev) for _, _, t in jobs]
        rc = L.bsplat_mcmc_add(N, n_add, _lib.ptr(added), ctypes.byref(prm), len(jobs), descriptors(outs),
                               _lib.ptr(ws), ws.numel(), None, stream)
        _lib.check(rc, "bsplat_mcmc_add")
    counts["n_added"], counts["n_out"] = n_add, N + n_add
    return _rebind(jobs, outs, owner, optimizer), counts


def mcmc_inject_noise(params: dict, scale: float, *, opacity_logits: bool = False, generator=None) -> None:
    """3DGS-MCMC's position noise, in place on ``params["means3d"]``: ``mu += scale * sigmoid(100 ((1 - o) - 0.995)) *
    R S^2 R^T n`` with ``S = diag(exp(s))``, ``R`` the rotation of the normalised quaternion and ``n`` from
    ``torch.randn((N, 3), generator=generator)``.  ``scale`` is the means' learning rate times ``noise_lr`` (5e5 in
    gsplat), rounded to fp32; the gate is evaluated in double.  Opaque Gaussians barely move; ``scale = 0`` leaves the
    means bit for bit as they were."""
    if not math.isfinite(float(scale)):
        raise ValueError(f"scale must be finite, got {scale}")
    N, dev = _check_params(params)
    if N == 0:
        return
    L = _lib.require_device(dev)
    prm = _mcmc_params(0.005, opacity_logits)
    with torch.no_grad(), torch.cuda.device(dev):
        noise = _noise_draw(N, dev, generator)
        rc = L.bsplat_mcmc_noise(N, _lib.ptr(params["means3d"]), _lib.ptr(params["scales"]), _lib.ptr(params["quats"]),
                                 _lib.ptr(params["opacities"]), _lib.ptr(noise), float(scale), ctypes.byref(prm),
                                 _lib.stream_ptr(dev))
    _lib.check(rc, "bsplat_mcmc_noise")
