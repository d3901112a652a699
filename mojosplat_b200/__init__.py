"""mojosplat_b200 -- B200-native (sm_100a) backend of the MojoSplat forward path.

Public surface = the reference's (mojosplat/render.py, projection.py, binning.py,
rasterization.py, utils.py) plus additive batched / multi-GPU / host-buffer entry points and the
differentiable ``*_diff`` entry points, the ``ssim`` / ``l1_dssim_loss`` photometric loss and
``DensifyStats`` / ``densify_and_prune`` adaptive density control and the ``mcmc_refine`` / ``mcmc_inject_noise``
3DGS-MCMC densification (training).
Importing the package needs neither a GPU nor the built library; the first call that selects
a CUDA backend loads ``csrc/libbsplat.so`` and fails loudly if it is missing (no CPU fallback).
"""
from .utils import Camera  # noqa: F401
from .projection import project_gaussians, project_gaussians_diff  # noqa: F401
from .binning import bin_gaussians_to_tiles  # noqa: F401
from .rasterization import rasterize_gaussians  # noqa: F401
from .render import TILE_SIZE, render_gaussians, render_gaussians_diff, render_gaussians_host, render_fused  # noqa: F401
from .sh import eval_sh, eval_sh_diff  # noqa: F401
from .loss import l1_dssim_loss, ssim  # noqa: F401
from .densify import DensifyStats, densify_and_prune, scene_extent  # noqa: F401
from .mcmc import mcmc_inject_noise, mcmc_refine  # noqa: F401

__all__ = ["Camera", "project_gaussians", "bin_gaussians_to_tiles", "rasterize_gaussians",
           "render_gaussians", "render_gaussians_host", "render_fused", "eval_sh", "TILE_SIZE",
           "project_gaussians_diff", "eval_sh_diff", "render_gaussians_diff", "ssim", "l1_dssim_loss",
           "DensifyStats", "densify_and_prune", "scene_extent", "mcmc_refine", "mcmc_inject_noise"]
