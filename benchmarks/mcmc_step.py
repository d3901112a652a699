"""3DGS-MCMC densification on the GPU (mcmc_inject_noise, mcmc_refine; bsplat_mcmc_*) against the same work in torch.

Workloads: config 3 (1 M Gaussians) and config 5's 6 M scene, each with (N, 16, 3) SH coefficients, opacities and Adam
state (exp_avg, exp_avg_sq) for every parameter: 59 floats of parameters and 118 of moments, 708 B per Gaussian, 15
tensors.  About 5 % of the Gaussians are dead (opacity <= 0.005) and cap_max = 2 N, so every refinement relocates and
adds 5 %.  CUDA events; the L2 is overwritten (512 MiB memset) before every timed call.  Reported per workload:
  - the noise kernel alone (bsplat_mcmc_noise on a pre-drawn noise tensor), its bytes model of 68 B per Gaussian (56 read,
    12 written) and their share of the HBM peak (MEASURED_PEAKS.json if present, else 6.65 TB/s); mcmc_inject_noise
    with its torch.randn draw; the same noise written in torch (gsplat's fp32 element-wise formulation); the largest
    error of both against fp64 over the bound of tests/test_gpu_mcmc.py;
  - mcmc_refine (relocate + add; both index draws on the host) against refine_reference, the torch restatement of
    tests/test_gpu_mcmc.py, on the same inputs and draws, with a check that both give the same outputs.
The card's name and power limit are read in the same run.

    python benchmarks/mcmc_step.py [--reps 20] [--out profiles/r05_mcmc_step.json]
"""
import argparse
import ctypes
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "benchmarks"))
sys.path.insert(0, str(ROOT / "tests"))
import torch

from mojosplat_b200 import _lib, synthetic
from mojosplat_b200.mcmc import _mcmc_params, _noise_draw, mcmc_inject_noise, mcmc_refine
from densify_step import timed_setup
from test_gpu_mcmc import noise_reference, refine_reference, ulps
from train_step import hbm_peak_gbs, power_limit, timed

KEYS = ("means3d", "scales", "quats", "opacities", "sh")
NOISE_BYTES = 68


def make_workload(name, dev):
    sc = synthetic.make_scene(name)
    N = sc.N
    g = torch.Generator().manual_seed(7)
    m, s, q, o, _ = sc.gaussians()
    o = torch.where(torch.rand(N, generator=g) < 0.05, torch.rand(N, generator=g) * 0.004, o.reshape(N))
    sh = torch.randn(N, 16, 3, generator=g) * 0.3
    params = {k: v.to(dev).contiguous() for k, v in zip(KEYS, (m, s, q, o, sh))}
    state = {(k, sk): (torch.randn(params[k].shape, generator=g).abs() * 1e-3).to(dev)
             for k in KEYS for sk in ("exp_avg", "exp_avg_sq")}
    return N, params, state


def with_optimizer(params, state):
    """A fresh Adam over copies of the params and of their state."""
    ps = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    opt = torch.optim.Adam([{"params": [p], "lr": 1e-3} for p in ps.values()])
    for k, p in ps.items():
        opt.state[p] = {"step": torch.tensor(10.0), "exp_avg": state[(k, "exp_avg")].clone(),
                        "exp_avg_sq": state[(k, "exp_avg_sq")].clone()}
    return ps, opt


def torch_noise(params, noise, scale):
    """gsplat's inject_noise_to_position in fp32 torch: covariance from the normalised quaternion and exp(s)."""
    q = params["quats"] / params["quats"].norm(dim=1, keepdim=True).clamp_min(1e-12)
    w, x, y, z = q.unbind(1)
    R = torch.stack([
        torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], 1),
        torch.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], 1),
        torch.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], 1)], 1)
    M = R * torch.exp(params["scales"])[:, None, :]
    cov = M @ M.transpose(1, 2)
    gate = torch.sigmoid(100 * ((1 - params["opacities"]) - 0.995))
    return params["means3d"] + torch.einsum("bij,bj->bi", cov, noise * gate[:, None] * scale)


def mcmc_times(name, reps, flush, dev, hbm):
    L = _lib.load()
    N, params, state = make_workload(name, dev)
    scale = 1e-4 * 5e5
    sp = _lib.stream_ptr(dev)
    prm = _mcmc_params(0.005, False)

    # ---- noise ----
    noise = _noise_draw(N, dev, torch.Generator(device=dev).manual_seed(2))
    means = params["means3d"].clone()

    def kernel():
        _lib.check(L.bsplat_mcmc_noise(N, _lib.ptr(means), _lib.ptr(params["scales"]), _lib.ptr(params["quats"]),
                                       _lib.ptr(params["opacities"]), _lib.ptr(noise), scale, ctypes.byref(prm), sp),
                   "bsplat_mcmc_noise")
    noise_ms = timed(kernel, flush, reps)
    pn = dict(params, means3d=means)
    inject_ms = timed(lambda: mcmc_inject_noise(pn, scale), flush, reps)
    torch_noise_ms = timed(lambda: torch_noise(params, noise, scale), flush, reps)
    # accuracy: one kernel call and the torch formulation against fp64
    means.copy_(params["means3d"])
    kernel()
    ref, mag, _ = noise_reference(params, noise, scale, False)
    bound = 16 * 2.0 ** -24 * mag + 1e-30
    noise_err = float(((means.double() - ref).abs() / bound).max())
    torch_err = float(((torch_noise(params, noise, scale).double() - ref).abs() / bound).max())
    del means, pn, ref, mag, bound

    # ---- refine against the torch restatement ----
    kw = dict(cap_max=2 * N)

    def fused(arg):
        ps, opt = arg
        return mcmc_refine(ps, optimizer=opt, generator=torch.Generator().manual_seed(1), **kw)

    def reference(_):
        return refine_reference(params, state, generator=torch.Generator().manual_seed(1), **kw)

    refine_ms = timed_setup(lambda: with_optimizer(params, state), fused, flush, reps)
    ref_ms = timed_setup(lambda: None, reference, flush, max(3, reps // 4))
    ps, opt = with_optimizer(params, state)
    new, counts = fused((ps, opt))
    ref, ref_state, ref_counts = reference(None)
    max_ulps = max(int(ulps(new[k].detach(), ref[k]).max()) for k in ("opacities", "scales"))
    agree = counts == ref_counts and max_ulps <= 2 and all(
        torch.equal(new[k].detach(), ref[k]) for k in KEYS if k not in ("opacities", "scales")) and all(
        torch.equal(opt.state[new[k]][sk], ref_state[(k, sk)]) for k in KEYS for sk in ("exp_avg", "exp_avg_sq"))
    del new, ref, ref_state, ps, opt
    return dict(workload=name, N=N, counts=counts, tensors=3 * len(KEYS),
                noise_kernel_ms=round(noise_ms, 4), noise_bytes=NOISE_BYTES * N,
                noise_gbs=round(NOISE_BYTES * N / (noise_ms * 1e-3) / 1e9, 1),
                noise_frac_hbm=round(NOISE_BYTES * N / (noise_ms * 1e-3) / (hbm * 1e9), 3),
                noise_least_time_ms=round(NOISE_BYTES * N / (hbm * 1e9) * 1e3, 4),
                mcmc_inject_noise_ms=round(inject_ms, 4), torch_noise_ms=round(torch_noise_ms, 4),
                noise_speedup=round(torch_noise_ms / noise_ms, 2),
                noise_err_over_bound=noise_err, torch_noise_err_over_bound=torch_err,
                mcmc_refine_ms=round(refine_ms, 4), torch_reference_ms=round(ref_ms, 4),
                refine_speedup=round(ref_ms / refine_ms, 2),
                outputs_agree=bool(agree and noise_err <= 1.0), relocated_max_ulps=max_ulps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r05_mcmc_step.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("mcmc_step.py needs a CUDA device")
    dev = torch.device("cuda:0")
    _lib.require_device(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    hbm, hbm_src = hbm_peak_gbs()
    out = dict(gpu=torch.cuda.get_device_name(dev), power_limit=power_limit(),
               l2="512 MiB memset before every timed call", reps=args.reps, hbm_peak_gbs=hbm,
               hbm_peak_source=hbm_src,
               noise_bytes_note="68 B per Gaussian: means, log-scales, quats, opacity, noise read (56), means written (12)",
               err_note="largest |error| vs fp64 over 16 * 2^-24 * magnitude (the test's bound): <= 1 passes")
    out["config3_1m"] = mcmc_times("config3_1m_1080p", args.reps, flush, dev, hbm)
    torch.cuda.empty_cache()
    out["config5_6m"] = mcmc_times("config5_6m_4k", args.reps, flush, dev, hbm)
    line = json.dumps(out)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
