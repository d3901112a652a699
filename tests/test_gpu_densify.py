"""Adaptive density control (DensifyStats, densify_and_prune; bsplat_densify_*) against a pure-torch restatement.

``densify_reference`` restates the semantics of ``densify_and_prune`` in torch with the same generator draw: decisions,
row order, copies, reduced log-scales and optimizer-state remap must match bit for bit; split-child means are compared
with an fp64 evaluation.  The argument checks and the struct sizes at the top need no GPU.
"""
import ctypes
import math

import pytest
import torch

import mojosplat_b200 as ms
from mojosplat_b200 import _lib
from mojosplat_b200.densify import DensifyStats, densify_and_prune


def f32(x):
    """x computed in double, rounded once to fp32 (how the thresholds reach the kernels)."""
    return float(torch.tensor(x, dtype=torch.float64).float())


def quat_rotmat64(q):
    q = q.double()
    q = q / q.norm(dim=1, keepdim=True).clamp_min(1e-12)
    w, x, y, z = q.unbind(1)
    return torch.stack([
        torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], 1),
        torch.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], 1),
        torch.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], 1)], 1)


def densify_reference(params, grad2d, count, max_radius, scene_extent, opacities, *, grad_threshold=2e-4,
                      percent_dense=0.01, min_opacity=0.005, max_screen_radius=None, max_world_scale=None,
                      state=None, generator=None):
    """Torch restatement of densify_and_prune.  ``state``: {(key, name): (N, ...) tensor}.  Returns (new params,
    new state, counts, extra) with extra = dict(child (n_out,) bool mask of split children, means64 (fp64 child means),
    tol_scale (|mu| + |exp(s) * n| per child row), new_row (n_out,) bool mask of the rows that start with zero
    moments)."""
    N, dev = grad2d.shape[0], grad2d.device
    s = params["scales"]
    smax = s.max(dim=1).values if N else torch.zeros(0, device=dev)
    high = (count > 0) & (grad2d / count.float() >= f32(grad_threshold))
    small = smax <= f32(math.log(percent_dense * scene_extent))
    clone, split = high & small, high & ~small
    ln16 = f32(math.log(1.6))
    prune = opacities.reshape(N) < f32(min_opacity)
    if max_world_scale is not None:
        prune |= torch.where(split, smax - ln16, smax) > f32(math.log(max_world_scale))
    if max_screen_radius is not None:
        prune |= max_radius > int(max_screen_radius)
    n_split = int(split.sum())
    noise = torch.randn((n_split, 2, 3), generator=generator, device=dev)
    rows = torch.where(high, 2, 1)
    kept = torch.where(prune, 0, rows)
    parent = torch.repeat_interleave(torch.arange(N, device=dev), kept)
    j = torch.arange(parent.shape[0], device=dev) - (torch.cumsum(kept, 0) - kept)[parent]
    rank = (torch.cumsum(split.long(), 0) - split.long())[parent]
    child = split[parent]
    new_row = (clone[parent] & (j == 1)) | child
    out = {k: t[parent].clone() for k, t in params.items()}
    out["scales"][child] = params["scales"][parent[child]] - ln16
    pc = parent[child]
    mu = params["means3d"][pc].double()
    e = params["scales"][pc].double().exp() * noise[rank[child], j[child]].double()
    means64 = mu + (quat_rotmat64(params["quats"][pc]) @ e[..., None])[..., 0]
    out["means3d"][child] = means64.float()
    new_state = {}
    for key, t in (state or {}).items():
        o = t[parent].clone()
        o[new_row] = 0
        new_state[key] = o
    counts = dict(n_out=int(parent.shape[0]), n_clone=int(clone.sum()), n_split=n_split,
                  n_pruned=int((rows * prune).sum()))
    return out, new_state, counts, dict(child=child, new_row=new_row, means64=means64,
                                        tol_scale=mu.abs() + e.norm(dim=1, keepdim=True))


def make_case(N, seed, dev, prune_max=False):
    """Parameters of widths 3, 3, 4, 1, 3, 4 and 48 plus statistics seeded for a mix of keep / clone / split / prune."""
    g = torch.Generator().manual_seed(seed)
    params = dict(
        means3d=torch.randn(N, 3, generator=g) * 2.0,
        scales=torch.rand(N, 3, generator=g) * 5.0 - 5.5,
        quats=torch.randn(N, 4, generator=g) * (0.3 + torch.rand(N, 1, generator=g)),  # unnormalised
        opacities=torch.rand(N, generator=g),
        colors=torch.rand(N, 3, generator=g),
        extra4=torch.randn(N, 4, generator=g),
        sh=torch.randn(N, 16, 3, generator=g))
    count = torch.randint(0, 5, (N,), generator=g, dtype=torch.int32)
    grad2d = torch.rand(N, generator=g) * 4.5e-4 * count
    max_radius = torch.randint(0, 80, (N,), generator=g, dtype=torch.int32)
    params = {k: v.to(dev) for k, v in params.items()}
    kw = dict(grad_threshold=2e-4, percent_dense=0.01, min_opacity=0.05)
    if prune_max:
        kw.update(max_screen_radius=70, max_world_scale=math.exp(-1.0))
    return params, grad2d.to(dev), count.to(dev), max_radius.to(dev), kw


def stats_from(N, dev, grad2d, count, max_radius):
    st = DensifyStats(N, dev)
    st.grad2d.copy_(grad2d)
    st.count.copy_(count)
    st.max_radius.copy_(max_radius)
    return st


def adam_state(params, seed):
    """An Adam optimizer over params (one group each) after one step on seeded gradients."""
    opt = torch.optim.Adam([{"params": [p], "lr": 1e-3} for p in params.values()])
    g = torch.Generator(device=next(iter(params.values())).device).manual_seed(seed)
    for p in params.values():
        p.grad = torch.randn(p.shape, generator=g, device=p.device)
    opt.step()
    return opt


def assert_matches_reference(new, counts, ref, ref_counts, extra, state_new=None, state_ref=None):
    assert counts == ref_counts, (counts, ref_counts)
    for k, t in ref.items():
        got = new[k].detach()
        assert got.shape == t.shape, (k, got.shape, t.shape)
        if k == "means3d":
            child = extra["child"]
            assert torch.equal(got[~child], t[~child]), k
            err = (got[child].double() - extra["means64"]).abs()
            assert bool((err <= 2e-6 * extra["tol_scale"]).all()), float((err / extra["tol_scale"]).max())
        else:
            assert torch.equal(got, t), k
    for key, t in (state_ref or {}).items():
        assert torch.equal(state_new[key], t), key


# ---------------------------------------------------------------- arguments and ABI (no GPU) -------------------------

@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        _lib.build()
    return _lib.load()


def test_struct_sizes():
    assert ctypes.sizeof(_lib.BsplatDensifyParams) == 24
    assert ctypes.sizeof(_lib.BsplatDensifyTensor) == 24
    assert ctypes.sizeof(_lib.BsplatDensifyCounts) == 32


def test_arguments_rejected_without_gpu():
    z = torch.zeros
    p = dict(means3d=z(4, 3), scales=z(4, 3), quats=z(4, 4), opacities=z(4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        densify_and_prune(p, None, 1.0)
    with pytest.raises(ValueError, match="must hold 'quats'"):
        densify_and_prune(dict(means3d=z(4, 3), scales=z(4, 3)), None, 1.0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        DensifyStats(4, "cpu")


def test_c_abi_rejections_without_gpu(lib):
    """Argument rules of the C entry points: every one of these returns before anything reaches a device."""
    fake = [ctypes.c_void_p(0x1000 * (i + 1)) for i in range(8)]

    def desc(rows):
        d = (_lib.BsplatDensifyTensor * max(len(rows), 1))()
        for x, (src, dst, w, role) in zip(d, rows):
            x.src, x.dst, x.width, x.role = src, dst, w, role
        return d

    M, S = _lib.DENSIFY_MEANS, _lib.DENSIFY_LOG_SCALES
    base = [(0x1000, 0x9000, 3, M), (0x2000, 0xa000, 3, S)]

    def apply(rows, n=None, means=0x1000, scales=0x2000):
        return lib.bsplat_densify_apply(10, fake[0], ctypes.c_void_p(means), ctypes.c_void_p(scales), fake[2], None,
                                        len(rows) if n is None else n, desc(rows), None)

    assert apply(base, n=0) == _lib.E_ARG
    assert apply(base + [(0x3000, 0xb000, 1, 0)] * 31) == _lib.E_ARG                 # 33 tensors
    assert apply(base + [(0x3000, 0xb000, 0, 0)]) == _lib.E_ARG                      # width 0
    assert apply(base + [(0x3000, 0xb000, 257, 0)]) == _lib.E_ARG                    # width 257
    assert apply(base + [(0x3000, 0x3000, 4, 0)]) == _lib.E_ARG                      # dst == src
    assert apply(base + [(0x3000, 0, 4, 0)]) == _lib.E_ARG                           # null dst
    assert apply(base + [(0x3000, 0xb000, 4, 7)]) == _lib.E_ARG                      # unknown role
    assert apply(base[:1]) == _lib.E_ARG                                             # no LOG_SCALES
    assert apply(base[1:]) == _lib.E_ARG                                             # no MEANS
    assert apply(base, means=0x5000) == _lib.E_ARG                                   # MEANS src != means3d
    assert apply(base + [(0x3000, 0xb000, 3, M)]) == _lib.E_ARG                      # two MEANS
    assert lib.bsplat_densify_apply(0, None, ctypes.c_void_p(0x1000), ctypes.c_void_p(0x2000), None, None, 2,
                                    desc(base), None) == _lib.OK                     # N = 0: nothing launched
    # plan: workspace too small -> E_WORKSPACE with the size; N = 0 -> zero counts, nothing launched
    prm = _lib.BsplatDensifyParams()
    counts = _lib.BsplatDensifyCounts(7, 7, 7, 7)
    need = ctypes.c_size_t(0)
    rc = lib.bsplat_densify_plan(5000, *fake[:5], ctypes.byref(prm), fake[5], 16, ctypes.byref(need),
                                 ctypes.addressof(counts), None)
    assert rc == _lib.E_WORKSPACE and need.value == lib.bsplat_densify_workspace_bytes(5000) > 5000
    assert lib.bsplat_densify_plan(5000, *fake[:5], None, fake[5], 1 << 20, None, ctypes.addressof(counts),
                                   None) == _lib.E_ARG
    assert lib.bsplat_densify_plan(0, None, None, None, None, None, ctypes.byref(prm), None, 0, None,
                                   ctypes.addressof(counts), None) == _lib.OK
    assert (counts.n_out, counts.n_clone, counts.n_split, counts.n_pruned) == (0, 0, 0, 0)
    assert lib.bsplat_densify_stats(-1, *fake[:2], 8, 8, *fake[2:5], None) == _lib.E_ARG
    assert lib.bsplat_densify_stats(10, *fake[:2], 0, 8, *fake[2:5], None) == _lib.E_ARG
    assert lib.bsplat_densify_stats(10, ctypes.c_void_p(0x1004), fake[1], 8, 8, *fake[2:5], None) == _lib.E_ARG
    assert lib.bsplat_densify_stats(0, None, None, 8, 8, None, None, None, None) == _lib.OK


@pytest.mark.gpu
def test_arguments_rejected_on_gpu(cuda_device):
    params, grad2d, count, max_radius, _ = make_case(16, 0, cuda_device)
    st = stats_from(16, cuda_device, grad2d, count, max_radius)
    with pytest.raises(ValueError, match="leading rows"):
        densify_and_prune(dict(params, colors=params["colors"][:15]), st, 1.0)
    with pytest.raises(ValueError, match="float32"):
        densify_and_prune(dict(params, colors=params["colors"].double()), st, 1.0)
    with pytest.raises(ValueError, match="stats hold"):
        densify_and_prune(params, DensifyStats(15, cuda_device), 1.0)
    with pytest.raises(ValueError, match="at most 32"):
        densify_and_prune(dict(params, **{f"x{i}": torch.zeros(16, device=cuda_device) for i in range(26)}), st, 1.0)
    with pytest.raises(ValueError, match="1..256"):
        densify_and_prune(dict(params, big=torch.zeros(16, 257, device=cuda_device)), st, 1.0)
    with pytest.raises(ValueError, match="opacities"):
        densify_and_prune({k: v for k, v in params.items() if k != "opacities"}, st, 1.0)
    stray = torch.zeros(16, 3, device=cuda_device, requires_grad=True)
    opt = torch.optim.Adam([params["means3d"].requires_grad_(True), stray])
    with pytest.raises(ValueError, match="not in params"):
        densify_and_prune(params, st, 1.0, optimizer=opt)
    with pytest.raises(ValueError, match="shape"):
        st.accumulate(torch.zeros(15, 2, device=cuda_device), torch.zeros(15, 2, dtype=torch.int32,
                                                                           device=cuda_device), 8, 8)


# ---------------------------------------------------------------- statistics -----------------------------------------

def torch_stats_step(ref, g, radii, W, H):
    vis = radii.max(dim=1).values > 0
    n = torch.sqrt((g[:, 0] * (W / 2)) ** 2 + (g[:, 1] * (H / 2)) ** 2)
    ref["grad2d"] = torch.where(vis, ref["grad2d"] + n, ref["grad2d"])
    ref["count"] = ref["count"] + vis.int()
    ref["max_radius"] = torch.where(vis, torch.maximum(ref["max_radius"], radii.max(dim=1).values), ref["max_radius"])


def assert_stats_equal(st, ref):
    assert torch.equal(st.count, ref["count"]) and torch.equal(st.max_radius, ref["max_radius"])
    ulp = (st.grad2d.view(torch.int32).long() - ref["grad2d"].view(torch.int32).long()).abs()
    assert int(ulp.max()) <= 1, int(ulp.max())


@pytest.mark.gpu
def test_stats_match_torch(cuda_device):
    N = 100_003
    g = torch.Generator().manual_seed(3)
    st = DensifyStats(N, cuda_device)
    ref = dict(grad2d=torch.zeros(N, device=cuda_device), count=torch.zeros(N, dtype=torch.int32, device=cuda_device),
               max_radius=torch.zeros(N, dtype=torch.int32, device=cuda_device))
    for step in range(6):
        W, H = (1920, 1080) if step % 2 else (128, 96)
        v = (torch.randn(N, 2, generator=g) * 10.0 ** float(torch.randint(-7, -2, (1,), generator=g))).to(cuda_device)
        radii = torch.randint(0, 40, (N, 2), generator=g, dtype=torch.int32)
        radii[torch.rand(N, generator=g) < 0.3] = 0
        one = torch.rand(N, generator=g) < 0.1
        radii[one, 0] = 0  # one component zero: still visible when the other is positive
        radii = radii.to(cuda_device)
        st.accumulate(v, radii, W, H)
        torch_stats_step(ref, v, radii, W, H)
    assert_stats_equal(st, ref)
    assert 0 < int((st.count == 0).sum()) < N


@pytest.mark.gpu
def test_stats_through_render(cuda_device):
    """render_gaussians_diff -> l1_dssim_loss -> backward with retain_grad() on aux["means2d"]."""
    from test_gpu_train import e2e_scene
    cam, m, s, q, o, c, _ = e2e_scene(400, 96, 5, 3)
    target = torch.rand(96, 96, 3, generator=torch.Generator().manual_seed(1)).to(cuda_device)
    p = [x.to(cuda_device).requires_grad_(True) for x in (m, s, q, o, c)]
    st = DensifyStats(400, cuda_device)
    ref = dict(grad2d=torch.zeros(400, device=cuda_device), count=torch.zeros(400, dtype=torch.int32,
                                                                            device=cuda_device),
               max_radius=torch.zeros(400, dtype=torch.int32, device=cuda_device))
    for _ in range(3):
        img, aux = ms.render_gaussians_diff(*p, cam, return_aux=True)
        aux["means2d"].retain_grad()
        ms.l1_dssim_loss(img, target).backward()
        st.accumulate(aux["means2d"].grad, aux["radii"], cam.W, cam.H)
        torch_stats_step(ref, aux["means2d"].grad, aux["radii"], cam.W, cam.H)
    assert_stats_equal(st, ref)
    assert int((st.count == 3).sum()) > 100 and float(st.grad2d.max()) > 0


# ---------------------------------------------------------------- densify vs the restatement ------------------------

def run_both(params, grad2d, count, max_radius, kw, dev, seed, extent=5.0, with_state=True):
    N = grad2d.shape[0]
    opt = adam_state(params, seed) if with_state else None
    state = {}
    if opt is not None:
        names = {id(t): k for k, t in params.items()}
        for p, stt in opt.state.items():
            for sk, sv in stt.items():
                if sv.dim() >= 1:
                    state[(names[id(p)], sk)] = sv.clone()
    det = {k: v.detach() for k, v in params.items()}
    ref, ref_state, ref_counts, extra = densify_reference(
        det, grad2d, count, max_radius, extent, det["opacities"], state=state,
        generator=torch.Generator(device=dev).manual_seed(seed), **kw)
    st = stats_from(N, dev, grad2d, count, max_radius)
    new, counts = densify_and_prune(params, st, extent, optimizer=opt,
                                    generator=torch.Generator(device=dev).manual_seed(seed), **kw)
    new_state = {}
    if opt is not None:
        names = {id(t): k for k, t in new.items()}
        for p, stt in opt.state.items():
            for sk, sv in stt.items():
                if sv.dim() >= 1:
                    new_state[(names[id(p)], sk)] = sv
        assert set(new_state) == set(ref_state)
    assert_matches_reference(new, counts, ref, ref_counts, extra, new_state, ref_state)
    assert st.N == counts["n_out"] and int(st.count.abs().sum()) == 0
    return new, counts


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 7, 1023, 1024, 1025, 100_003, 1_000_000])
@pytest.mark.parametrize("prune_max", [False, True])
def test_densify_matches_reference(cuda_device, N, prune_max):
    params, grad2d, count, max_radius, kw = make_case(N, N % 97 + prune_max, cuda_device, prune_max)
    new, counts = run_both(params, grad2d, count, max_radius, kw, cuda_device, seed=N + 11)
    print(N, prune_max, counts)
    if N >= 1023:
        assert counts["n_clone"] > 0 and counts["n_split"] > 0 and counts["n_pruned"] > 0
        assert N - counts["n_pruned"] < counts["n_out"]
    for k, t in new.items():
        assert t.is_leaf and t.requires_grad and t.shape[1:] == params[k].shape[1:]


# ---------------------------------------------------------------- edge cases -----------------------------------------

@pytest.mark.gpu
def test_nothing_to_do(cuda_device):
    N = 5000
    params, grad2d, count, max_radius, kw = make_case(N, 1, cuda_device)
    opt = adam_state(params, 2)
    old = {k: v.detach().clone() for k, v in params.items()}
    old_state = {k: {sk: sv.clone() for sk, sv in opt.state[params[k]].items()} for k in params}
    st = stats_from(N, cuda_device, grad2d * 0, count, max_radius)
    # (the Adam step moved some opacities below 0: -inf switches the opacity prune off)
    new, counts = densify_and_prune(params, st, 5.0, min_opacity=-math.inf, optimizer=opt)
    assert counts == dict(n_out=N, n_clone=0, n_split=0, n_pruned=0)
    for k in params:
        assert torch.equal(new[k].detach(), old[k]), k
        for sk, sv in old_state[k].items():
            assert torch.equal(opt.state[new[k]][sk], sv), (k, sk)


@pytest.mark.gpu
def test_everything_pruned(cuda_device):
    N = 3000
    params, grad2d, count, max_radius, kw = make_case(N, 4, cuda_device)
    opt = adam_state(params, 5)
    st = stats_from(N, cuda_device, grad2d, count, max_radius)
    new, counts = densify_and_prune(params, st, 5.0, min_opacity=2.0, optimizer=opt)
    assert counts["n_out"] == 0 and counts["n_pruned"] == N + counts["n_clone"] + counts["n_split"]
    for k, t in new.items():
        assert t.shape == (0, *params[k].shape[1:]), k
    for t in new.values():
        t.grad = torch.zeros_like(t)
    opt.step()
    assert st.N == 0


@pytest.mark.gpu
def test_everything_split(cuda_device):
    N = 2049
    params, grad2d, count, max_radius, kw = make_case(N, 6, cuda_device)
    params["scales"] = params["scales"].abs() + 0.1  # all large
    params["opacities"] = params["opacities"] * 0.5 + 0.5
    count = torch.full_like(count, 2)
    grad2d = torch.full_like(grad2d, 1.0)
    new, counts = run_both(params, grad2d, count, max_radius, kw, cuda_device, seed=8)
    assert counts == dict(n_out=2 * N, n_clone=0, n_split=N, n_pruned=0)


@pytest.mark.gpu
def test_zero_count_never_grows(cuda_device):
    N = 1500
    params, grad2d, count, max_radius, kw = make_case(N, 9, cuda_device)
    new, counts = run_both(params, torch.full_like(grad2d, 1e3), torch.zeros_like(count), max_radius,
                           dict(kw, min_opacity=-math.inf), cuda_device, seed=10)
    assert counts == dict(n_out=N, n_clone=0, n_split=0, n_pruned=0)


@pytest.mark.gpu
def test_empty_set(cuda_device):
    params, grad2d, count, max_radius, kw = make_case(0, 0, cuda_device)
    new, counts = run_both(params, grad2d, count, max_radius, kw, cuda_device, seed=1, with_state=False)
    assert counts == dict(n_out=0, n_clone=0, n_split=0, n_pruned=0)
    assert new["sh"].shape == (0, 16, 3)


# ---------------------------------------------------------------- optimizer remap ------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("amsgrad", [False, True])
def test_optimizer_remap(cuda_device, amsgrad):
    N = 20_000
    params, grad2d, count, max_radius, kw = make_case(N, 12, cuda_device, prune_max=True)
    params = {k: v.requires_grad_(True) for k, v in params.items()}
    opt = torch.optim.Adam([{"params": [p], "lr": 1e-3} for p in params.values()], amsgrad=amsgrad)
    for _ in range(2):
        opt.zero_grad()
        sum((p * p).sum() for p in params.values()).backward()
        opt.step()
    old_params = set(map(id, params.values()))
    old_step = {k: opt.state[p]["step"].clone() for k, p in params.items()}
    state = {(k, sk): sv.clone() for k, p in params.items() for sk, sv in opt.state[p].items() if sv.dim() >= 1}
    st = stats_from(N, cuda_device, grad2d, count, max_radius)
    det = {k: v.detach() for k, v in params.items()}
    ref, ref_state, ref_counts, extra = densify_reference(det, grad2d, count, max_radius, 5.0, det["opacities"],
                                                          state=state, **kw)
    new, counts = densify_and_prune(params, st, 5.0, optimizer=opt, **kw)
    assert counts == ref_counts and counts["n_clone"] > 0 and counts["n_split"] > 0
    moments = {"exp_avg", "exp_avg_sq"} | ({"max_exp_avg_sq"} if amsgrad else set())
    for k, t in new.items():
        stt = opt.state[t]
        assert {sk for sk, sv in stt.items() if sv.dim() >= 1} == moments
        assert torch.equal(stt["step"], old_step[k])
        for sk in moments:
            assert torch.equal(stt[sk], ref_state[(k, sk)]), (k, sk)
            assert not bool(stt[sk][extra["new_row"]].any()), (k, sk)   # new rows: zero moments
            assert bool((stt[sk][~extra["new_row"]] != 0).any()), (k, sk)  # kept rows: the old ones
    groups = [p for g in opt.param_groups for p in g["params"]]
    assert {id(p) for p in groups} == {id(t) for t in new.values()}
    assert not ({id(p) for p in opt.state} & old_params) and len(opt.state) == len(new)
    opt.zero_grad()
    sum((p * p).sum() for p in new.values()).backward()
    opt.step()


# ---------------------------------------------------------------- determinism ----------------------------------------

@pytest.mark.gpu
def test_deterministic_at_1m(cuda_device):
    N = 1_000_000
    params, grad2d, count, max_radius, kw = make_case(N, 13, cuda_device, prune_max=True)
    outs = []
    for _ in range(2):
        st = stats_from(N, cuda_device, grad2d, count, max_radius)
        outs.append(densify_and_prune(dict(params), st, 5.0, generator=torch.Generator(device=cuda_device)
                                      .manual_seed(99), **kw))
    assert outs[0][1] == outs[1][1]
    for k in params:
        assert torch.equal(outs[0][0][k], outs[1][0][k]), k


# ---------------------------------------------------------------- training from a sparse start ----------------------

def sparse_fit(dev, densify, steps=600, every=100):
    """A seeded scene of 3 000 Gaussians rendered at 128 x 128 is the target; the fit starts from 150 of them with
    scales x e, l1_dssim_loss with Adam, densification every `every` steps when `densify`."""
    g = torch.Generator().manual_seed(31)
    N = 3000
    z = torch.rand(N, generator=g) * 2.0 + 2.0
    m = torch.stack([(torch.rand(N, generator=g) * 2 - 1) * 0.66 * z, (torch.rand(N, generator=g) * 2 - 1) * 0.66 * z,
                     z], 1)
    s = torch.randn(N, 3, generator=g) * 0.3 - 3.4
    q = torch.randn(N, 4, generator=g)
    o = torch.rand(N, generator=g) * 0.5 + 0.45
    c = torch.rand(N, 3, generator=g)
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=128, W=128, fx=100.0, fy=100.0, cx=64.0, cy=64.0)
    target = ms.render_gaussians_diff(*[x.to(dev) for x in (m, s, q, o, c)], cam).detach()
    pick = torch.randperm(N, generator=g)[:150]
    params = dict(means3d=m[pick], scales=s[pick] + 1.0, quats=q[pick], opacities=o[pick] * 0 + 0.5, colors=c[pick])
    params = {k: v.to(dev).requires_grad_(True) for k, v in params.items()}
    lrs = dict(means3d=2e-3, scales=1e-2, quats=1e-2, opacities=1e-2, colors=1e-2)
    opt = torch.optim.Adam([{"params": [params[k]], "lr": lrs[k]} for k in params])
    stats = DensifyStats(150, dev)
    gen = torch.Generator(device=dev).manual_seed(5)
    sizes = [150]
    for step in range(1, steps + 1):
        opt.zero_grad()
        img, aux = ms.render_gaussians_diff(*[params[k] for k in ("means3d", "scales", "quats", "opacities",
                                                                   "colors")], cam, return_aux=True)
        aux["means2d"].retain_grad()
        loss = ms.l1_dssim_loss(img, target)
        loss.backward()
        stats.accumulate(aux["means2d"].grad, aux["radii"], cam.W, cam.H)
        opt.step()
        with torch.no_grad():
            params["opacities"].clamp_(0.0, 1.0)
        if densify and step % every == 0 and step < steps:
            params, _ = densify_and_prune(params, stats, 4.0, optimizer=opt, generator=gen)
            sizes.append(params["means3d"].shape[0])
    return float(loss), sizes


@pytest.mark.gpu
def test_training_from_sparse_start(cuda_device):
    """600 steps of l1_dssim_loss from 150 enlarged Gaussians of a 3 000-Gaussian target, with and without densification
    every 100 steps.  Measured on a B200: see the printed line; the test asks N to grow at least 2x and the densified
    run to end at most 0.8x the loss of the run without."""
    loss_d, sizes = sparse_fit(cuda_device, True)
    loss_n, _ = sparse_fit(cuda_device, False)
    print(f"sparse fit: N {sizes}, final loss {loss_d:.4e} with densification, {loss_n:.4e} without "
          f"(ratio {loss_d / loss_n:.3f})")
    assert sizes[-1] >= 2 * sizes[0], sizes
    assert loss_d <= 0.8 * loss_n, (loss_d, loss_n)
