"""3DGS-MCMC densification (mcmc_refine, mcmc_inject_noise; bsplat_mcmc_*) against torch restatements.

``refine_reference`` restates ``mcmc_refine`` in torch with the same draws (the private ``_*_draws`` helpers of
mcmc.py, called with an identically seeded generator): row order, copies and optimizer state must match bit for bit,
the relocated opacities and log-scales (double in both, rounded once) within 2 fp32 ulps.  The relocation values are
also checked against the literal double sum with exact binomials, and the noise against fp64.  The argument checks,
C ABI rejections and struct sizes at the top need no GPU.
"""
import ctypes
import math

import pytest
import torch

import mojosplat_b200 as ms
from mojosplat_b200 import _lib
from mojosplat_b200.mcmc import (_add_draws, _n_add, _noise_draw, _relocate_draws, mcmc_inject_noise, mcmc_refine)

KEYS = ("means3d", "scales", "quats", "opacities", "colors", "sh")


def f32(x):
    return float(torch.tensor(x, dtype=torch.float64).float())


def ulps(a, b):
    """Distance in fp32 ulps of two fp32 tensors of one sign (the ordered integer views)."""
    return (a.contiguous().view(torch.int32).long() - b.contiguous().view(torch.int32).long()).abs()


def quat_rotmat64(q):
    q = q.double()
    q = q / q.norm(dim=1, keepdim=True).clamp_min(1e-12)
    w, x, y, z = q.unbind(1)
    return torch.stack([
        torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)], 1),
        torch.stack([2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)], 1),
        torch.stack([2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], 1)], 1)


# ---------------------------------------------------------------- fp64 restatements -----------------------------------

def relocation_literal(o, s, n, min_opacity):
    """The definition, in Python doubles: o' and s + log(o / D) with D the double sum over exact binomials."""
    o = min(o, 1.0)
    op = min(max(-math.expm1(math.log1p(-o) / n), min_opacity), 1.0 - 2.0 ** -23)
    D = 0.0
    for i in range(1, n + 1):
        for k in range(i):
            D += math.comb(i - 1, k) * (-1) ** k * op ** (k + 1) / math.sqrt(k + 1)
    return op, [si + math.log(o / D) for si in s]


BINOM = torch.tensor([[float(math.comb(n, k)) for k in range(52)] for n in range(52)], dtype=torch.float64)


def relocation_torch(o_stored, s, c, min_opacity, logits):
    """Vectorised fp64 values of rows sampled c > 0 times: (stored opacity, log-scales), fp32."""
    n = (c + 1).clamp(max=51)
    x = o_stored.double()
    o = (torch.sigmoid(x) if logits else x).clamp(max=1.0)
    op = (-torch.expm1(torch.log1p(-o) / n)).clamp(min=f32(min_opacity), max=1.0 - 2.0 ** -23)
    B = BINOM.to(o.device)
    D = torch.zeros_like(op)
    for k in range(51):
        term = B[n, k + 1] * op ** (k + 1) / math.sqrt(k + 1)
        D = D + torch.where(k < n, term * (-1) ** k, torch.zeros_like(term))
    stored = torch.log(op / (1 - op)) if logits else op
    return stored.float(), (s.double() + torch.log(o / D)[:, None]).float()


def update_sampled(p, idx, min_opacity, logits):
    N = p["means3d"].shape[0]
    c = torch.bincount(idx, minlength=N)
    rows = torch.nonzero(c).flatten()
    op = p["opacities"].view(-1)
    o_new, s_new = relocation_torch(op[rows], p["scales"][rows], c[rows], min_opacity, logits)
    op[rows] = o_new
    p["scales"][rows] = s_new
    return rows


def refine_reference(params, state, *, cap_max, min_opacity=0.005, growth=1.05, logits=False, generator=None):
    """Torch restatement of mcmc_refine.  state: {(key, name): (N, ...) tensor}.  Returns (params, state, counts)."""
    p = {k: v.detach().clone() for k, v in params.items()}
    st = {k: v.clone() for k, v in state.items()}
    N = p["means3d"].shape[0]
    counts = dict(n_dead=0, n_relocated=0, n_added=0, n_out=N)
    if N == 0:
        return p, st, counts
    dead, sampled = _relocate_draws(p, min_opacity, logits, generator)
    counts["n_dead"] = dead.numel()
    if sampled is not None:
        rows = update_sampled(p, sampled, min_opacity, logits)
        for k in p:
            p[k][dead] = p[k][sampled]
        for t in st.values():
            t[rows] = 0
            t[dead] = 0
        counts["n_relocated"] = dead.numel()
    n_add = _n_add(N, cap_max, growth)
    added = _add_draws(p, n_add, logits, generator)
    if added is None:
        return p, st, counts
    update_sampled(p, added, min_opacity, logits)
    p = {k: torch.cat([v, v[added]]) for k, v in p.items()}
    st = {k: torch.cat([v, torch.zeros_like(v[added])]) for k, v in st.items()}
    counts.update(n_added=n_add, n_out=N + n_add)
    return p, st, counts


def assert_params_match(got, ref):
    for k, t in ref.items():
        g = got[k].detach()
        assert g.shape == t.shape, (k, g.shape, t.shape)
        if k in ("opacities", "scales"):
            assert g.numel() == 0 or int(ulps(g, t).max()) <= 2, (k, int(ulps(g, t).max()))
        else:
            assert torch.equal(g, t), k


# ---------------------------------------------------------------- cases ----------------------------------------------

def make_case(N, seed, dev, logits=False, dup=False, dead_frac=0.3):
    """Parameters of widths 3, 3, 4, 1, 3 and 48; a fraction `dead_frac` of rows below the 0.005 default.  dup: a few
    opaque rows and many faint ones, so the samples are heavy with duplicates."""
    g = torch.Generator().manual_seed(seed)
    o = torch.rand(N, generator=g) * 0.9 + 0.05
    if dup:
        o = torch.where(torch.rand(N, generator=g) < 0.002, 0.99, 0.0052 + torch.rand(N, generator=g) * 0.002)
    o = torch.where(torch.rand(N, generator=g) < dead_frac, torch.rand(N, generator=g) * 0.004, o)
    params = dict(
        means3d=torch.randn(N, 3, generator=g) * 2.0,
        scales=torch.rand(N, 3, generator=g) * 3.0 - 5.0,
        quats=torch.randn(N, 4, generator=g) * (0.3 + torch.rand(N, 1, generator=g)),
        opacities=torch.log(o / (1 - o)) if logits else o,
        colors=torch.rand(N, 3, generator=g),
        sh=torch.randn(N, 16, 3, generator=g))
    return {k: v.to(dev).contiguous() for k, v in params.items()}


def make_adam(params, amsgrad=False):
    ps = {k: v.requires_grad_(True) for k, v in params.items()}
    opt = torch.optim.Adam([{"params": [p], "lr": 1e-3} for p in ps.values()], amsgrad=amsgrad)
    for _ in range(2):
        opt.zero_grad()
        sum((p * p).sum() for p in ps.values()).backward()
        opt.step()
    return ps, opt


def state_of(params, opt):
    if opt is None:
        return {}
    return {(k, sk): sv for k, p in params.items() for sk, sv in opt.state[p].items() if sv.dim() >= 1}


def run_both(params, opt, dev, seed, **kw):
    state = {key: t.clone() for key, t in state_of(params, opt).items()}
    ref, ref_state, ref_counts = refine_reference(params, state, generator=torch.Generator().manual_seed(seed),
                                                  logits=kw.get("opacity_logits", False),
                                                  **{k: v for k, v in kw.items() if k != "opacity_logits"})
    new, counts = mcmc_refine(params, optimizer=opt, generator=torch.Generator().manual_seed(seed), **kw)
    assert counts == ref_counts, (counts, ref_counts)
    assert_params_match(new, ref)
    if opt is not None:
        got_state = state_of(new, opt)
        assert set(got_state) == set(ref_state)
        for key, t in ref_state.items():
            assert torch.equal(got_state[key], t), key
    return new, counts


# ---------------------------------------------------------------- arguments and ABI (no GPU) -------------------------

@pytest.fixture(scope="module")
def lib():
    if not _lib.LIB_PATH.exists():
        _lib.build()
    return _lib.load()


def test_struct_sizes():
    assert ctypes.sizeof(_lib.BsplatMcmcParams) == 8
    assert ctypes.sizeof(_lib.BsplatMcmcTensor) == 24


def test_arguments_rejected_without_gpu():
    z = torch.zeros
    p = dict(means3d=z(4, 3), scales=z(4, 3), quats=z(4, 4), opacities=z(4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mcmc_refine(p, cap_max=10)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mcmc_inject_noise(p, 1.0)
    with pytest.raises(ValueError, match="must hold 'opacities'"):
        mcmc_refine({k: v for k, v in p.items() if k != "opacities"}, cap_max=10)
    with pytest.raises(ValueError, match="min_opacity"):
        mcmc_refine(p, cap_max=10, min_opacity=0.0)
    with pytest.raises(ValueError, match="cap_max"):
        mcmc_refine(p, cap_max=-1)
    with pytest.raises(ValueError, match="finite"):
        mcmc_inject_noise(p, float("nan"))
    # 2^24 + 1 rows (expanded views: no memory) are rejected before anything touches a device
    big = 2 ** 24 + 1
    pb = dict(means3d=z(1, 3).expand(big, 3), scales=z(1, 3).expand(big, 3), quats=z(1, 4).expand(big, 4),
              opacities=z(1).expand(big))
    with pytest.raises(ValueError, match="2\\^24"):
        mcmc_refine(pb, cap_max=big)
    with pytest.raises(ValueError, match="2\\^24"):
        mcmc_inject_noise(pb, 1.0)


def test_c_abi_rejections_without_gpu(lib):
    """Argument rules of the C entry points: every one of these returns before anything reaches a device."""
    prm = _lib.BsplatMcmcParams(0.005, 0)
    O, S, C, T = _lib.MCMC_OPACITY, _lib.MCMC_LOG_SCALES, _lib.MCMC_COPY, _lib.MCMC_STATE
    need = lib.bsplat_mcmc_workspace_bytes(1000)
    assert need >= 20 * 1000 and lib.bsplat_mcmc_workspace_bytes(-1) == 0

    def desc(rows, in_place):
        d = (_lib.BsplatMcmcTensor * max(len(rows), 1))()
        for x, (src, w, role) in zip(d, rows):
            x.src, x.dst, x.width, x.role = src, src if in_place else src + 0x100000, w, role
        return d

    base = [(0x1000, 1, O), (0x2000, 3, S), (0x3000, 3, C), (0x4000, 3, T)]
    ws = ctypes.c_void_p(0x10000)

    def reloc(rows, n=None, N=1000, n_dead=10, ws_bytes=need, params=prm, needed=None, in_place=True):
        return lib.bsplat_mcmc_relocate(N, n_dead, ctypes.c_void_p(0x5000), ctypes.c_void_p(0x6000),
                                        None if params is None else ctypes.byref(params),
                                        len(rows) if n is None else n, desc(rows, in_place), ws, ws_bytes, needed,
                                        None)

    def add(rows, n=None, N=1000, n_add=10, ws_bytes=need, in_place=False):
        return lib.bsplat_mcmc_add(N, n_add, ctypes.c_void_p(0x6000), ctypes.byref(prm),
                                   len(rows) if n is None else n, desc(rows, in_place), ws, ws_bytes, None, None)

    E = _lib.E_ARG
    assert reloc(base, n=0) == E
    assert reloc(base + [(0x7000, 1, C)] * 29) == E                        # 33 tensors
    assert reloc(base + [(0x7000, 0, C)]) == E                             # width 0
    assert reloc(base + [(0x7000, 257, C)]) == E                           # width 257
    assert reloc(base + [(0x7000, 4, 9)]) == E                             # unknown role
    assert reloc(base[1:]) == E                                            # no OPACITY
    assert reloc([base[0]] + base[2:]) == E                                # no LOG_SCALES
    assert reloc([(0x1000, 3, O)] + base[1:]) == E                         # OPACITY of width 3
    assert reloc(base + [(0x7000, 1, O)]) == E                             # two OPACITY
    assert reloc(base, in_place=False) == E                                # relocate is in place
    assert add(base, in_place=True) == E                                   # add is not
    assert reloc(base + [(0, 3, C)]) == E                                  # null src
    assert reloc(base, params=None) == E
    assert reloc(base, N=-1) == E
    assert reloc(base, n_dead=1001) == E and reloc(base, n_dead=-1) == E
    assert add(base, n_add=-1) == E
    got = ctypes.c_size_t(0)
    assert reloc(base, ws_bytes=need - 1, needed=ctypes.byref(got)) == _lib.E_WORKSPACE and got.value == need
    assert add(base, ws_bytes=16) == _lib.E_WORKSPACE
    assert reloc(base, n_dead=0) == _lib.OK                                # nothing dead: nothing launched
    assert lib.bsplat_mcmc_relocate(0, 0, None, None, ctypes.byref(prm), 4, desc(base, True), None, 0, None,
                                    None) == _lib.OK                       # N = 0
    f = [ctypes.c_void_p(0x1000 * (i + 1)) for i in range(5)]
    assert lib.bsplat_mcmc_noise(-1, *f, 1.0, ctypes.byref(prm), None) == E
    assert lib.bsplat_mcmc_noise(10, *f, 1.0, None, None) == E
    assert lib.bsplat_mcmc_noise(10, f[0], f[1], ctypes.c_void_p(0x3004), f[3], f[4], 1.0, ctypes.byref(prm),
                                 None) == E                                # quats not 16-byte aligned
    assert lib.bsplat_mcmc_noise(10, f[0], None, f[2], f[3], f[4], 1.0, ctypes.byref(prm), None) == E
    assert lib.bsplat_mcmc_noise(0, None, None, None, None, None, 1.0, ctypes.byref(prm), None) == _lib.OK


@pytest.mark.gpu
def test_arguments_rejected_on_gpu(cuda_device):
    params = make_case(16, 0, cuda_device)
    with pytest.raises(ValueError, match="leading rows"):
        mcmc_refine(dict(params, colors=params["colors"][:15]), cap_max=20)
    with pytest.raises(ValueError, match="contiguous"):
        mcmc_refine(dict(params, colors=params["colors"].t().contiguous().t()), cap_max=20)
    with pytest.raises(ValueError, match="at most 32"):
        mcmc_refine(dict(params, **{f"x{i}": torch.zeros(16, device=cuda_device) for i in range(27)}), cap_max=20)
    with pytest.raises(ValueError, match="1..256"):
        mcmc_refine(dict(params, big=torch.zeros(16, 257, device=cuda_device)), cap_max=20)
    stray = torch.zeros(16, 3, device=cuda_device, requires_grad=True)
    opt = torch.optim.Adam([params["means3d"].requires_grad_(True), stray])
    with pytest.raises(ValueError, match="not in params"):
        mcmc_refine(params, cap_max=20, optimizer=opt)
    with pytest.raises(ValueError, match="CPU torch.Generator"):
        mcmc_refine(params, cap_max=20, generator=torch.Generator(device=cuda_device))


# ---------------------------------------------------------------- relocation values ----------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("logits", [False, True])
@pytest.mark.parametrize("min_opacity", [1e-8, 0.005])
def test_relocation_values(cuda_device, logits, min_opacity):
    """Every o in the list sampled c = 1..50 times (n = 2..51) and 55 / 80 times (n clamped to 51), through the C ABI;
    an unsampled row (n = 1) of every o comes back bit for bit."""
    lib = _lib.require_device(cuda_device)
    os_ = [1e-6, 0.005, 0.1, 0.5, 0.9, 0.99, 1 - 2 ** -23]
    cs = list(range(0, 51)) + [55, 80]
    rows = [(o, c) for o in os_ for c in cs]
    n_alive = len(rows)
    sampled = [i for i, (_, c) in enumerate(rows) for _ in range(c)]
    n_dead = len(sampled)
    N = n_alive + n_dead
    o32 = torch.tensor([o for o, _ in rows] + [0.0] * n_dead, dtype=torch.float32)
    stored = torch.log(o32.double() / (1 - o32.double())).float() if logits else o32
    stored[n_alive:] = -30.0 if logits else 0.0
    g = torch.Generator().manual_seed(1)
    scales = torch.rand(N, 3, generator=g) * 4 - 4
    colors = torch.rand(N, 5, generator=g)
    state = torch.rand(N, 3, generator=g) + 1
    before = [t.clone() for t in (stored, scales, colors, state)]
    dev_t = [t.to(cuda_device) for t in (stored, scales, colors, state)]
    perm = torch.randperm(n_dead, generator=g)   # dead rows in a shuffled order
    dead = (torch.arange(n_alive, N)[perm]).to(cuda_device)
    samp = torch.tensor(sampled, dtype=torch.int64).to(cuda_device)
    desc = (_lib.BsplatMcmcTensor * 4)()
    for d, t, w, role in zip(desc, dev_t, (1, 3, 5, 3), (_lib.MCMC_OPACITY, _lib.MCMC_LOG_SCALES, _lib.MCMC_COPY,
                                                         _lib.MCMC_STATE)):
        d.src = d.dst = t.data_ptr()
        d.width, d.role = w, role
    ws = torch.empty(lib.bsplat_mcmc_workspace_bytes(N), dtype=torch.uint8, device=cuda_device)
    prm = _lib.BsplatMcmcParams(min_opacity, 1 if logits else 0)
    _lib.check(lib.bsplat_mcmc_relocate(N, n_dead, _lib.ptr(dead), _lib.ptr(samp), ctypes.byref(prm), 4, desc,
                                        _lib.ptr(ws), ws.numel(), None, _lib.stream_ptr(cuda_device)),
               "bsplat_mcmc_relocate")
    got = [t.cpu() for t in dev_t]
    worst = 0
    for i, (o, c) in enumerate(rows):
        if c == 0:
            for a, b in zip(got, before):
                assert torch.equal(a[i], b[i]), i
            continue
        x = float(before[0][i])
        oo = 1.0 / (1.0 + math.exp(-x)) if logits else x
        op, s_new = relocation_literal(oo, before[1][i].double().tolist(), min(c + 1, 51), f32(min_opacity))
        ref_o = torch.tensor([math.log(op / (1 - op)) if logits else op], dtype=torch.float64).float()
        ref_s = torch.tensor(s_new, dtype=torch.float64).float()
        worst = max(worst, int(ulps(got[0][i:i + 1], ref_o).max()), int(ulps(got[1][i], ref_s).max()))
        assert torch.equal(got[2][i], before[2][i]) and not bool(got[3][i].any()), i
    print(f"relocation values: worst {worst} fp32 ulps from the fp64 double sum")
    assert worst <= 2
    # dead row perm-order k is a copy of updated sampled row k, with zero state
    src = torch.tensor(sampled)
    dst = torch.arange(n_alive, N)[perm]
    for a in got[:3]:
        assert torch.equal(a[dst], a[src])
    assert not bool(got[3][n_alive:].any())


# ---------------------------------------------------------------- mcmc_refine vs the restatement ---------------------

@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 1000, 100_000, 1_000_000])
@pytest.mark.parametrize("logits", [False, True])
def test_refine_matches_reference(cuda_device, N, logits):
    params, opt = make_adam(make_case(N, N % 89 + logits, cuda_device, logits=logits))
    new, counts = run_both(params, opt, cuda_device, seed=N + 3, cap_max=int(1.2 * N) + 10, opacity_logits=logits)
    print(N, logits, counts)
    if N >= 1000:
        assert counts["n_relocated"] == counts["n_dead"] > 0.2 * N and counts["n_added"] == int(1.05 * N) - N
    for k, t in new.items():
        assert t.requires_grad and t.shape[1:] == params[k].shape[1:]
        assert (t is params[k]) == (counts["n_added"] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("logits", [False, True])
def test_refine_heavy_duplicates(cuda_device, logits):
    params = make_case(50_000, 7, cuda_device, logits=logits, dup=True)
    new, counts = run_both(params, None, cuda_device, seed=9, cap_max=60_000, opacity_logits=logits)
    assert counts["n_added"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("amsgrad", [False, True])
def test_refine_optimizer_state(cuda_device, amsgrad):
    params, opt = make_adam(make_case(20_000, 12, cuda_device), amsgrad)
    old_step = {k: opt.state[p]["step"].clone() for k, p in params.items()}
    dead = torch.nonzero(params["opacities"].detach() <= f32(0.005)).flatten()
    new, counts = run_both(params, opt, cuda_device, seed=4, cap_max=30_000)
    moments = {"exp_avg", "exp_avg_sq"} | ({"max_exp_avg_sq"} if amsgrad else set())
    N = 20_000
    for k, t in new.items():
        st = opt.state[t]
        assert {sk for sk, sv in st.items() if sv.dim() >= 1} == moments and torch.equal(st["step"], old_step[k])
        for sk in moments:
            assert not bool(st[sk][dead].any()) and not bool(st[sk][N:].any()), (k, sk)
    assert {id(p) for g in opt.param_groups for p in g["params"]} == {id(t) for t in new.values()}
    opt.zero_grad()
    sum((p * p).sum() for p in new.values()).backward()
    opt.step()


# ---------------------------------------------------------------- edge cases -----------------------------------------

@pytest.mark.gpu
def test_no_dead_rows(cuda_device):
    params = make_case(5000, 2, cuda_device, dead_frac=0.0)
    new, counts = run_both(params, None, cuda_device, seed=1, cap_max=10_000)
    assert counts == dict(n_dead=0, n_relocated=0, n_added=250, n_out=5250)


@pytest.mark.gpu
@pytest.mark.parametrize("logits", [False, True])
def test_every_row_dead(cuda_device, logits):
    params = make_case(3000, 3, cuda_device, logits=logits, dead_frac=1.0)
    new, counts = run_both(params, None, cuda_device, seed=2, cap_max=10_000, opacity_logits=logits)
    assert counts == dict(n_dead=3000, n_relocated=0, n_added=150, n_out=3150)
    params["opacities"].zero_()   # raw 0 / sigmoid(0) = 0.5: no weight left in raw mode only
    _, counts = mcmc_refine(params, cap_max=10_000, opacity_logits=logits)
    assert counts["n_added"] == (150 if logits else 0)


@pytest.mark.gpu
@pytest.mark.parametrize("N, cap", [(4000, 4000), (4000, 100), (19, 100)])
def test_nothing_added_returns_same_objects(cuda_device, N, cap):
    """Cap reached (or below N), and a small N where int(1.05 N) == N: the same tensors come back, relocated in place."""
    params, opt = make_adam(make_case(N, 5, cuda_device))
    ids = {k: id(v) for k, v in params.items()}
    new, counts = run_both(params, opt, cuda_device, seed=3, cap_max=cap)
    assert counts["n_added"] == 0 and counts["n_relocated"] > 0 and counts["n_out"] == N
    assert {k: id(v) for k, v in new.items()} == ids


@pytest.mark.gpu
def test_empty_set(cuda_device):
    params = make_case(0, 0, cuda_device)
    new, counts = mcmc_refine(params, cap_max=10)
    assert counts == dict(n_dead=0, n_relocated=0, n_added=0, n_out=0) and new["sh"].shape == (0, 16, 3)
    mcmc_inject_noise(params, 1.0)


# ---------------------------------------------------------------- noise ----------------------------------------------

def noise_reference(params, noise, scale, logits):
    """fp64 mu + scale * sigmoid(100 ((1 - o) - 0.995)) * R S^2 R^T n, and a magnitude for the fp32 error bound:
    |mu| + |R| S^2 |R^T| |v| + sum_j S^2_j (|R^T| |v|)_j.  The last term covers the absolute error of every entry of R
    (a few ulps of 1, whatever the entry's size) times the intermediate S^2 R^T v."""
    x = params["opacities"].double().reshape(-1)
    one_m_o = torch.sigmoid(-x) if logits else 1 - x
    g = torch.sigmoid(100 * (one_m_o - 0.995))
    R = quat_rotmat64(params["quats"])
    S2 = torch.exp(2 * params["scales"].double())
    v = noise.double() * (f32(scale) * g)[:, None]
    cov = R @ torch.diag_embed(S2) @ R.transpose(1, 2)
    mu = params["means3d"].double()
    d = (cov @ v[..., None])[..., 0]
    t_abs = (R.abs().transpose(1, 2) @ v.abs()[..., None])[..., 0] * S2
    mag = mu.abs() + (R.abs() @ t_abs[..., None])[..., 0] + t_abs.sum(dim=1, keepdim=True)
    return mu + d, mag, d


@pytest.mark.gpu
@pytest.mark.parametrize("logits", [False, True])
def test_noise_matches_fp64(cuda_device, logits):
    N = 200_003
    params = make_case(N, 21, cuda_device, logits=logits)
    params["quats"][:50] = 0.0                      # degenerate: R = I
    params["quats"][50:100] *= 1e4                  # far from unit length
    o = torch.linspace(0, 1, N, device=cuda_device)  # the whole gate, opaque rows included
    params["opacities"] = torch.log(o / (1 - o)).contiguous() if logits else o
    scale = 2e-3 * 5e5
    before = {k: v.clone() for k, v in params.items()}
    noise = _noise_draw(N, cuda_device, torch.Generator(device=cuda_device).manual_seed(8))
    ref, mag, d = noise_reference(before, noise, scale, logits)
    mcmc_inject_noise(params, scale, opacity_logits=logits, generator=torch.Generator(device=cuda_device).manual_seed(8))
    for k in KEYS[1:]:
        assert torch.equal(params[k], before[k]), k
    err = (params["means3d"].double() - ref).abs()
    assert bool((err <= 16 * 2.0 ** -24 * mag + 1e-30).all()), float((err / mag.clamp_min(1e-30)).max())
    opaque = o > 0.9
    assert float(d[opaque].abs().max()) < 1e-20 and bool(torch.equal(params["means3d"][opaque],
                                                                       before["means3d"][opaque]))
    assert float(d[~opaque].abs().max()) > 1e-3


@pytest.mark.gpu
def test_noise_scale_zero_is_identity(cuda_device):
    params = make_case(10_000, 22, cuda_device)
    params["means3d"][:10] = -0.0
    before = params["means3d"].clone()
    mcmc_inject_noise(params, 0.0)
    assert torch.equal(params["means3d"].view(torch.int32), before.view(torch.int32))


# ---------------------------------------------------------------- determinism ----------------------------------------

@pytest.mark.gpu
def test_deterministic_at_1m(cuda_device):
    N = 1_000_000
    base = make_case(N, 13, cuda_device)
    outs = []
    for _ in range(2):
        params, opt = make_adam({k: v.clone() for k, v in base.items()})
        mcmc_inject_noise(params, 1e3, generator=torch.Generator(device=cuda_device).manual_seed(99))
        new, counts = mcmc_refine(params, cap_max=2 * N, optimizer=opt, generator=torch.Generator().manual_seed(98))
        outs.append((new, counts, state_of(new, opt)))
    assert outs[0][1] == outs[1][1] and outs[0][1]["n_added"] > 0
    for k in KEYS:
        assert torch.equal(outs[0][0][k], outs[1][0][k]), k
    for key in outs[0][2]:
        assert torch.equal(outs[0][2][key], outs[1][2][key]), key


# ---------------------------------------------------------------- training from a sparse random start ---------------

@pytest.mark.gpu
def test_training_fit(cuda_device):
    """400 steps of l1_dssim_loss plus gsplat's two regularisers from 150 random Gaussians towards a 3 000-Gaussian
    target at 128 x 128, logit opacities, noise every step, refine every 50 steps from step 50 to 300 with growth 1.5
    and cap_max 600."""
    dev = cuda_device
    g = torch.Generator().manual_seed(31)
    N = 3000
    z = torch.rand(N, generator=g) * 2.0 + 2.0
    m = torch.stack([(torch.rand(N, generator=g) * 2 - 1) * 0.66 * z, (torch.rand(N, generator=g) * 2 - 1) * 0.66 * z,
                     z], 1)
    cam = ms.Camera(R=torch.eye(3), T=torch.zeros(3), H=128, W=128, fx=100.0, fy=100.0, cx=64.0, cy=64.0)
    target = ms.render_gaussians_diff(m.to(dev), (torch.randn(N, 3, generator=g) * 0.3 - 3.4).to(dev),
                                      torch.randn(N, 4, generator=g).to(dev),
                                      (torch.rand(N, generator=g) * 0.5 + 0.45).to(dev),
                                      torch.rand(N, 3, generator=g).to(dev), cam).detach()
    n0 = 150
    z0 = torch.rand(n0, generator=g) * 2.0 + 2.0
    params = dict(means3d=torch.stack([(torch.rand(n0, generator=g) * 2 - 1) * 0.66 * z0,
                                       (torch.rand(n0, generator=g) * 2 - 1) * 0.66 * z0, z0], 1),
                  scales=torch.full((n0, 3), -2.4), quats=torch.randn(n0, 4, generator=g),
                  opacities=torch.full((n0,), 0.0), colors=torch.rand(n0, 3, generator=g))
    params = {k: v.to(dev).contiguous().requires_grad_(True) for k, v in params.items()}
    lrs = dict(means3d=2e-3, scales=1e-2, quats=1e-2, opacities=5e-2, colors=1e-2)
    opt = torch.optim.Adam([{"params": [params[k]], "lr": lrs[k]} for k in params])
    gen, cpu_gen = torch.Generator(device=dev).manual_seed(5), torch.Generator().manual_seed(6)
    sizes, losses = [n0], []
    for step in range(1, 401):
        opt.zero_grad()
        o = torch.sigmoid(params["opacities"])
        img = ms.render_gaussians_diff(params["means3d"], params["scales"], params["quats"], o, params["colors"], cam)
        loss = ms.l1_dssim_loss(img, target)
        losses.append(float(loss))
        (loss + 0.01 * o.abs().mean() + 0.01 * torch.exp(params["scales"]).abs().mean()).backward()
        opt.step()
        if step % 50 == 0 and step <= 300:
            params, _ = mcmc_refine(params, cap_max=600, growth=1.5, opacity_logits=True, optimizer=opt,
                                    generator=cpu_gen)
            sizes.append(params["means3d"].shape[0])
        mcmc_inject_noise(params, lrs["means3d"] * 5e5, opacity_logits=True, generator=gen)
    first, last = sum(losses[:5]) / 5, sum(losses[-5:]) / 5
    print(f"MCMC fit: N {sizes}, loss {first:.4e} -> {last:.4e} (x{first / last:.2f})")
    assert max(sizes) <= 600 and sizes[-1] == 600, sizes
    assert last <= first / 2.0, (first, last)
