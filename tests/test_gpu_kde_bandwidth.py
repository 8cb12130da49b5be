"""GPU parity of the KDE kernels across the bandwidths users choose, against float64 evaluations of the reference's
dense form (diagnostics/histogram.py:11-74).

The kernels compile one window per bandwidth range: R = 4 bins on either side up to sigma / bin spacing = 0.5085, 9 up
to 1.0734 and (1-D only) 13 up to 1.5254; each range ends where the window stops at 8.85 sigma.  The taps come from
recurrences, whose factors must stay finite for nearly hard screens (sigma of 0.05 bin) as well.  These tests run every
template, both sides of every boundary and the top of each range, screens with different edges and bandwidths in one
launch, both 2-D paths, the functional interface and the refusal of bandwidths beyond the compiled windows.

Inputs are chosen so that the fp32 projection and the bin position are exact: coordinates on a 2^-12 grid, projection
rows in steps of 1/16, bin widths that are powers of two.  The comparisons then measure the kernels' tap arithmetic and
reductions, not the rounding of u = w . x, which at sigma = 0.05 bin would move a tap by 1e-4 of itself."""
import math

import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200 import _lib, ops
from mentflow_b200.diagnostics.histogram import kde_histogram_1d, kde_histogram_2d
from mentflow_b200.simulate import simulate as sim
from mfb_testutil import profile_err
from oracle import hotpath as hp

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1.0e-4        # profiles, KL, gradients (relative to max |grad|)
TOL_SUMS = 2.0e-5   # unnormalised sums, relative to the largest sum


# ---- inputs and geometry --------------------------------------------------------------------------------------
def grid_x(n, d, gen, scale=1.0):
    """particles on a 2^-12 grid (|x| < 8: 15 significant bits)"""
    x = torch.randn(n, d, generator=gen, dtype=torch.float64) * scale
    return (torch.round(x * 4096) / 4096).float()


def grid_w(k, d, gen):
    """projection rows in steps of 1/16: every product and partial sum with grid_x is exact in fp32"""
    w = torch.round(torch.randn(k, d, generator=gen, dtype=torch.float64) / math.sqrt(d) * 16) / 16
    w[w.abs().sum(dim=1) == 0, 0] = 1.0
    return w.float()


def geom_1d(edges_list, rel_bandwidths):
    """One C-ABI geometry record [c0, spacing, sigma, delta, 0...] per screen, each with its own edges and bandwidth
    (relative to the bin width, as ``Histogram1D(bandwidth=...)``).  Returns (geom (K, 8), sigmas, launch ratio)."""
    rows, sigmas, ratio = [], [], 0.0
    for e, bw in zip(edges_list, rel_bandwidths):
        e = e.float()
        c = 0.5 * (e[:-1] + e[1:])
        spacing = float((c[-1].double() - c[0].double()) / (c.numel() - 1))
        sigma = float(torch.tensor(bw, dtype=torch.float32) * (e[1] - e[0]))
        rows.append([float(c[0]), spacing, sigma, float(c[1] - c[0]), 0.0, 0.0, 0.0, 0.0])
        sigmas.append(sigma)
        ratio = max(ratio, sigma / spacing)
    return torch.tensor(rows, dtype=torch.float32), sigmas, ratio


def template_radius(ratio, dims=1):
    """compiled window the kernels run for a launch ratio sigma / bin spacing (kde1d.cu window_radius)"""
    r = max(1, math.ceil(8.85 * float(torch.tensor(ratio, dtype=torch.float32)) - 0.5))
    return 4 if r <= 4 else (9 if r <= 9 else (13 if dims == 1 else None))


def measurements(k, nb, delta, gen):
    """normalised targets with empty bins (0 log 0 = 0)"""
    m = torch.rand(k, nb, generator=gen, dtype=torch.float64)
    m[:, : nb // 4] = 0.0
    return m / (m.sum(dim=1, keepdim=True) * delta)


def rel_max(a, b):
    a, b = a.detach().to(DEV, torch.float64), b.detach().to(DEV, torch.float64)
    return float((a - b).abs().max() / b.abs().max())


# ---- float64 oracles ----------------------------------------------------------------------------------------------
def oracle_1d(x, w, edges_list, sigmas, meas, coef, side, gsums):
    """float64 sums, profiles, KL, dL/dx of L = sum_k coef_k KL_k + <side, profiles> and d<gsums, sums>/dx."""
    xd = x.to(DEV, torch.float64).requires_grad_(True)
    wd = w.to(DEV, torch.float64)
    u = [xd @ wd[k] for k in range(len(sigmas))]
    edges = [e.to(DEV, torch.float64) for e in edges_list]
    sums = torch.stack([hp.kde_sums_1d(u[k], edges[k], sigmas[k]) for k in range(len(sigmas))])
    prof = torch.stack([hp.kde_profile_1d(u[k], edges[k], sigmas[k]) for k in range(len(sigmas))])
    kl = torch.stack([hp.kl_div(prof[k], meas[k]) for k in range(len(sigmas))])
    grad_sums, = torch.autograd.grad((sums * gsums).sum(), xd, retain_graph=True)
    grad_loss, = torch.autograd.grad((kl * coef).sum() + (prof * side).sum(), xd)
    return sums.detach(), prof.detach(), kl.detach(), grad_loss, grad_sums


def check_1d(x, w, edges_list, rel_bandwidths, gen, what):
    """kde1d_sums, the fused loss tail (profiles + KL) and dL/dx of one launch against the float64 oracle."""
    k, nb = w.shape[0], edges_list[0].numel() - 1
    geom, sigmas, ratio = geom_1d(edges_list, rel_bandwidths)
    delta = float(geom[0, 3])
    meas = measurements(k, nb, delta, gen).to(DEV)
    coef = torch.linspace(0.5, 1.5, k, dtype=torch.float64, device=DEV)
    side = torch.randn(k, nb, generator=gen, dtype=torch.float64).to(DEV)
    gsums = torch.randn(k, nb, generator=gen).to(DEV)
    ref_sums, ref_prof, ref_kl, ref_grad, ref_grad_sums = oracle_1d(x, w, edges_list, sigmas, meas, coef, side,
                                                                    gsums.double())

    xg, wg, gg = x.to(DEV), w.to(DEV), geom.to(DEV)
    sums = ops.kde1d_sums(xg, wg, gg, ratio, nb)
    assert torch.isfinite(sums).all(), f"{what}: non-finite sums"
    err = rel_max(sums, ref_sums)
    assert err < TOL_SUMS, f"{what}: sums {err:.2e}"
    # the particle backward kernel alone: dL/dx for a given dL/dsums
    gx = ops.kde1d_grad_x(xg, wg, gg, ratio, gsums)
    assert torch.isfinite(gx).all(), f"{what}: non-finite d<gsums, sums>/dx"
    err = rel_max(gx, ref_grad_sums)
    assert err < TOL, f"{what}: d<gsums, sums>/dx {err:.2e} of max |grad|"

    xr = xg.clone().requires_grad_(True)
    prof, kl = ops.project_kde1d(xr, wg, gg, ratio, nb, None, meas.float())     # deposit + fused finish kernel
    assert torch.isfinite(prof).all() and torch.isfinite(kl).all(), f"{what}: non-finite profiles / KL"
    err = profile_err(prof.detach(), ref_prof)
    assert err < TOL, f"{what}: profiles {err:.2e}"
    err = float(((kl.double() - ref_kl).abs() / ref_kl.abs().clamp_min(1e-30)).max())
    assert err < TOL, f"{what}: KL {err:.2e}"
    ((kl.double() * coef).sum() + (prof.double() * side).sum()).backward()
    assert torch.isfinite(xr.grad).all(), f"{what}: non-finite dL/dx"
    if x.shape[0] == 1 and ratio < 0.25:
        # One particle under a kernel narrower than a quarter bin: p_b delta ~ 1 in its bin whatever u, so the
        # normalisation's backward cancels the O(1 / sigma) terms of that bin and dL/dx is the residual of taps 1e-9 ..
        # 1e-18 below the peak (1e-6 of the cancelling terms at bandwidth 0.08).  Any fp32 evaluation keeps ~1e-7 of
        # the cancelling terms, so the loss gradient is only checked for finiteness here; the backward kernel itself
        # was checked against d<gsums, sums>/dx above, which has no such cancellation.
        return
    err = rel_max(xr.grad, ref_grad)
    assert err < TOL, f"{what}: dL/dx {err:.2e} of max |grad|"


# ---- 1-D: every template, both sides of every boundary -------------------------------------------------------------
BANDWIDTHS = [0.05, 0.08, 0.1, 0.2, 0.505, 0.515, 0.75, 1.07, 1.08, 1.52]


@pytest.mark.parametrize("d", [2, 3, 6])          # D = 3 runs the generic (runtime dimension) template
@pytest.mark.parametrize("bw", BANDWIDTHS)
def test_kde1d_bandwidth_sweep_vs_float64(bw, d):
    gen = torch.Generator().manual_seed(round(bw * 1000) + d)
    k, nb = 5, 64
    edges = [torch.linspace(-4.0, 4.0, nb + 1)] * k
    assert template_radius(geom_1d(edges, [bw] * k)[2]) == (4 if bw < 0.51 else (9 if bw < 1.075 else 13))
    w = grid_w(k, d, gen)
    for n in (1, 4099):                           # one particle; a batch that fills no tile evenly
        x = grid_x(n, d, gen, scale=0.5 if n == 1 else 1.0)      # the single particle lands on the screen
        check_1d(x, w, edges, [bw] * k, gen, f"bw={bw} d={d} n={n}")


@pytest.mark.parametrize("k,bw,n", [(300, 1.52, 3001), (600, 0.5, 2049), (600, 1.52, 1000)])
def test_kde1d_projection_count_edges(k, bw, n):
    """K = 300 at R = 13: the backward's gradient tables fit 286 projections per launch (D = 6, B = 64), so the
    second launch accumulates into dL/dx.  K = 600: two blocks of projections (gridDim.y) in the deposit."""
    gen = torch.Generator().manual_seed(k + n)
    nb = 64
    edges = [torch.linspace(-4.0, 4.0, nb + 1)] * k
    check_1d(grid_x(n, 6, gen), grid_w(k, 6, gen), edges, [bw] * k, gen, f"K={k} bw={bw}")


@pytest.mark.parametrize("d,order,skew", [(2, 4, False), (6, 3, True)])
def test_multipole_chain_at_the_widest_window(d, order, skew):
    """linear -> kick -> linear at bandwidth 1.25 (R = 13 template of the multipole deposit and backward) vs the dense
    float64 oracle through the transform classes, profiles and the particle gradient."""
    gen = torch.Generator().manual_seed(10 * d + order)
    n, k, nb = 5000, 5, 64
    x = (torch.randn(n, d, generator=gen) * 0.7).float()
    edges = torch.linspace(-3.5, 3.5, nb + 1)
    chains, cpu_chains = [], []
    for i in range(k):
        pre = torch.eye(d) + 0.3 * torch.randn(d, d, generator=gen)
        post = torch.eye(d) + 0.3 * torch.randn(d, d, generator=gen)
        st = 0.5 - 0.2 * i
        cpu_chains.append(mf.simulate.CompositeTransform(mf.simulate.LinearTransform(pre.double()),
                                                         mf.simulate.MultipoleTransform(order, st, skew),
                                                         mf.simulate.LinearTransform(post.double())))
        chains.append(mf.simulate.CompositeTransform(mf.simulate.LinearTransform(pre.cuda()),
                                                     mf.simulate.MultipoleTransform(order, st, skew),
                                                     mf.simulate.LinearTransform(post.cuda())))
    diag = mf.diagnostics.Histogram1D(axis=0, edges=edges, bandwidth=1.25).to(DEV)
    xg = x.cuda().requires_grad_(True)
    sim._plan_cache.clear()
    out = mf.simulate.forward(xg, chains, [[diag] for _ in chains])
    plan = next(iter(sim._plan_cache.values()))
    grp = plan.groups[("1d-mp", True, nb)]
    assert template_radius(grp.cache["ratio"]) == 13
    side = torch.randn(k, nb, generator=gen).cuda()
    got = torch.stack([o[0] for o in out])
    (got * side).sum().backward()
    sigma = float(diag.bandwidth)
    xr = x.double().requires_grad_(True)
    ref = torch.stack([hp.kde_profile_1d(c(xr)[:, 0], edges.double(), sigma) for c in cpu_chains])
    (ref * side.cpu().double()).sum().backward()
    assert torch.isfinite(got).all() and torch.isfinite(xg.grad).all()
    assert float((got.detach().cpu().double() - ref.detach()).abs().max()) <= TOL * float(ref.abs().max())
    assert float((xg.grad.cpu().double() - xr.grad).abs().max()) <= TOL * float(xr.grad.abs().max())


# ---- mixed screens in one launch ---------------------------------------------------------------------------------
def test_mixed_screens_in_one_launch_through_simulate():
    """1-D screens with equal nbins share ONE launch (simulate._build_plan groups them by nbins) although their edges and
    bandwidths differ: the launch takes the template of the largest ratio and each screen reads its own geometry.
    Group of 64 bins: bandwidths 0.1 / 0.5 / 1.25 (an R = 13 launch), one screen along a direction; group of 48
    bins: 0.5 / 0.08 / 0.3 (an R = 4 launch holding a nearly hard screen)."""
    gen = torch.Generator().manual_seed(21)
    n, d = 6000, 4
    x = grid_x(n, d, gen)
    mats = [torch.round((torch.eye(d) + 0.3 * torch.randn(d, d, generator=gen)) * 16) / 16 for _ in range(3)]
    tfs = [mf.simulate.LinearTransform(m.cuda()) for m in mats]
    H = mf.diagnostics.Histogram1D
    group64 = [H(axis=0, edges=torch.linspace(-4.0, 4.0, 65), bandwidth=0.1),
               H(axis=1, edges=torch.linspace(-3.0, 5.0, 65), bandwidth=0.5),
               H(edges=torch.linspace(-2.0, 2.0, 65), bandwidth=1.25, direction=torch.tensor([1.0, 1.0, 0.0, 0.0]))]
    group48 = [H(axis=2, edges=torch.linspace(-3.0, 3.0, 49), bandwidth=0.5),
               H(axis=0, edges=torch.linspace(-1.5, 4.5, 49), bandwidth=0.08),
               H(axis=3, edges=torch.linspace(-6.0, 6.0, 49), bandwidth=0.3)]
    diags = [[a.to(DEV), b.to(DEV)] for a, b in zip(group64, group48)]

    xg = x.cuda().requires_grad_(True)
    sim._plan_cache.clear()
    out = mf.simulate.forward(xg, tfs, diags)
    plan = next(iter(sim._plan_cache.values()))
    assert not plan.fallback and list(plan.groups) == [("1d", True, 64), ("1d", True, 48)]
    assert template_radius(plan.groups[("1d", True, 64)].cache["ratio"]) == 13
    assert template_radius(plan.groups[("1d", True, 48)].cache["ratio"]) == 4
    sides = [[torch.randn(p.shape[0], generator=gen).cuda() for p in row] for row in out]
    sum((p * s).sum() for row, srow in zip(out, sides) for p, s in zip(row, srow)).backward()

    xd = x.to(DEV, torch.float64).requires_grad_(True)
    loss = 0.0
    for i, row in enumerate(diags):
        for j, diag in enumerate(row):
            what = f"transform {i}, screen {j}"
            u = xd @ diag.projection_vector(tfs[i].matrix, d, DEV).double()
            ref = hp.kde_profile_1d(u, diag.edges.double(), float(diag.bandwidth))
            loss = loss + (ref * sides[i][j].double()).sum()
            got = out[i][j]
            assert torch.isfinite(got).all(), f"{what}: non-finite profile"
            err = profile_err(got.detach()[None], ref.detach()[None])
            assert err < TOL, f"{what}: profile {err:.2e}"
            with torch.no_grad():
                alone = mf.simulate.forward(x.cuda(), [tfs[i]], [[diag]])[0][0]
            err = profile_err(got.detach()[None], alone[None])
            assert err < 1e-5, f"{what}: fused launch vs the screen alone {err:.2e}"
    loss.backward()
    assert torch.isfinite(xg.grad).all(), "non-finite dL/dx"
    err = rel_max(xg.grad, xd.grad)
    assert err < TOL, f"dL/dx {err:.2e} of max |grad|"


# ---- 2-D: both forward paths, per-axis bandwidths, backward at R = 4 and R = 9 -------------------------------------
@pytest.fixture(params=[True, False], ids=["tensor_cores", "fixed_point"])
def kde2d_path(request):
    """Run a test once per 2-D forward path (kde2d_tc.cu / kde2d.cu)."""
    old = ops.KDE2D_USE_TENSOR_CORES
    ops.KDE2D_USE_TENSOR_CORES = request.param
    yield request.param
    ops.KDE2D_USE_TENSOR_CORES = old


SCREEN_EDGES_2D = [(torch.linspace(-5.0, 5.0, 41), torch.linspace(-3.0, 3.0, 25)),
                   (torch.linspace(-2.5, 2.5, 41), torch.linspace(-1.0, 2.0, 25)),
                   (torch.linspace(-4.0, 6.0, 41), torch.linspace(-1.5, 1.5, 25))]


def geom_2d(screens, bandwidths):
    edges = [e for ex_ey in screens for e in ex_ey]
    geom, sigmas, ratio = geom_1d(edges, [b for pair in bandwidths for b in pair])
    return geom.reshape(len(screens), 2, -1), sigmas, ratio


def uses_tensor_cores(n, d, bx, by):
    flags = 0 if ops.KDE2D_USE_TENSOR_CORES else ops.FLAG_NO_TENSOR_CORES
    return bool(_lib.load().mfb_kde2d_uses_tensor_cores(n, d, bx, by, flags))


@pytest.mark.parametrize("bandwidths,radius", [([(0.05, 0.5), (0.2, 0.3)], 4),
                                               ([(0.05, 0.5), (0.3, 0.75), (1.0, 1.05)], 9)])
def test_kde2d_per_axis_bandwidths_both_paths_vs_float64(kde2d_path, bandwidths, radius):
    gen = torch.Generator().manual_seed(radius)
    n, d = 5000, 4
    k = len(bandwidths)
    screens = SCREEN_EDGES_2D[:k]
    bx, by = screens[0][0].numel() - 1, screens[0][1].numel() - 1
    geom, sigmas, ratio = geom_2d(screens, bandwidths)
    assert template_radius(ratio, dims=2) == radius
    x = grid_x(n, d, gen)
    w = torch.stack([grid_w(2, d, gen) for _ in range(k)])
    side = torch.randn(k, bx, by, generator=gen, dtype=torch.float64).to(DEV)

    xg = x.cuda().requires_grad_(True)
    prof = ops.project_kde2d(xg, w.cuda(), geom.cuda(), ratio, bx, by)
    (prof.double() * side).sum().backward()

    xd = x.to(DEV, torch.float64).requires_grad_(True)
    wd = w.to(DEV, torch.float64)
    ref = torch.stack([hp.kde_profile_2d(xd @ wd[i, 0], xd @ wd[i, 1], screens[i][0].to(DEV, torch.float64),
                                         screens[i][1].to(DEV, torch.float64), sigmas[2 * i], sigmas[2 * i + 1])
                       for i in range(k)])
    (ref * side).sum().backward()
    assert torch.isfinite(prof).all(), "non-finite profiles"
    err = profile_err(prof.detach(), ref.detach())
    assert err < TOL, f"profiles {err:.2e}"
    assert torch.isfinite(xg.grad).all(), "non-finite dL/dx"
    err = rel_max(xg.grad, xd.grad)
    assert err < TOL, f"dL/dx {err:.2e} of max |grad|"
    assert uses_tensor_cores(n, d, bx, by) == kde2d_path


# ---- functional interface (absolute bandwidths) ----------------------------------------------------------------
def test_kde_histogram_functional_interface_vs_float64():
    """``kde_histogram_1d / _2d(..., bandwidth=...)`` take absolute bandwidths; values and gradients w.r.t. x (and y)
    against the reference's dense form in float64."""
    gen = torch.Generator().manual_seed(3)
    bins = torch.linspace(-4.0, 4.0, 65)                         # bin width 1/8
    for n, bw in [(3001, 0.006), (3001, 0.05), (1, 0.05), (3001, 0.15)]:     # sigma / bin = 0.048, 0.4, 1.2
        x = grid_x(n, 1, gen)[:, 0]
        side = torch.randn(64, generator=gen, dtype=torch.float64).to(DEV)
        xg = x.cuda().requires_grad_(True)
        prof = kde_histogram_1d(xg, bins.cuda(), bandwidth=bw)
        (prof.double() * side).sum().backward()
        xd = x.to(DEV, torch.float64).requires_grad_(True)
        ref = hp.kde_profile_1d(xd, bins.to(DEV, torch.float64), float(torch.tensor(bw, dtype=torch.float32)))
        (ref * side).sum().backward()
        assert torch.isfinite(prof).all() and torch.isfinite(xg.grad).all(), (n, bw)
        assert profile_err(prof.detach()[None], ref.detach()[None]) < TOL, (n, bw)
        assert rel_max(xg.grad, xd.grad) < TOL, (n, bw)

    bx_edges, by_edges = torch.linspace(-5.0, 5.0, 41), torch.linspace(-3.0, 3.0, 25)    # widths 1/4, 1/4
    for n, bws in [(3001, (0.015, 0.1)), (5000, (0.015, 0.1)), (5000, (0.25, 0.2))]:     # fixed point; tensor cores
        xy = grid_x(n, 2, gen)
        side = torch.randn(40, 24, generator=gen, dtype=torch.float64).to(DEV)
        xg, yg = xy[:, 0].cuda().requires_grad_(True), xy[:, 1].cuda().requires_grad_(True)
        prof = kde_histogram_2d(xg, yg, [bx_edges.cuda(), by_edges.cuda()], bandwidth=bws)
        (prof.double() * side).sum().backward()
        xd, yd = (xy[:, i].to(DEV, torch.float64).requires_grad_(True) for i in range(2))
        sx, sy = (float(torch.tensor(b, dtype=torch.float32)) for b in bws)
        ref = hp.kde_profile_2d(xd, yd, bx_edges.to(DEV, torch.float64), by_edges.to(DEV, torch.float64), sx, sy)
        (ref * side).sum().backward()
        assert torch.isfinite(prof).all() and torch.isfinite(xg.grad).all() and torch.isfinite(yg.grad).all(), (n, bws)
        assert profile_err(prof.detach()[None], ref.detach()[None]) < TOL, (n, bws)
        assert rel_max(xg.grad, xd.grad) < TOL and rel_max(yg.grad, yd.grad) < TOL, (n, bws)


# ---- the supported range is explicit ----------------------------------------------------------------------------
def test_bandwidth_beyond_the_compiled_windows_is_refused_before_launch():
    gen = torch.Generator().manual_seed(4)
    x = grid_x(5000, 4, gen).cuda()
    # the reference's default absolute bandwidth (1.0) on typical bins is sigma = 9 bins
    with pytest.raises(ValueError, match="bandwidth too wide"):
        kde_histogram_1d(x[:, 0].contiguous(), torch.linspace(-3.5, 3.5, 65).cuda())
    edges = [torch.linspace(-4.0, 4.0, 65)] * 3
    w = grid_w(3, 4, gen).cuda()
    geom, _, ratio = geom_1d(edges, [1.52] * 3)
    ops.kde1d_sums(x, w, geom.cuda(), ratio, 64)                  # the top of the widest template still runs
    geom, _, ratio = geom_1d(edges, [0.5, 1.53, 0.5])
    with pytest.raises(ValueError, match="1.5254"):
        ops.kde1d_sums(x, w, geom.cuda(), ratio, 64)
    with pytest.raises(ValueError, match="bandwidth too wide"):
        ops.project_kde1d(x.clone().requires_grad_(True), w, geom.cuda(), ratio, 64)
    diag = mf.diagnostics.Histogram1D(axis=0, edges=edges[0], bandwidth=1.6).to(DEV)
    with pytest.raises(ValueError, match="bandwidth too wide"):
        mf.simulate.forward(x, [mf.simulate.LinearTransform(torch.eye(4, device=DEV))], [[diag]])
    # the private bins of the 1-D deposit fill shared memory at about 1800 bins: wider screens are refused
    geom, _, ratio = geom_1d([torch.linspace(-4.0, 4.0, 8193)] * 3, [0.5] * 3)
    with pytest.raises(RuntimeError, match="not supported"):
        ops.kde1d_sums(x, w, geom.cuda(), ratio, 8192)
    with pytest.raises(RuntimeError, match="not supported"):
        ops.project_kde1d(x.clone().requires_grad_(True), w, geom.cuda(), ratio, 8192)

    # 2-D: the tensor-core forward takes any width, the fixed-point deposit and the backward stop at R = 9
    screens = SCREEN_EDGES_2D[:2]
    geom2, sigmas, ratio2 = geom_2d(screens, [(0.5, 0.5), (1.2, 0.3)])
    w2 = torch.stack([grid_w(2, 4, gen) for _ in range(2)]).cuda()
    old = ops.KDE2D_USE_TENSOR_CORES
    try:
        ops.KDE2D_USE_TENSOR_CORES = True
        assert uses_tensor_cores(x.shape[0], 4, 40, 24)
        prof = ops.project_kde2d(x, w2, geom2.cuda(), ratio2, 40, 24)
        xd, wd = x.double(), w2.double()
        ref = torch.stack([hp.kde_profile_2d(xd @ wd[i, 0], xd @ wd[i, 1], screens[i][0].to(DEV, torch.float64),
                                             screens[i][1].to(DEV, torch.float64), sigmas[2 * i], sigmas[2 * i + 1])
                           for i in range(2)])
        assert profile_err(prof, ref) < TOL
        with pytest.raises(ValueError, match="1.0734"):
            ops.project_kde2d(x.clone().requires_grad_(True), w2, geom2.cuda(), ratio2, 40, 24)
        with pytest.raises(ValueError, match="bandwidth too wide"):
            ops.project_kde2d(x[:4095].contiguous(), w2, geom2.cuda(), ratio2, 40, 24)   # below the tensor-core batch
        ops.KDE2D_USE_TENSOR_CORES = False
        with pytest.raises(ValueError, match="1.0734"):
            ops.project_kde2d(x, w2, geom2.cuda(), ratio2, 40, 24)
    finally:
        ops.KDE2D_USE_TENSOR_CORES = old
    with pytest.raises(ValueError, match="bandwidth too wide"):
        kde_histogram_2d(x[:, 0].contiguous().requires_grad_(True), x[:, 1].contiguous(),
                         [screens[0][0].cuda(), screens[0][1].cuda()], bandwidth=(0.3, 0.3))
    torch.cuda.synchronize()              # no sticky error left behind
    assert float(torch.ones(1, device=DEV).sum()) == 1.0
