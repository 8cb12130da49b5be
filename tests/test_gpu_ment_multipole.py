"""GPU parity: classical MENT through thin multipole kicks (experiments/rec_2d/nonlinear and random chains
linear* -> MultipoleTransform -> linear*) against a float64 evaluation built from the package's transform classes:
rho(x) = prior(x) * prod clamp(h(project(transform.forward(x)))), integrate mode through transform.inverse."""
import itertools

import numpy as np
import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200.simulate.transform import CompositeTransform, LinearTransform, MultipoleTransform
from mfb_testutil import t32
from oracle import hotpath as hp

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------- float64 oracle
def _cpu64(t):
    """float64 CPU copy of a transfer map."""
    if isinstance(t, LinearTransform):
        return LinearTransform(t.matrix.detach().to("cpu", torch.float64))
    if isinstance(t, CompositeTransform):
        return CompositeTransform(*[_cpu64(s) for s in t.transforms])
    return MultipoleTransform(order=t.order, strength=t.strength, skew=t.skew)


def _h(diag, table, u):
    """Lagrange function of ``diag`` at the transformed points u (float64), as the reference's interpolator."""
    if isinstance(diag, mf.diagnostics.Histogram2D):
        cx, cy = (hp.centres(e.cpu()) for e in (diag.edges_x, diag.edges_y))
        return hp.lagrange_interp_2d(table.cpu(), cx, cy, u[:, list(diag.axis)])
    return hp.lagrange_interp(table.cpu(), hp.centres(diag.edges.cpu()), u[:, diag.axis])


def oracle_prob(model, x):
    """hp.ment_prob with transform.forward in float64 in place of the matrix."""
    x = x.detach().cpu().double()
    prob = torch.ones(x.shape[0], dtype=torch.float32)
    for i, t in enumerate(model.transforms):
        u = _cpu64(t)(x)
        for j, diag in enumerate(model.diagnostics[i]):
            h = _h(diag, model.lagrange_functions[i][j].values, u)
            prob = prob * torch.clamp(h.type(torch.float32), 0.0, 1.0e10)
    return prob * torch.exp(hp.gaussian_log_prob(x, float(model.prior.scale)).float())


def oracle_integrate(model, i, j):
    """Normalised integrate-mode prediction: sum over the integration grid of rho(transform.inverse(points))."""
    diag = model.diagnostics[i][j]
    limits, shape = model.integration_limits[i][j], model.integration_shape[i][j]
    grid = [torch.linspace(float(lo), float(hi), int(n), dtype=torch.float64) for (lo, hi), n in zip(limits, shape)]
    if isinstance(diag, mf.diagnostics.Histogram2D):
        meas = [hp.centres(diag.edges_x.cpu()).double(), hp.centres(diag.edges_y.cpu()).double()]
        axes = list(diag.axis)
    else:
        meas = [hp.centres(diag.edges.cpu()).double()]
        axes = [diag.axis]
    d = model.ndim
    others = [a for a in range(d) if a not in axes]
    mesh = torch.meshgrid(*meas, *grid, indexing="ij")
    u = torch.zeros(mesh[0].numel(), d, dtype=torch.float64)
    for a, m in zip(axes + others, mesh):
        u[:, a] = m.reshape(-1)
    x = _cpu64(model.transforms[i]).inverse(u)
    rho = oracle_prob(model, x).double().reshape(*[m.numel() for m in meas], -1).sum(dim=-1)
    if isinstance(diag, mf.diagnostics.Histogram2D):
        vol = float(diag.edges_x[1] - diag.edges_x[0]) * float(diag.edges_y[1] - diag.edges_y[0])
    else:
        vol = float(diag.edges[1] - diag.edges[0])
    return (rho / rho.sum() / vol).float()


def oracle_sweeps(model, n, lr=1.0, thresh=1.0e-10):
    """``n`` Gauss-Seidel sweeps of integrate mode on the oracle (model's tables are read, not changed)."""
    saved = [[lf.values.clone() for lf in row] for row in model.lagrange_functions]
    out = None
    try:
        for _ in range(n):
            for i in range(len(model.transforms)):
                for j in range(len(model.diagnostics[i])):
                    pred = oracle_integrate(model, i, j)
                    lf = model.lagrange_functions[i][j]
                    meas = model.measurements[i][j].cpu()
                    new = hp.gauss_seidel_table(lf.values.cpu(), meas, pred, lr, thresh)
                    lf.set_values(new.to(lf.values.device))
        out = [[lf.values.cpu().clone() for lf in row] for row in model.lagrange_functions]
    finally:
        for row, vals in zip(model.lagrange_functions, saved):
            for lf, v in zip(row, vals):
                lf.set_values(v)
    return out


def _positive_tables(model, seed):
    """Positive random tables, zero on the outermost centres so that h is continuous (a point whose fp32 and float64
    projections straddle the last centre would otherwise see a jump)."""
    gen = torch.Generator().manual_seed(seed)
    for row in model.lagrange_functions:
        for lf in row:
            v = torch.rand(lf.values.shape, generator=gen) + 0.2
            if v.ndim == 1:
                v[0] = v[-1] = 0.0
            else:
                v[0], v[-1], v[:, 0], v[:, -1] = 0.0, 0.0, 0.0, 0.0
            lf.set_values(v.cuda())


def _check_density(model, x, want_x):
    """prob at explicit points, prob_on_grid and prob at the materialised grid points against the float64 oracle.
    The kernels project in fp32: where a factor sits near the zero end of its table its relative error is that of
    the projection over the distance to the end (a fp32 emulation of the kernels' arithmetic reaches 7e-7 of the
    maximum there), hence an absolute tolerance of 2e-6 of the maximum at the explicit points as on the grid."""
    prob = model.prob(x.cuda()).cpu()
    assert int((want_x > 0).sum()) > 0.2 * want_x.numel()               # not vacuous
    assert torch.allclose(prob, want_x, rtol=1e-4, atol=2e-6 * float(want_x.max()))
    grid = model.prob_on_grid(model.sampler).cpu()
    pts = model.sampler.get_grid_points()
    refg = oracle_prob(model, pts)
    assert int((refg > 0).sum()) > 0.05 * refg.numel()
    # grid points come from the index (lo + i*step) instead of fp32 linspace centres: 1-ulp shifts
    assert torch.allclose(grid, refg, rtol=1e-4, atol=2e-6 * float(refg.max()))
    assert torch.allclose(model.prob(pts).cpu(), refg, rtol=1e-4, atol=2e-6 * float(refg.max()))


# ---------------------------------------------------------------------------------------------- rec_2d/nonlinear
def _nonlinear(golden, mode="sample", res=128, n_samples=100_000, int_points=250):
    g = golden("multipole")
    matrix = t32(g["nl_matrix"]).cuda()
    tfs = [CompositeTransform(MultipoleTransform(order=int(g["nl_order"]), strength=float(st)), LinearTransform(matrix))
           for st in g["nl_strengths"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=t32(g["nl_edges"]), bandwidth=0.5).to("cuda")
    kw = {}
    if mode == "sample":
        kw["sampler"] = mf.sample.GridSampler(limits=2 * [(-4.0, 4.0)], shape=(res, res), device="cuda")
        kw["n_samples"] = n_samples
    else:
        kw["integration_limits"] = [[[(-4.0, 4.0)]] for _ in tfs]
        kw["integration_shape"] = [[(int_points,)] for _ in tfs]
    return mf.ment.MENT(ndim=2, transforms=tfs, diagnostics=[[diag] for _ in tfs],
                        measurements=[[m.cuda()] for m in t32(g["nl_meas"])],
                        prior=mf.prior.Gaussian(ndim=2, scale=1.5), mode=mode, device="cuda", **kw)


def test_nonlinear_setup_density_matches_float64(golden):
    model = _nonlinear(golden)
    _positive_tables(model, 1)
    x = torch.randn(20000, 2, generator=torch.Generator().manual_seed(2)) * 1.3
    _check_density(model, x, oracle_prob(model, x))


# ---------------------------------------------------------------------------------------------- random chains
def _orth(d, gen, scale=1.0):
    q, _ = torch.linalg.qr(torch.randn(d, d, generator=gen))
    return (q * scale).float()


def _random_model(d, flip, mode="sample", seed=0):
    """Kicks of every order, normal and skew (``flip`` swaps them), with and without pre / post, next to plain linear
    maps; 1-D and 2-D screens, one transform with both."""
    gen = torch.Generator().manual_seed(seed + 10 * d + int(flip))
    lin = lambda: LinearTransform(_orth(d, gen).cuda())                      # noqa: E731
    kick = lambda order, skew, s: MultipoleTransform(order=order, strength=s, skew=skew != flip)   # noqa: E731
    tfs = [CompositeTransform(lin(), kick(3, False, 0.4), lin()),
           CompositeTransform(lin(), kick(4, True, 0.3), lin()),
           lin(),
           CompositeTransform(kick(5, False, 0.2), lin()),
           CompositeTransform(lin(), lin()),
           CompositeTransform(lin(), kick(3, True, 0.4))]
    e1 = torch.linspace(-4.0, 4.0, 33)
    ex, ey = torch.linspace(-4.0, 4.0, 17), torch.linspace(-3.5, 3.5, 15)
    s1 = lambda axis: mf.diagnostics.Histogram1D(axis=axis, edges=e1, bandwidth=0.5).to("cuda")        # noqa: E731
    s2 = lambda: mf.diagnostics.Histogram2D(axis=(0, 2), edges=(ex, ey), bandwidth=(0.5, 0.5)).to("cuda")  # noqa: E731
    diags = [[s1(0)], [s1(1), s2()], [s1(0)], [s2()], [s2()], [s1(2)]]
    meas = [[torch.ones(32).cuda() if isinstance(dg, mf.diagnostics.Histogram1D) else torch.ones(16, 14).cuda()
             for dg in row] for row in diags]
    kw = {}
    if mode == "sample":
        res = 16 if d == 4 else 8
        kw["sampler"] = mf.sample.GridSampler(limits=d * [(-3.0, 3.0)], shape=tuple(d * [res]), device="cuda")
    else:
        kw["integration_limits"] = [[[(-3.5, 3.5)] * (d - (2 if isinstance(dg, mf.diagnostics.Histogram2D) else 1))
                                     for dg in row] for row in diags]
        kw["integration_shape"] = [[(8,) * (d - (2 if isinstance(dg, mf.diagnostics.Histogram2D) else 1))
                                    for dg in row] for row in diags]
    return mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                        prior=mf.prior.Gaussian(ndim=d, scale=1.2), mode=mode, device="cuda", **kw)


@pytest.mark.parametrize("d,flip", list(itertools.product([4, 6], [False, True])))
def test_random_chains_density_matches_float64(d, flip):
    model = _random_model(d, flip)
    _positive_tables(model, 3 + d)
    x = torch.randn(20000, d, generator=torch.Generator().manual_seed(d)) * 0.9
    _check_density(model, x, oracle_prob(model, x))


# ---------------------------------------------------------------------------------------------- integrate mode
def _integrate_check(model, slots):
    """simulate(i, j) against the oracle, then two Gauss-Seidel sweeps against the oracle's sweeps.  A screen's own
    pixels sit exactly on its bin centres: where the table is 0 next to a nonzero value, fp32 rounding of the pixel's
    own projection (a few 1e-7) turns h = 0 into slope x rounding, up to ~1e-5 of the maximum prediction.  Such entries
    stay 0 through the update (0 x anything), so the tables keep the tight tolerances."""
    for i, j in slots:
        pred = model.simulate(i, j).cpu()
        want = oracle_integrate(model, i, j)
        assert pred.shape == want.shape and int((want > 0).sum()) > 5
        assert torch.allclose(pred, want, rtol=1e-4, atol=1e-5 * float(want.max())), (i, j)
    want = oracle_sweeps(model, 2)
    model.gauss_seidel_update(lr=1.0, thresh=1.0e-10)
    model.gauss_seidel_step(lr=1.0, thresh=1.0e-10)
    for row_g, row_w in zip(model.lagrange_functions, want):
        for lf, w in zip(row_g, row_w):
            got = lf.values.cpu()
            assert torch.allclose(got, w, rtol=2e-4, atol=1e-6)
            assert torch.equal(got == 0, w == 0)


def test_integrate_mode_nonlinear_setup_matches_float64(golden):
    """Tables zero on the outermost centres: a screen's own pixels sit exactly on its centres, and T(T^-1(c)) lands a
    rounding error above or below the last centre, where a nonzero end value would make h jump to 0."""
    model = _nonlinear(golden, mode="integrate", int_points=250)
    _positive_tables(model, 8)
    _integrate_check(model, [(0, 0), (3, 0), (5, 0)])


def test_integrate_mode_2d_screen_behind_a_kick_matches_float64():
    model = _random_model(4, False, mode="integrate")
    # keep the oracle affordable: the 2-D screens behind kicks (1, 3), a 1-D one behind a kick and a linear one
    keep = [1, 3, 2]
    model.transforms = [model.transforms[i] for i in keep]
    model.diagnostics = [model.diagnostics[i] for i in keep]
    model.measurements = [model.measurements[i] for i in keep]
    model.integration_limits = [model.integration_limits[i] for i in keep]
    model.integration_shape = [model.integration_shape[i] for i in keep]
    model.initialize_lagrange_functions()
    _positive_tables(model, 9)
    _integrate_check(model, [(0, 1), (1, 0), (0, 0), (2, 0)])


def test_integrate_mode_composite_of_linear_maps_equals_product():
    gen = torch.Generator().manual_seed(21)
    a, b = _orth(4, gen, 1.1).cuda(), _orth(4, gen, 0.9).cuda()
    e = torch.linspace(-4.0, 4.0, 33)

    def build(tf):
        diag = mf.diagnostics.Histogram1D(axis=0, edges=e, bandwidth=0.5).to("cuda")
        diag2 = mf.diagnostics.Histogram2D(axis=(1, 3), edges=(e[::2], e[::2]), bandwidth=(0.5, 0.5)).to("cuda")
        m = mf.ment.MENT(ndim=4, transforms=[tf, LinearTransform(_orth(4, torch.Generator().manual_seed(5)).cuda())],
                         diagnostics=[[diag, diag2], [diag]],
                         measurements=[[torch.ones(32).cuda(), torch.ones(16, 16).cuda()], [torch.ones(32).cuda()]],
                         prior=mf.prior.Gaussian(ndim=4, scale=1.0), mode="integrate",
                         integration_limits=[[[(-3.0, 3.0)] * 3, [(-3.0, 3.0)] * 2], [[(-3.0, 3.0)] * 3]],
                         integration_shape=[[(10, 10, 10), (12, 12)], [(10, 10, 10)]], device="cuda")
        _positive_tables(m, 4)
        return m

    comp = build(CompositeTransform(LinearTransform(a), LinearTransform(b)))
    prod = build(LinearTransform(b @ a))
    for j in range(2):
        p, q = comp.simulate(0, j), prod.simulate(0, j)
        assert torch.isfinite(p).all() and float(p.max()) > 0
        assert torch.allclose(p, q, rtol=1e-6, atol=1e-9 * float(q.max()))


# ---------------------------------------------------------------------------------------------- sample mode
def test_sample_mode_sweep_nonlinear_setup_is_consistent_and_converges(golden):
    """One sample-mode sweep (grid density -> particles -> fused 1-D KDE behind the kick) agrees with the integrate-mode
    sweep of the same model, and three sweeps lower the mean KL against the measurements.  On the float64 oracle the
    sample-mode expectation (KDE of the grid density) differs from the integrate-mode sweep by a median of 1.1 % on the
    solid bins, and the mean KL of either mode falls at every sweep (0.0094 -> 0.0034 -> 0.0013 -> 0.0008 for the
    KDE): sampling noise of 2M particles, ~85 / 4e6 in KL, is far below those steps."""
    torch.manual_seed(0)
    model = _nonlinear(golden, mode="sample", res=256, n_samples=2_000_000)

    def mean_kl():
        pred = model.simulate_all()
        return float(np.mean([float(mf.loss.kl_divergence(p[0], m[0])) for p, m in zip(pred, model.measurements)]))

    kls = [mean_kl()]
    model.gauss_seidel_update(lr=1.0, thresh=1.0e-10)
    ref = _nonlinear(golden, mode="integrate", int_points=250)
    ref.gauss_seidel_update(lr=1.0, thresh=1.0e-10)
    got = torch.stack([row[0].values.cpu() for row in model.lagrange_functions])
    want = torch.stack([row[0].values.cpu() for row in ref.lagrange_functions])
    meas = t32(golden("multipole")["nl_meas"])
    solid = meas > 0.02 * meas.max(dim=1, keepdim=True).values
    rel = ((got - want).abs() / want.abs().clamp_min(1e-12))[solid]
    assert float(rel.median()) < 0.02 and float(rel.max()) < 0.25
    assert torch.equal(got == 0, want == 0)
    kls.append(mean_kl())
    for _ in range(2):
        model.gauss_seidel_update(lr=1.0, thresh=1.0e-10)
        kls.append(mean_kl())
    assert all(b <= a for a, b in zip(kls, kls[1:])), kls
    assert model.epoch == 3


def test_sharded_draws_of_a_kicked_model_are_slices_of_one_stream(golden):
    """MENT.shard needs nothing new behind kicks: the density is replicated, rank r draws its slice of one stream."""
    model = _nonlinear(golden, n_samples=100_003)
    _positive_tables(model, 6)
    torch.manual_seed(17)
    full = model.sample(100_003)
    parts = []
    for r in range(3):
        model.shard = (r, 3)
        torch.manual_seed(17)
        parts.append(model.sample(100_003))
    model.shard = None
    assert torch.equal(torch.cat(parts), full)
