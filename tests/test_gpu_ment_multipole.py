"""GPU parity: classical MENT through thin multipole kicks (experiments/rec_2d/nonlinear and random chains
linear* -> MultipoleTransform -> linear*) against a float64 evaluation built from the package's transform classes:
rho(x) = prior(x) * prod clamp(h(project(transform.forward(x)))), integrate mode through transform.inverse."""
import itertools

import numpy as np
import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200.simulate.transform import CompositeTransform, LinearTransform, MultipoleTransform
from mfb_testutil import (check_density as _check_density, integrate_check as _integrate_check, oracle_prob,
                          positive_tables as _positive_tables, t32)

pytestmark = pytest.mark.gpu


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
