"""GPU parity: classical MENT with linear transfer maps (the kernels without multipole terms) against float64.

- density (prob at points, prob_on_grid, prob at the materialised grid points) for every compiled D, against the
  float64 oracle of mfb_testutil: random well-conditioned maps, 1-D screens on any axis, 2-D screens on any ordered
  axis pair, B from 2 to 64, Gaussian and flat priors, tables with zero runs, negative entries and entries above the
  1e10 clamp;
- the interpolation exactly at the table edges (unit projection rows: the fp32 projection is exact) on non-uniform
  centres, against scipy's rule: closed interval, zero outside;
- the 200 KB shared-memory limit: the largest K that fits runs and is right, one more is refused before any launch;
- integrate mode and two Gauss-Seidel sweeps for D = 2 ... 8, ragged integration grids, composite maps;
- the CDF build and the sampler draw by draw: the CDF against a compensated float64 prefix, monotone, its last entry
  the total; every draw's cell against a bisection of that CDF with the kernel's Philox stream replayed in numpy, its
  coordinates against an fp32 emulation;
- the Gauss-Seidel rule at its edges."""
import math

import numpy as np
import pytest
import torch
from scipy.interpolate import RegularGridInterpolator

import mentflow_b200 as mf
from mentflow_b200 import _lib, ops
from mentflow_b200.simulate.transform import CompositeTransform, LinearTransform
from mfb_testutil import (check_density, fmaf, integrate_check, oracle_integrate, oracle_prob, positive_tables,
                          sampler_uniforms, u01)
from oracle import hotpath as hp

pytestmark = pytest.mark.gpu


def _matrix(d, gen):
    """Well-conditioned: Q1 diag(s) Q2 with s in [0.75, 1.3]."""
    q1, _ = torch.linalg.qr(torch.randn(d, d, generator=gen, dtype=torch.float64))
    q2, _ = torch.linalg.qr(torch.randn(d, d, generator=gen, dtype=torch.float64))
    s = 0.75 + 0.55 * torch.rand(d, generator=gen, dtype=torch.float64)
    return ((q1 * s) @ q2).float()


def _s1(axis, b, lim=4.0):
    return mf.diagnostics.Histogram1D(axis=axis, edges=torch.linspace(-lim, lim, b + 1), bandwidth=0.5).to("cuda")


def _s2(axes, bx=9, by=6):
    ex, ey = torch.linspace(-4.0, 4.0, bx + 1), torch.linspace(-3.5, 3.5, by + 1)
    return mf.diagnostics.Histogram2D(axis=axes, edges=(ex, ey), bandwidth=(0.5, 0.5)).to("cuda")


def _pairs(d):
    return [(0, 1)] + ([(2, 0), (d - 1, 1)] if d >= 3 else [])


def _prior(kind, d):
    if kind == "uniform":
        return mf.prior.Uniform(ndim=d, scale=10.0)
    return mf.prior.Gaussian(ndim=d, scale={"gauss0.7": 0.7, "gauss3": 3.0}[kind])


def _tables(model, seed):
    """positive_tables, except that 1-D tables of fewer than 4 centres keep their ends (they would be all zero)."""
    positive_tables(model, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    for row in model.lagrange_functions:
        for lf in row:
            if lf.values.ndim == 1 and lf.values.numel() < 4:
                lf.set_values((torch.rand(lf.values.shape, generator=gen) + 0.2).cuda())


def _model(d, b, prior, seed, shape, only2d=False):
    """One transform per 2-D axis pair (`_pairs`) plus one more, each with a 1-D screen on a random axis (the last on
    axis D - 1) unless ``only2d``; the 2-D screens sit on the pair transforms.  Sampler grid of ``shape`` cells."""
    gen = torch.Generator().manual_seed(seed)
    pairs = _pairs(d)
    n = len(pairs) + 1
    axes = [int(a) for a in torch.randint(0, d, (n - 1,), generator=gen)] + [d - 1]
    tfs = [LinearTransform(_matrix(d, gen).cuda()) for _ in range(n)]
    diags = []
    for i in range(n):
        row = [] if only2d else [_s1(axes[i], b)]
        if i < len(pairs):
            row.append(_s2(pairs[i]))
        diags.append(row)
    if only2d:
        tfs, diags = tfs[:-1], diags[:-1]
    meas = [[torch.ones(b).cuda() if isinstance(dg, mf.diagnostics.Histogram1D) else torch.ones(9, 6).cuda()
             for dg in row] for row in diags]
    lim = 3.0 if d <= 4 else 2.0
    sampler = mf.sample.GridSampler(limits=d * [(-lim, lim)], shape=shape, device="cuda")
    return mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas, prior=_prior(prior, d),
                        mode="sample", sampler=sampler, device="cuda")


def _extreme_tables(model, seed):
    """_tables, then one 1-D table (B >= 8) with an interior zero run, a negative entry and an entry above the
    clamp of 1e10 (ment.py:246), scaled so that the clamp matters but leaves the other points' factors within 10x."""
    _tables(model, seed)
    lf = next((lf for row in model.lagrange_functions for lf in row if lf.values.ndim == 1), None)
    if lf is None or lf.values.numel() < 8:
        return False
    v = lf.values.cpu().clone()
    b = v.numel()
    v[b // 4:b // 4 + 3] = 0.0
    v[b // 2 - 1] = -0.7
    v *= 3.0e9
    v[b // 2 + 1] = 5.0e10
    lf.set_values(v.cuda())
    return True


_SHAPE = (3, 5, 7, 2, 4, 3, 5, 2)
_CASES = [(2, 2, "gauss0.7"), (3, 3, "gauss3"), (4, 33, "uniform"), (5, 64, "gauss0.7"), (6, 2, "gauss3"),
          (7, 3, "uniform"), (8, 33, "gauss0.7")]


@pytest.mark.parametrize("d,b,prior", _CASES)
def test_density_every_dimension_matches_float64(d, b, prior):
    model = _model(d, b, prior, d, _SHAPE[:d])
    extreme = _extreme_tables(model, 30 + d)
    x = torch.randn(20000, d, generator=torch.Generator().manual_seed(d)) * 0.9
    want = oracle_prob(model, x)
    if extreme:   # the clamp is reached and the zero run / negative entry zero some points
        vals = next(lf.values for row in model.lagrange_functions for lf in row if lf.values.ndim == 1)
        assert float(vals.max()) > 1e10 and float(vals.min()) < 0
    check_density(model, x, want)


@pytest.mark.parametrize("d,prior", [(3, "gauss3"), (5, "uniform"), (8, "gauss0.7")])
def test_density_only_2d_screens_matches_float64(d, prior):
    model = _model(d, 2, prior, 40 + d, _SHAPE[:d], only2d=True)
    assert model._groups(torch.device("cuda"))[0] is None      # no 1-D family: k = 0
    _tables(model, 50 + d)
    x = torch.randn(20000, d, generator=torch.Generator().manual_seed(60 + d)) * 0.9
    check_density(model, x, oracle_prob(model, x))


def test_density_1d_through_ment_prob():
    """D = 1 (no MENT model in one dimension on the reference's path): K tables on scaled projections."""
    gen = torch.Generator().manual_seed(7)
    k, b = 3, 33
    proj = torch.tensor([[1.0], [-0.8], [1.3]])
    coords = torch.stack([hp.centres(torch.linspace(-4.0, 4.0, b + 1))] * k)
    tables = torch.rand(k, b, generator=gen) + 0.2
    tables[:, 0] = tables[:, -1] = 0.0
    x = torch.randn(50000, 1, generator=gen) * 1.5
    s = 1.3
    got = ops.ment_prob(x.cuda(), (proj.cuda(), coords.cuda(), tables.cuda()), None, -0.5 / s ** 2,
                        -(math.log(s) + 0.5 * math.log(2 * math.pi))).cpu()
    want = torch.ones(x.shape[0])
    for i in range(k):
        h = hp.lagrange_interp(tables[i], coords[i], x[:, 0].double() * float(proj[i, 0]))
        want = want * torch.clamp(h.float(), 0.0, 1.0e10)
    want = want * torch.exp(hp.gaussian_log_prob(x.double(), s).float())
    assert int((want > 0).sum()) > 0.5 * want.numel()
    assert torch.allclose(got, want, rtol=1e-4, atol=2e-6 * float(want.max()))


# ---------------------------------------------------------------------------------------------- table edges
def _geometric(n, lo, hi, ratio):
    steps = ratio ** np.arange(n - 1)
    return (lo + np.concatenate([[0.0], np.cumsum(steps)]) * ((hi - lo) / steps.sum())).astype(np.float32)


def _specials(c):
    """Every centre, one fp32 ulp inside and outside both ends, interval midpoints."""
    inf = np.float32(np.inf)
    ends = [np.nextafter(c[0], -inf), np.nextafter(c[0], inf), np.nextafter(c[-1], -inf), np.nextafter(c[-1], inf)]
    return np.concatenate([c, np.array(ends, np.float32), (0.5 * (c[:-1] + c[1:])).astype(np.float32)])


def _scipy(c, t, u):
    grid = tuple(np.asarray(ci, np.float64) for ci in c)
    f = RegularGridInterpolator(grid, np.asarray(t, np.float64), method="linear", bounds_error=False, fill_value=0.0)
    return f(np.asarray(u, np.float64).reshape(-1, len(c))).astype(np.float32)


def test_table_edges_1d_exactly_on_non_uniform_centres():
    """Unit projection rows (axes 2, 0, 1): u is x's coordinate exactly.  Points put each table in turn on its centres,
    one ulp inside / outside its ends and its midpoints while the other coordinates sit inside their tables."""
    rng = np.random.default_rng(3)
    d, b = 3, 24
    axes = [2, 0, 1]
    coords = np.stack([_geometric(b, -3.0, 2.5, 1.25), _geometric(b, -2.0, 3.5, 0.8), _geometric(b, -4.0, 4.0, 1.1)])
    tables = (rng.random((3, b)) + 0.2).astype(np.float32)
    proj = np.eye(d, dtype=np.float32)[axes]
    safe = np.zeros(d, np.float32)
    for k, a in enumerate(axes):
        safe[a] = 0.5 * (coords[k][b // 2] + coords[k][b // 2 + 1])
    pts = []
    for k, a in enumerate(axes):
        sp = _specials(coords[k])
        p = np.tile(safe, (sp.size, 1))
        p[:, a] = sp
        pts.append(p)
    x = np.concatenate(pts)
    got = ops.ment_prob(torch.from_numpy(x).cuda(), tuple(torch.from_numpy(t).cuda() for t in (proj, coords, tables)),
                        None, 0.0, 0.0).cpu().numpy()
    want = np.ones(x.shape[0], np.float32)
    for k, a in enumerate(axes):
        want = want * np.clip(_scipy([coords[k]], tables[k], x[:, a]), 0.0, 1.0e10)
    n_out = 2 * len(axes)                               # one ulp outside either end, per table
    assert np.count_nonzero(want == 0) == n_out and np.count_nonzero(got == 0) == n_out
    assert np.allclose(got, want, rtol=1e-6, atol=0.0)


def test_table_edges_2d_exactly_on_non_uniform_centres():
    """Two 2-D tables on the axis pairs (2, 0) and (1, 3) with Bx != By; each in turn on the product of its special
    points while the other sits inside."""
    rng = np.random.default_rng(4)
    d, bx, by = 4, 11, 7
    pairs = [(2, 0), (1, 3)]
    cx = np.stack([_geometric(bx, -3.0, 2.5, 1.3), _geometric(bx, -2.5, 3.0, 0.85)])
    cy = np.stack([_geometric(by, -3.5, 3.0, 0.75), _geometric(by, -1.5, 2.0, 1.4)])
    tab = (rng.random((2, bx, by)) + 0.2).astype(np.float32)
    eye = np.eye(d, dtype=np.float32)
    proj2 = np.stack([eye[list(p)] for p in pairs])
    safe = np.zeros(d, np.float32)
    for k, (ax, ay) in enumerate(pairs):
        safe[ax] = 0.5 * (cx[k][bx // 2] + cx[k][bx // 2 + 1])
        safe[ay] = 0.5 * (cy[k][by // 2] + cy[k][by // 2 + 1])
    pts = []
    for k, (ax, ay) in enumerate(pairs):
        gx, gy = np.meshgrid(_specials(cx[k]), _specials(cy[k]), indexing="ij")
        p = np.tile(safe, (gx.size, 1))
        p[:, ax], p[:, ay] = gx.reshape(-1), gy.reshape(-1)
        pts.append(p)
    x = np.concatenate(pts)
    g2 = tuple(torch.from_numpy(t).cuda() for t in (proj2, cx, cy, tab))
    got = ops.ment_prob(torch.from_numpy(x).cuda(), None, g2, 0.0, 0.0).cpu().numpy()
    want = np.ones(x.shape[0], np.float32)
    for k, (ax, ay) in enumerate(pairs):
        want = want * np.clip(_scipy([cx[k], cy[k]], tab[k], x[:, [ax, ay]]), 0.0, 1.0e10)
    assert 0.3 * want.size < np.count_nonzero(want) < want.size     # the edges are crossed
    assert np.array_equal(got == 0, want == 0)
    assert np.allclose(got, want, rtol=1e-6, atol=0.0)


# ---------------------------------------------------------------------------------------------- shared-memory limit
def _ment_smem(k, b, d):
    """ment.cu ment_smem: projections (padded to 4), centres, values, 1 / spacing (padded to 2) in fp32, and the
    double table of 1 / spacing."""
    return ((((k * d + 3) & ~3) + 2 * k * b + ((k + 1) & ~1)) * 4 + k * b * 8 + 16)


def _smem_tables(k, d, b, seed):
    gen = torch.Generator().manual_seed(seed)
    proj = torch.randn(k, d, generator=gen)
    proj = proj / proj.norm(dim=1, keepdim=True) / 3.0
    coords = torch.stack([hp.centres(torch.linspace(-4.0, 4.0, b + 1))] * k)
    tables = 1.0 + 0.1 * (torch.rand(k, b, generator=gen) - 0.5)   # 194 factors near 1: no underflow
    return proj, coords, tables


def _oracle_factors(proj, coords, tables, x):
    want = torch.ones(x.shape[0])
    u = x.double() @ proj.double().T
    for i in range(proj.shape[0]):
        want = want * torch.clamp(hp.lagrange_interp(tables[i], coords[i], u[:, i]).float(), 0.0, 1.0e10)
    return want


def test_largest_table_count_runs_and_one_more_is_refused():
    d, b, limit = 6, 64, 200 * 1024
    kmax = max(k for k in range(1, 1000) if _ment_smem(k, b, d) <= limit)
    assert _ment_smem(kmax + 1, b, d) > limit
    proj, coords, tables = _smem_tables(kmax + 1, d, b, 11)
    x = torch.randn(4096, d, generator=torch.Generator().manual_seed(12))
    g = tuple(t[:kmax].cuda() for t in (proj, coords, tables))
    got = ops.ment_prob(x.cuda(), g, None, 0.0, 0.0).cpu()
    want = _oracle_factors(*(t[:kmax] for t in (proj, coords, tables)), x)
    assert int((want > 0).sum()) > 0.9 * want.numel()
    assert torch.allclose(got, want, rtol=1e-4, atol=0.0)
    with pytest.raises(RuntimeError, match="code"):
        ops.ment_prob(x.cuda(), tuple(t.cuda() for t in (proj, coords, tables)), None, 0.0, 0.0)
    # no sticky error: the next op and the next MENT call work
    assert float(torch.ones(8, device="cuda").sum()) == 8.0
    assert torch.equal(ops.ment_prob(x.cuda(), g, None, 0.0, 0.0).cpu(), got)

    # integrate mode: one screen (measured axis 0, 8 pixels) over a 3^5 grid, the same two table counts
    minv = torch.eye(d).cuda()
    mc = hp.centres(torch.linspace(-2.0, 2.0, 9))
    shape, first, step = [3] * 5, [-1.5] * 5, [1.5] * 5
    pred = ops.ment_integrate(d, mc.cuda(), 0, None, -1, shape, first, step, minv, g, None, 0.0, 0.0).cpu()
    mesh = torch.meshgrid(mc.double(), *[torch.tensor([-1.5, 0.0, 1.5], dtype=torch.float64)] * 5, indexing="ij")
    u = torch.stack([m.reshape(-1) for m in mesh], 1)
    want = _oracle_factors(*(t[:kmax] for t in (proj, coords, tables)), u).double().reshape(8, -1).sum(1).float()
    assert float(want.min()) > 0
    assert torch.allclose(pred, want, rtol=1e-4, atol=0.0)
    with pytest.raises(RuntimeError, match="code"):
        ops.ment_integrate(d, mc.cuda(), 0, None, -1, shape, first, step, minv,
                           tuple(t.cuda() for t in (proj, coords, tables)), None, 0.0, 0.0)
    assert torch.equal(ops.ment_integrate(d, mc.cuda(), 0, None, -1, shape, first, step, minv, g, None, 0.0,
                                          0.0).cpu(), pred)


# ---------------------------------------------------------------------------------------------- integrate mode
_RAGGED = [4, 3, 1, 5, 2, 3, 4]


def _int_shapes(dg, d):
    n = d - (2 if isinstance(dg, mf.diagnostics.Histogram2D) else 1)
    return tuple(_RAGGED[:n]) if n > 1 else (40,)


def _integrate_model(d, seed, twod):
    """1-D screens on every axis (``twod`` False) or the 2-D pairs of `_pairs` beside one 1-D screen; ragged
    integration grids with an axis of size 1 (a few hundred to a few thousand points per pixel)."""
    gen = torch.Generator().manual_seed(seed)
    if twod:
        rows = [[_s2(p, 8, 6)] for p in _pairs(d)] + [[_s1(d - 1, 16)]]
    else:
        rows = [[_s1(a, 16)] for a in range(d)]
    tfs = [LinearTransform(_matrix(d, gen).cuda()) for _ in rows]
    meas = [[torch.ones(16).cuda() if isinstance(dg, mf.diagnostics.Histogram1D) else torch.ones(8, 6).cuda()
             for dg in row] for row in rows]
    return mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=rows, measurements=meas,
                        prior=mf.prior.Gaussian(ndim=d, scale=1.0), mode="integrate",
                        integration_limits=[[[(-3.5, 3.5)] * len(_int_shapes(dg, d)) for dg in row] for row in rows],
                        integration_shape=[[_int_shapes(dg, d) for dg in row] for row in rows], device="cuda")


def _tables_and_measurements(model, seed):
    """positive_tables, then measurements within 15 % of the float64 prediction of those tables (one measured zero per
    screen, whose entry keeps its table value): the sweeps correct by factors near 1, as on data MENT can fit.  Random
    measurements that no density fits drive the tables over decades within two sweeps, where the factors meas / pred of
    the tails amplify fp32 rounding beyond any fixed tolerance."""
    positive_tables(model, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    for i, row in enumerate(model.diagnostics):
        for j in range(len(row)):
            w = oracle_integrate(model, i, j)
            m = w * (0.85 + 0.3 * torch.rand(w.shape, generator=gen))
            m.view(-1)[3] = 0.0
            model.measurements[i][j] = m.cuda()


@pytest.mark.parametrize("d", [2, 3, 5, 7, 8])
def test_integrate_1d_screens_on_every_axis_match_float64(d):
    model = _integrate_model(d, 70 + d, twod=False)
    _tables_and_measurements(model, 80 + d)
    integrate_check(model, [(i, 0) for i in range(d)])


@pytest.mark.parametrize("d", [3, 5, 8])
def test_integrate_2d_screens_match_float64(d):
    model = _integrate_model(d, 90 + d, twod=True)
    assert any(dg.axis == (2, 0) for row in model.diagnostics for dg in row)
    _tables_and_measurements(model, 100 + d)
    integrate_check(model, [(i, 0) for i in range(len(model.transforms))])


def test_integrate_composite_of_linear_maps_matches_float64():
    """A composite of two linear maps in front of the 1-D screen on axis 1.  (In front of a 2-D screen, one table entry
    next to the zero border ended two sweeps 2.2e-4 from float64 while every prediction above 1e-3 of the largest
    agreed to 4e-6: that pixel's prediction carries the fp32 rounding near the zero ends of the other tables, which the
    update's meas / pred passes on in full.  The 2-D screens are checked behind single maps above.)"""
    d = 5
    model = _integrate_model(d, 111, twod=False)
    gen = torch.Generator().manual_seed(112)
    model.transforms[1] = CompositeTransform(LinearTransform(_matrix(d, gen).cuda()),
                                             LinearTransform(_matrix(d, gen).cuda()))
    model._packed = None
    _tables_and_measurements(model, 113)
    integrate_check(model, [(i, 0) for i in range(len(model.transforms))])


# ---------------------------------------------------------------------------------------------- CDF and sampler
def _cdf_draw(rho, shape, first, cell, size, seed, offset, jitter, pad):
    """mfb_cdf_build + mfb_cdf_sample as ops.cdf_sample calls them, keeping the cdf and the total (workspace[0])."""
    lib = _lib.load()
    g, d = rho.numel(), len(shape)
    cdf = torch.empty(g, dtype=torch.float64, device="cuda")
    out = torch.empty((size, d), dtype=torch.float32, device="cuda")
    wbytes = lib.mfb_cdf_workspace_bytes(g)
    work = torch.empty(wbytes, dtype=torch.uint8, device="cuda")
    a1, p1 = ops._host_i32(shape)
    a2, p2 = ops._host_f32(first)
    a3, p3 = ops._host_f32(cell)
    _lib.check(lib.mfb_cdf_build(ops._ptr(rho), g, float(pad), ops._ptr(cdf), ops._ptr(work), wbytes, ops._stream()))
    _lib.check(lib.mfb_cdf_sample(ops._ptr(cdf), g, ops._ptr(work), d, p1, p2, p3, int(jitter), seed, offset, size,
                                  ops._ptr(out), ops._stream()))
    return cdf.cpu().numpy(), float(work[:8].view(torch.float64).cpu()), out.cpu().numpy()


def _compensated_prefix(x):
    """Inclusive prefix of x (float64): cumsum inside tiles of 4096, math.fsum of the tile sums before each tile."""
    n = x.size
    tiles = -(-n // 4096)
    xp = np.zeros(tiles * 4096)
    xp[:n] = x
    xp = xp.reshape(tiles, 4096)
    sums = [math.fsum(t) for t in xp]
    offs, acc = np.zeros(tiles), []
    for j in range(tiles):
        offs[j] = math.fsum(acc)
        acc.append(sums[j])
        if len(acc) > 64:
            acc = [math.fsum(acc)]
    return (np.cumsum(xp, axis=1) + offs[:, None]).reshape(-1)[:n]


def _rho(kind, g, seed):
    rng = np.random.default_rng(seed)
    if kind == "ment":      # a Gaussian-ish bump with 9 cells in 10 zero (outside some screen)
        v = np.exp(-0.5 * ((np.arange(g) - g / 2) / (0.2 * g + 1)) ** 2) * rng.random(g)
        v[rng.random(g) < 0.9] = 0.0
        if g > 1:
            v[rng.integers(g)] = 1.0  # never all zero
        return v.astype(np.float32)
    return (10.0 ** rng.uniform(-30, 3, g)).astype(np.float32)   # "span": 1e-30 ... 1e3


# (shape, rho, pad, seed, offset, size, jitter)
_CDF_CASES = [
    ((1,), "span", 1e-15, 1, 0, 1000, False),
    ((2,), "ment", 0.0, 2, 0, 1000, True),
    ((3, 1), "span", 0.0, 3, 0, 1000, False),
    ((2, 2), "ment", 1e-15, 4, 7, 1000, False),
    ((5, 1, 1), "span", 1e-15, 5, 0, 1000, True),
    ((2, 2, 2, 2), "ment", 0.0, 6, 0, 4000, False),
    ((17, 1, 1, 1, 1), "ment", 1e-15, 7, 0, 4000, False),
    ((3, 3, 5, 7, 13), "span", 0.0, 2**40 + 9, 0, 20000, True),
    ((4, 4, 4, 4, 4, 4), "ment", 1e-15, 9, 2**32 - 5000, 10000, False),
    ((17, 241), "ment", 0.0, 10, 0, 20000, False),
    ((3, 4, 5, 2, 3, 4, 5), "span", 1e-15, 11, 0, 20000, True),
    ((2, 3, 2, 3, 2, 3, 2, 3), "ment", 0.0, 12, 2**33, 20000, False),
    ((65537, 1, 1, 1, 1, 1, 1, 1), "ment", 1e-15, 13, 0, 400000, False),      # 4^8 + 1; size > SMs x 8 x 256
    ((16,) * 6, "ment", 0.0, 14, 0, 100000, False),                           # 4096 tiles
    ((16,) * 6, "ment", 1e-15, 2**63 + 15, 2**32 - 50000, 100000, True),
    ((3, 2796203), "ment", 1e-15, 16, 0, 100000, False),                      # 2049 tiles: ragged offset chunks
]


def _ulps(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


@pytest.mark.parametrize("shape,kind,pad,seed,offset,size,jitter", _CDF_CASES)
def test_cdf_and_every_draw_match_an_exact_replay(shape, kind, pad, seed, offset, size, jitter):
    d, g = len(shape), int(np.prod(shape))
    rho = _rho(kind, g, seed % 1000)
    lo = np.linspace(-3.0, -1.0, d).astype(np.float32)
    cell = np.linspace(0.3, 0.05, d).astype(np.float32)
    cdf, total, out = _cdf_draw(torch.from_numpy(rho).cuda(), list(shape), lo.tolist(), cell.tolist(), size, seed,
                                offset, jitter, pad)
    w = rho.astype(np.float64) + pad
    # the CDF: the exact prefix to 1e-11 of the total, non-decreasing, its last entry the total
    ref = _compensated_prefix(w)
    assert np.max(np.abs(cdf - ref)) <= 1e-11 * ref[-1]
    dec = np.nonzero(np.diff(cdf) < 0)[0]
    assert dec.size == 0, f"cdf decreases at {dec.size} of {g - 1} steps, by up to {np.max(cdf[dec] - cdf[dec + 1])}"
    assert total == cdf[-1], (total, cdf[-1], total - cdf[-1])
    assert np.all(np.diff(cdf)[w[1:] == 0] == 0)           # a zero-weight cell adds nothing
    # the cells: a bisection of the CDF with the kernel's Philox stream
    uu, rnd = sampler_uniforms(seed, offset, size, d)
    cellidx = np.minimum(np.searchsorted(cdf, uu * total, side="right"), g - 1)
    idx = np.stack(np.unravel_index(cellidx, shape), axis=1)
    assert np.all(w[cellidx] > 0), "a draw landed in a cell of zero weight"
    # the coordinates against an fp32 emulation: lb = fmaf(idx, step, lo), v = fmaf(step, u01(rnd[2i]), lb), clamped
    # below ub (emulated exactly; 1 ulp allowed)
    lb = fmaf(idx.astype(np.float32), cell, lo)
    ub = fmaf((idx + 1).astype(np.float32), cell, lo)
    v = fmaf(cell, u01(rnd[:, 0::2]), lb)
    v = np.where(v < ub, v, np.nextafter(ub, lb))
    if jitter:
        # v += 0.5 step (2 u01(rnd[2i+1]) - 1): exactly one of the separately rounded or the fused multiply-add (the
        # compiler may contract it); an ulp count would not do, as the sum cancels near zero
        half, t = np.float32(0.5) * cell, np.float32(2.0) * u01(rnd[:, 1::2]) - np.float32(1.0)
        assert np.all((out == v + half * t) | (out == fmaf(half, t, v)))
    else:
        assert int(_ulps(out, v).max()) <= 1
        # every point lies in the bisection's cell [lb, ub): the drawn cell is the bisection's, draw by draw
        assert np.all(out >= lb) and np.all(out < ub)


def test_ops_cdf_sample_is_the_same_build_and_draw():
    rho = torch.from_numpy(_rho("ment", 4097, 5)).cuda()
    a = ops.cdf_sample(rho, [17, 241], [-1.0, -2.0], [0.1, 0.02], 5000, seed=77, offset=3, jitter=True)
    _, _, b = _cdf_draw(rho, [17, 241], [-1.0, -2.0], [0.1, 0.02], 5000, 77, 3, True, 1e-15)
    assert np.array_equal(a.cpu().numpy(), b)


def test_cdf_build_is_bitwise_reproducible():
    rho = torch.from_numpy(_rho("ment", 16 ** 6, 21)).cuda()
    first = _cdf_draw(rho, [16] * 6, [-3.0] * 6, [0.375] * 6, 1000, 5, 0, False, 1e-15)
    second = _cdf_draw(rho, [16] * 6, [-3.0] * 6, [0.375] * 6, 1000, 5, 0, False, 1e-15)
    assert np.array_equal(first[0], second[0]) and first[1] == second[1] and np.array_equal(first[2], second[2])


# ---------------------------------------------------------------------------------------------- Gauss-Seidel rule
@pytest.mark.parametrize("lr", [0.25, 1.0, 1.5])
@pytest.mark.parametrize("n", [1, 255, 257, 85 * 85])
def test_gs_update_edges_match_the_rule(lr, n):
    """pred == thresh is kept, one ulp below is zeroed; meas == 0 and pred == 0 leave the entry; n off 256
    (n = 85 * 85: a flattened 2-D table)."""
    gen = torch.Generator().manual_seed(n)
    thresh = 1.0e-3
    table = torch.rand(n, generator=gen) + 0.5
    meas = torch.rand(n, generator=gen) + 0.1
    pred = torch.rand(n, generator=gen) * 2.0 + 0.01
    below = float(np.nextafter(np.float32(thresh), np.float32(0)))
    special = [(thresh, 0.7), (below, 0.7), (0.5, 0.0), (0.0, 0.4), (thresh, 0.0), (below, 0.0)]
    step = max(n // len(special), 1)
    for i, (p, m) in enumerate(special[:n]):
        pred[i * step], meas[i * step] = p, m
    want = hp.gauss_seidel_table(table.double(), meas.double(), pred.double(), lr, thresh)
    got = table.clone().cuda()
    ops.gs_update(got, meas.cuda(), pred.cuda(), lr, thresh)
    got = got.cpu()
    # 1e-6 of the size of the terms: with lr > 1, 1 + lr (g / p - 1) cancels where g / p is near 1 - 1 / lr, and the
    # kernel's fp32 arithmetic (g / p rounded, the multiply-add possibly fused) is then exact only to that size
    scale = table.double().abs() * (1.0 + lr * ((meas.double() / pred.double().clamp_min(1e-30)).abs() + 1.0))
    assert bool(((got.double() - want).abs() <= 1e-6 * scale).all())
    assert torch.equal(got == 0, want == 0)
    if n >= len(special):
        assert float(got[0]) != float(table[0])          # pred == thresh: updated
        assert float(got[step]) == float(table[step])    # one ulp below thresh: zeroed, entry kept
        assert torch.equal(got[2 * step:6 * step:step], table[2 * step:6 * step:step])
