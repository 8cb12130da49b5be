"""GPU parity: classical MENT with screens of different sizes (the ragged layout of the Lagrange tables).

- the ragged entry points on equal-size models return the uniform ones' output bit for bit: every compiled D, 1-D
  screens only, 2-D screens only and both, with and without kicks, Gaussian and flat priors; prob, prob_grid,
  integrate and the fused MH chains (states and accepted count);
- the density of a model whose screens all differ in size against the float64 oracle of mfb_testutil, with
  non-uniform centres and kicked chains of order 3, 4 and 5 beside linear maps; the interpolation at every table edge,
  one ulp inside and outside, against scipy;
- the shared-memory limit of the ragged layout: the largest total that fits evaluates correctly, one bin more is
  refused before any launch;
- integrate mode and two Gauss-Seidel sweeps against the oracle, linear and kicked;
- sample mode: fused chains against the step kernels around ragged densities, shards against one draw, and three
  sweeps lowering the KL in both modes."""
import numpy as np
import pytest
import torch
from scipy.interpolate import RegularGridInterpolator

import mentflow_b200 as mf
from mentflow_b200 import ops
from mentflow_b200.distributed import shard_slice
from mentflow_b200.simulate.transform import CompositeTransform, LinearTransform, MultipoleTransform
from mfb_testutil import check_density, fmaf, integrate_check, oracle_integrate, oracle_prob, positive_tables

pytestmark = pytest.mark.gpu

MH = mf.sample.MetropolisHastingsSampler


# ---------------------------------------------------------------------------------------------- ragged = uniform
def _centres(n, gen, lo=-3.0, hi=3.0):
    """n sorted, distinct, non-uniform centres in [lo, hi]."""
    steps = 0.3 + torch.rand(n - 1, generator=gen)
    c = torch.cat([torch.zeros(1), torch.cumsum(steps, 0)])
    return (lo + (hi - lo) * c / c[-1]).float()


def _mp_rows(k, d, gen, rows=1):
    """Multipole rows [wa | wb | a | b | order | 0] of orders 0 (a linear map), 3, 4 and 5: (k, 2D+4), or
    (k, 2, 2D+4) for 2-D screens (``rows`` = 2), whose two rows share wa, wb and the order."""
    mp = torch.zeros(k, rows, 2 * d + 4)
    mp[:, :, :2 * d] = (torch.randn(k, 1, 2 * d, generator=gen) * 0.4).expand(k, rows, 2 * d)
    mp[:, :, 2 * d:2 * d + 2] = torch.randn(k, rows, 2, generator=gen) * 0.05
    mp[:, :, 2 * d + 2] = torch.tensor([(0.0, 3.0, 4.0, 5.0)[i % 4] for i in range(k)])[:, None]
    return (mp[:, 0] if rows == 1 else mp).contiguous().cuda()


def _uniform_groups(d, kind, kick, seed):
    """Equal-size families as ops takes them: 1-D (K = 5, B = 17), 2-D (K2 = 3, 9 x 6)."""
    gen = torch.Generator().manual_seed(seed)
    g1 = g2 = None
    if kind in ("1d", "mixed"):
        k, b = 5, 17
        g1 = (torch.randn(k, d, generator=gen) * 0.6, torch.stack([_centres(b, gen) for _ in range(k)]),
              torch.rand(k, b, generator=gen) + 0.2)
        g1 = tuple(t.cuda() for t in g1) + ((_mp_rows(k, d, gen),) if kick else ())
    if kind in ("2d", "mixed"):
        k, bx, by = 3, 9, 6
        g2 = (torch.randn(k, 2, d, generator=gen) * 0.6, torch.stack([_centres(bx, gen) for _ in range(k)]),
              torch.stack([_centres(by, gen, -2.5, 2.5) for _ in range(k)]), torch.rand(k, bx, by, generator=gen) + 0.2)
        g2 = tuple(t.cuda() for t in g2) + ((_mp_rows(k, d, gen, 2),) if kick else ())
    return g1, g2


def _ragged(g1, g2):
    """The same tables as RaggedTables1D / RaggedTables2D."""
    r1 = r2 = None
    if g1 is not None:
        k, b = g1[2].shape
        r1 = ops.RaggedTables1D(g1[0], g1[1].reshape(-1), g1[2].reshape(-1), [i * b for i in range(k + 1)],
                                g1[3] if len(g1) > 3 else None)
    if g2 is not None:
        k, bx, by = g2[3].shape
        r2 = ops.RaggedTables2D(g2[0], g2[1].reshape(-1), g2[2].reshape(-1), g2[3].reshape(-1),
                                [[i * n for i in range(k + 1)] for n in (bx, by, bx * by)], g2[4] if len(g2) > 4 else None)
    return r1, r2


_PRIORS = {"gauss": (-0.5 / 1.5 ** 2, -1.0), "flat": (0.0, -2.0)}


@pytest.mark.parametrize("d", range(1, 9))
def test_ragged_entry_points_equal_the_uniform_ones_bit_for_bit(d):
    gen = torch.Generator().manual_seed(d)
    x = (torch.randn(30000, d, generator=gen) * 1.3).cuda()
    shape = [(9, 7, 5, 4, 3, 3, 2, 2)[i] for i in range(d)]
    first, step = [-2.5] * d, [5.0 / (s - 1) for s in shape]
    chol = torch.linalg.cholesky(torch.eye(d) * 0.3 + 0.05).float().cuda()
    for kind in ("1d", "2d", "mixed"):
        for kick in (False, True):
            for prior, (a, b) in _PRIORS.items():
                g1, g2 = _uniform_groups(d, kind, kick, seed=10 * d + len(kind))
                r1, r2 = _ragged(g1, g2)
                why = (kind, kick, prior)
                want = ops.ment_prob(x, g1, g2, a, b)
                assert int((want > 0).sum()) > 1000, why
                assert torch.equal(ops.ment_prob(x, r1, g2, a, b), want), why
                assert torch.equal(ops.ment_prob(x, r1, r2, a, b), want), why
                want = ops.ment_prob_grid(shape, first, step, g1, g2, a, b, "cuda")
                assert torch.equal(ops.ment_prob_grid(shape, first, step, r1, r2, a, b, "cuda"), want), why
                want, acc = ops.ment_mh(g1, g2, a, b, d, 3, 2000, chol, 4, 3, 2, seed=5, start_scale=1.0)
                got, acc_r = ops.ment_mh(r1, r2, a, b, d, 3, 2000, chol, 4, 3, 2, seed=5, start_scale=1.0)
                assert torch.equal(got, want) and int(acc_r) == int(acc) > 0, why
                if d >= 2:
                    minv = (torch.eye(d) + 0.1 * torch.randn(d, d, generator=gen)).cuda()
                    inv_mp = None
                    if kick:
                        inv_mp = torch.cat([torch.randn(4 * d, generator=gen) * 0.1, torch.tensor([3.0, 0.0])]).cuda()
                    mc = _centres(11, gen).cuda()
                    ishape = [5] * (d - 1)
                    args = (ishape, [-2.0] * (d - 1), [1.0] * (d - 1), minv)
                    want = ops.ment_integrate(d, mc, 0, None, -1, *args, g1, g2, a, b, inv_mp=inv_mp)
                    got = ops.ment_integrate(d, mc, 0, None, -1, *args, r1, r2, a, b, inv_mp=inv_mp)
                    assert torch.equal(got, want) and float(want.max()) > 0, why


# ---------------------------------------------------------------------------------------------- density vs float64
def _s1(axis, b, lim=4.0):
    return mf.diagnostics.Histogram1D(axis=axis, edges=torch.linspace(-lim, lim, b + 1), bandwidth=0.5).to("cuda")


def _s2(axes, bx, by, seed):
    """Non-uniform centres: edges with random spacing."""
    gen = torch.Generator().manual_seed(seed)
    ex, ey = _centres(bx + 1, gen, -4.0, 4.0), _centres(by + 1, gen, -3.5, 3.5)
    return mf.diagnostics.Histogram2D(axis=axes, edges=(ex, ey), bandwidth=(0.5, 0.5)).to("cuda")


def _matrix(d, gen):
    q1, _ = torch.linalg.qr(torch.randn(d, d, generator=gen, dtype=torch.float64))
    q2, _ = torch.linalg.qr(torch.randn(d, d, generator=gen, dtype=torch.float64))
    s = 0.75 + 0.55 * torch.rand(d, generator=gen, dtype=torch.float64)
    return ((q1 * s) @ q2).float()


def _kicked(d, gen, order):
    return CompositeTransform(LinearTransform(_matrix(d, gen).cuda()), MultipoleTransform(order=order, strength=0.2),
                              LinearTransform(_matrix(d, gen).cuda()))


def _mixed_model(d, kick, prior, sampler=None, mode="sample", seed=0):
    """1-D screens of 2, 3, 17, 64 and 85 bins and 2-D screens of 2 x 2, 40 x 50 and 85 x 85 on five maps; with
    ``kick`` the first three maps are chains behind kicks of order 3, 4 and 5."""
    gen = torch.Generator().manual_seed(seed)
    tfs = [(_kicked(d, gen, 3 + i) if kick and i < 3 else LinearTransform(_matrix(d, gen).cuda())) for i in range(5)]
    bins1 = (2, 3, 17, 64, 85)
    shapes2 = ((2, 2), (40, 50), (85, 85))
    diags = []
    for i in range(5):
        row = [_s1(i % d, bins1[i])]
        if i < 3:
            row.append(_s2((i % d, (i + 1) % d), *shapes2[i], seed=seed + i))
        diags.append(row)
    meas = [[torch.ones(dg.edges.numel() - 1).cuda() if isinstance(dg, mf.diagnostics.Histogram1D)
             else torch.ones(dg.edges_x.numel() - 1, dg.edges_y.numel() - 1).cuda() for dg in row] for row in diags]
    pr = mf.prior.Gaussian(ndim=d, scale=1.0) if prior == "gauss" else mf.prior.Uniform(ndim=d, scale=10.0)
    model = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas, prior=pr, mode=mode,
                         sampler=sampler, device="cuda")
    positive_tables(model, seed + 7)
    gen = torch.Generator().manual_seed(seed + 8)
    for row in model.lagrange_functions:      # tables of fewer than 4 centres on an axis keep their ends (else all 0)
        for lf in row:
            if min(lf.values.shape) < 4:
                lf.set_values((torch.rand(lf.values.shape, generator=gen) + 0.2).cuda())
    return model


@pytest.mark.parametrize("d,kick,prior", [(2, False, "gauss"), (4, True, "flat"), (5, False, "flat"),
                                          (6, True, "gauss")])
def test_density_of_screens_of_every_size_matches_float64(d, kick, prior):
    lim = 2.5 if d <= 4 else 1.8
    sampler = mf.sample.GridSampler(limits=d * [(-lim, lim)], shape=(5, 7, 4, 3, 3, 3)[:d], device="cuda")
    model = _mixed_model(d, kick, prior, sampler=sampler, seed=d)
    pk = model._pack(torch.device("cuda"))
    assert pk["offsets"] == [0, 2, 5, 22, 86, 171]
    assert pk["offsets2"][2] == [0, 4, 2004, 2004 + 85 * 85] and pk["kicked"] == kick
    x = torch.randn(20000, d, generator=torch.Generator().manual_seed(d)) * 0.8
    check_density(model, x, oracle_prob(model, x))


def test_interpolation_at_every_table_edge_matches_scipy():
    """Unit projection rows (the fp32 projection is exact): h at each table's first and last centre, one ulp inside
    and one outside, and at random points, against RegularGridInterpolator (linear, 0 outside)."""
    gen = torch.Generator().manual_seed(4)
    sizes = (2, 3, 17, 64, 85)
    coords = [_centres(b, gen) for b in sizes]
    values = [torch.rand(b, generator=gen) + 0.1 for b in sizes]
    off = [0]
    for b in sizes:
        off.append(off[-1] + b)
    for k, (c, v) in enumerate(zip(coords, values)):
        cn = c.numpy()
        pts = np.concatenate([[cn[0], cn[-1], np.nextafter(cn[0], np.float32(np.inf)),
                               np.nextafter(cn[-1], np.float32(-np.inf)), np.nextafter(cn[0], np.float32(-np.inf)),
                               np.nextafter(cn[-1], np.float32(np.inf))], cn,
                              np.random.default_rng(k).uniform(-3.2, 3.2, 500).astype(np.float32)]).astype(np.float32)
        # one model of all five tables, each evaluated through its own unit row; the others see u = 0 inside
        proj = torch.zeros(len(sizes), 1)
        proj[k, 0] = 1.0
        r1 = ops.RaggedTables1D(proj.cuda(), torch.cat(coords).cuda(),
                                torch.cat([vv if i == k else torch.ones_like(vv) for i, vv in enumerate(values)]).cuda(),
                                off)
        got = ops.ment_prob(torch.from_numpy(pts).reshape(-1, 1).cuda(), r1, None, 0.0, 0.0).cpu().numpy()
        want = RegularGridInterpolator((cn.astype(np.float64),), v.numpy().astype(np.float64), method="linear",
                                       bounds_error=False, fill_value=0.0)(pts.astype(np.float64)[:, None])
        np.testing.assert_allclose(got, want.astype(np.float32), rtol=1e-6, atol=0)
        assert got[4] == 0 and got[5] == 0 and got[0] > 0 and got[1] > 0
    # 2-D: 2 x 2, 40 x 50 and 85 x 85 with identity rows, the corners and edges of each table
    shapes = ((2, 2), (40, 50), (85, 85))
    cx = [_centres(a, gen) for a, _ in shapes]
    cy = [_centres(b, gen, -2.5, 2.5) for _, b in shapes]
    tabs = [torch.rand(a, b, generator=gen) + 0.1 for a, b in shapes]
    offs = [[0], [0], [0]]
    for a, b in shapes:
        offs[0].append(offs[0][-1] + a)
        offs[1].append(offs[1][-1] + b)
        offs[2].append(offs[2][-1] + a * b)
    for k in range(len(shapes)):
        proj2 = torch.zeros(len(shapes), 2, 2)
        proj2[k] = torch.eye(2)
        r2 = ops.RaggedTables2D(proj2.cuda(), torch.cat(cx).cuda(), torch.cat(cy).cuda(),
                                torch.cat([(t if i == k else torch.ones_like(t)).reshape(-1)
                                           for i, t in enumerate(tabs)]).cuda(), offs)
        xs, ys = cx[k].numpy(), cy[k].numpy()
        ex = [xs[0], xs[-1], np.nextafter(xs[0], np.float32(np.inf)), np.nextafter(xs[-1], np.float32(-np.inf)),
              np.nextafter(xs[0], np.float32(-np.inf)), np.nextafter(xs[-1], np.float32(np.inf)), 0.1]
        ey = [ys[0], ys[-1], np.nextafter(ys[0], np.float32(np.inf)), np.nextafter(ys[-1], np.float32(-np.inf)),
              np.nextafter(ys[0], np.float32(-np.inf)), np.nextafter(ys[-1], np.float32(np.inf)), -0.2]
        pts = np.array([(a, b) for a in ex for b in ey], dtype=np.float32)
        got = ops.ment_prob(torch.from_numpy(pts).cuda(), None, r2, 0.0, 0.0).cpu().numpy()
        want = RegularGridInterpolator((xs.astype(np.float64), ys.astype(np.float64)),
                                       tabs[k].numpy().astype(np.float64), method="linear", bounds_error=False,
                                       fill_value=0.0)(pts.astype(np.float64))
        np.testing.assert_allclose(got, want.astype(np.float32), rtol=1e-6, atol=0)
        assert (got > 0).sum() == 25 and (want > 0).sum() == 25      # 5 x 5 points in the closed box


# ---------------------------------------------------------------------------------------------- shared-memory limit
def _zero_ends(v):
    """h continuous at the ends of its table: a point whose fp32 and float64 projections straddle an end sees no
    jump."""
    v[0] = v[-1] = 0.0
    return v


def _smem_ragged(k, t, d):
    """ment.cu ment_smem_ragged (bytes): proj, offsets, centres, values, inverse steps, double inverse gaps."""
    return ((k * d + 3) // 4 * 4 + (k + 2) // 2 * 2 + 2 * t + (k + 1) // 2 * 2) * 4 + t * 8 + 16


def test_largest_ragged_total_that_fits_evaluates_and_one_more_bin_is_refused():
    d, k = 3, 7
    t = max(t for t in range(1, 20000) if _smem_ragged(k, t, d) <= 200 * 1024)
    assert _smem_ragged(k, t + 1, d) > 200 * 1024
    gen = torch.Generator().manual_seed(9)
    sizes = [4, 5, 100] + [0] * (k - 3)
    rest = t - sum(sizes)
    for i in range(3, k):
        sizes[i] = rest // (k - 3) + (1 if i - 3 < rest % (k - 3) else 0)
    assert sum(sizes) == t and min(sizes) >= 2 and len(set(sizes)) > 3
    coords = [_centres(b, gen, -4.0, 4.0) for b in sizes]
    values = [_zero_ends(torch.rand(b, generator=gen) + 0.3) for b in sizes]
    off = [0]
    for b in sizes:
        off.append(off[-1] + b)
    proj = torch.randn(k, d, generator=gen) * 0.4
    x = torch.randn(5000, d, generator=gen)
    r1 = ops.RaggedTables1D(proj.cuda(), torch.cat(coords).cuda(), torch.cat(values).cuda(), off)
    got = ops.ment_prob(x.cuda(), r1, None, 0.0, 0.0).cpu()
    # the tables of ~3000 bins are steep: take the kernel's fp32 projection (an fmaf chain over the axes) and check
    # the interpolation, clamp and product alone
    xn, pn = x.numpy(), proj.numpy()
    want = torch.ones(x.shape[0], dtype=torch.float32)
    for i in range(k):
        u = np.zeros(x.shape[0], dtype=np.float32)
        for j in range(d):
            u = fmaf(pn[i, j], xn[:, j], u)
        h = RegularGridInterpolator((coords[i].double().numpy(),), values[i].double().numpy(), method="linear",
                                    bounds_error=False, fill_value=0.0)(u.astype(np.float64)[:, None])
        want = want * torch.from_numpy(h).float()
    assert int((want > 0).sum()) > 1000
    assert torch.allclose(got, want, rtol=1e-5, atol=0), float(((got - want).abs() / want.max()).max())
    sizes[-1] += 1
    off[-1] += 1
    coords[-1] = _centres(sizes[-1], gen, -4.0, 4.0)
    values[-1] = _zero_ends(torch.rand(sizes[-1], generator=gen) + 0.3)
    r1 = ops.RaggedTables1D(proj.cuda(), torch.cat(coords).cuda(), torch.cat(values).cuda(), off)
    with pytest.raises(RuntimeError, match="code -2"):
        ops.ment_prob(x.cuda(), r1, None, 0.0, 0.0)


# ---------------------------------------------------------------------------------------------- integrate mode
def _integrate_model(kick):
    """4-D: 1-D screens of 60 and 85 bins, 2-D screens of 32 x 32 and 48 x 40; the second map behind a kick if
    ``kick``."""
    d = 4
    gen = torch.Generator().manual_seed(21)
    tfs = [LinearTransform(_matrix(d, gen).cuda()),
           (_kicked(d, gen, 3) if kick else LinearTransform(_matrix(d, gen).cuda()))]
    e32, e48, e40 = (torch.linspace(-3.5, 3.5, n + 1) for n in (32, 48, 40))
    diags = [[_s1(0, 60, 3.5), mf.diagnostics.Histogram2D(axis=(1, 2), edges=(e32, e32), bandwidth=(0.5, 0.5)).to("cuda")],
             [_s1(3, 85, 3.5), mf.diagnostics.Histogram2D(axis=(0, 2), edges=(e48, e40), bandwidth=(0.5, 0.5)).to("cuda")]]
    meas = [[torch.ones(60).cuda(), torch.ones(32, 32).cuda()], [torch.ones(85).cuda(), torch.ones(48, 40).cuda()]]
    lim = [(-3.0, 3.0)]
    model = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=d, scale=1.5), mode="integrate",
                         integration_limits=[[lim * 3, lim * 2], [lim * 3, lim * 2]],
                         integration_shape=[[(9, 9, 9), (12, 12)], [(9, 9, 9), (12, 12)]], device="cuda")
    # positive tables zero at their ends, and measurements within 15 % of their float64 prediction (one measured zero
    # per screen): the sweeps correct by factors near 1, as on data MENT can fit, and h has no jump at a table's end
    positive_tables(model, 22)
    gen = torch.Generator().manual_seed(23)
    for i, row in enumerate(model.diagnostics):
        for j in range(len(row)):
            w = oracle_integrate(model, i, j)
            m = w * (0.85 + 0.3 * torch.rand(w.shape, generator=gen))
            m.view(-1)[3] = 0.0
            model.measurements[i][j] = m.cuda()
    return model


@pytest.mark.parametrize("kick", [False, True])
def test_integrate_mode_and_two_sweeps_match_float64(kick):
    model = _integrate_model(kick)
    pk = model._pack(torch.device("cuda"))
    assert pk["offsets"] == [0, 60, 145] and pk["offsets2"][2] == [0, 1024, 1024 + 48 * 40]
    integrate_check(model, [(0, 0), (0, 1), (1, 0), (1, 1)])


# ---------------------------------------------------------------------------------------------- sample mode
def test_fused_chains_equal_the_step_kernels_around_ragged_densities():
    for d, kick in ((3, False), (4, True)):
        model = _mixed_model(d, kick, "gauss", seed=30 + d)
        assert isinstance(model._groups(torch.device("cuda"))[0], ops.RaggedTables1D)
        s = MH(d, burnin=3, steps=4, thin=2, start_scale=0.8)
        for offset in (0, 5):
            a = s(model.prob, 3001, seed=99, offset=offset)
            ra = s.acceptance_rate.clone()
            b = s(lambda x: model.prob(x), 3001, seed=99, offset=offset)
            assert torch.equal(a, b) and torch.equal(ra, s.acceptance_rate) and float(ra) > 0


def test_shards_of_ragged_chains_concatenate_to_one_draw():
    model = _mixed_model(3, False, "gauss", seed=40)
    s = MH(3, burnin=2, steps=5, thin=2)
    full = s(model.prob, 1000, seed=8)
    for world in (2, 3, 8):
        parts = []
        for r in range(world):
            sl = shard_slice(1000, r, world)
            parts.append(s(model.prob, sl.stop - sl.start, seed=8, offset=sl.start))
        assert torch.equal(torch.cat(parts), full)


def _kl_model(sampler, mode):
    """3-D Gaussian truth seen by 1-D screens of 40, 56 and 72 bins and 2-D screens of 24 x 24 and 30 x 20."""
    d = 3
    gen = torch.Generator().manual_seed(50)
    a = torch.randn(d, d, generator=gen) * 0.3 + torch.eye(d)
    truth = (torch.randn(400_000, d, generator=gen) @ a.T).cuda()
    tfs = [LinearTransform(_matrix(d, gen).cuda()) for _ in range(3)]
    e = lambda n: torch.linspace(-5.0, 5.0, n + 1)   # noqa: E731
    diags = [[_s1(0, 40, 5.0), mf.diagnostics.Histogram2D(axis=(1, 2), edges=(e(24), e(24)),
                                                          bandwidth=(0.5, 0.5)).to("cuda")],
             [_s1(1, 56, 5.0)],
             [_s1(2, 72, 5.0), mf.diagnostics.Histogram2D(axis=(0, 1), edges=(e(30), e(20)),
                                                          bandwidth=(0.5, 0.5)).to("cuda")]]
    with torch.no_grad():
        meas = mf.simulate.forward(truth, tfs, diags)
    lim = [(-5.0, 5.0)]
    return mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                        prior=mf.prior.Gaussian(ndim=d, scale=2.0), mode=mode, sampler=sampler, n_samples=1_000_000,
                        integration_limits=[[lim * 2, lim], [lim * 2], [lim * 2, lim]],
                        integration_shape=[[(40, 40), (40,)], [(40, 40)], [(40, 40), (40,)]], device="cuda")


@pytest.mark.parametrize("mode", ["integrate", "sample"])
def test_three_sweeps_lower_the_mean_kl(mode):
    sampler = mf.sample.GridSampler(limits=3 * [(-5.0, 5.0)], shape=(64, 64, 64), device="cuda")
    model = _kl_model(sampler, mode)
    torch.manual_seed(0)

    def mean_kl():
        pred = model.simulate_all()
        return float(np.mean([float(mf.loss.kl_divergence(p, m)) for row_p, row_m in zip(pred, model.measurements)
                              for p, m in zip(row_p, row_m)]))

    kls = [mean_kl()]
    for _ in range(3):
        model.gauss_seidel_update(lr=0.8)
        kls.append(mean_kl())
    # the first sweeps take the KL down by an order of magnitude; near the fit, sample noise may move it a little
    assert kls[1] < 0.2 * kls[0] and max(kls[1:]) < 0.2 * kls[0] and kls[-1] < 0.1 * kls[0], kls
