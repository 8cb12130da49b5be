"""GPU: MetropolisHastingsSampler, the fused chain kernel over the MENT density and the step kernels around any density.

- replay: start points and one step of 1e5 chains for D = 1 ... 8 (1-D and 2-D screens, kicks) against a numpy replay
  of the documented Philox layout with float64 Box-Muller, every accept decision against the float64 density;
- fused = step by step, bit for bit, for several burnin / steps / thin, linear and kicked models, ragged sizes;
- shards: slices of one draw for R = 2, 3, 8 (boundaries inside chains, empty shards, chains past 2^32), also
  through MENT.shard;
- statistics: exact N(0, I) draws, burn-in from a wide start, screen profiles against a fine GridSampler, and a
  sample-mode sweep that lowers the KL;
- edges: a start outside every screen, zero-density proposals, NaN / inf densities, reproducibility."""
import math

import numpy as np
import pytest
import torch
from scipy import stats

import mentflow_b200 as mf
from mentflow_b200.distributed import shard_slice
from mentflow_b200.simulate.transform import CompositeTransform, LinearTransform, MultipoleTransform
from mfb_testutil import oracle_prob, positive_tables, t32
from test_ment_mh_host import mh_draw64

pytestmark = pytest.mark.gpu

MH = mf.sample.MetropolisHastingsSampler


def _matrix(d, gen):
    q1, _ = torch.linalg.qr(torch.randn(d, d, generator=gen, dtype=torch.float64))
    q2, _ = torch.linalg.qr(torch.randn(d, d, generator=gen, dtype=torch.float64))
    s = 0.75 + 0.55 * torch.rand(d, generator=gen, dtype=torch.float64)
    return ((q1 * s) @ q2).float()


def _model(d, seed, one_d=True, two_d=True, kick=False, n_samples=1000, sampler=None):
    """Three maps (the first behind an order-3 kick if ``kick``) with a 1-D screen each and a 2-D screen on the first
    two (D >= 2); random positive tables, zero on the outermost centres."""
    gen = torch.Generator().manual_seed(seed)
    tfs = [LinearTransform(_matrix(d, gen).cuda()) for _ in range(3)]
    if kick:
        tfs[0] = CompositeTransform(LinearTransform(_matrix(d, gen).cuda()), MultipoleTransform(order=3, strength=0.3),
                                    LinearTransform(_matrix(d, gen).cuda()))
    e1 = torch.linspace(-4.0, 4.0, 33)
    ex, ey = torch.linspace(-4.0, 4.0, 17), torch.linspace(-3.5, 3.5, 15)
    diags, meas = [], []
    for i in range(3):
        row = [mf.diagnostics.Histogram1D(axis=i % d, edges=e1, bandwidth=0.5).to("cuda")] if one_d else []
        if two_d and d >= 2 and i < 2:
            row.append(mf.diagnostics.Histogram2D(axis=(0, 1), edges=(ex, ey), bandwidth=(0.5, 0.5)).to("cuda"))
        diags.append(row)
        meas.append([torch.ones(32).cuda() if isinstance(g, mf.diagnostics.Histogram1D) else torch.ones(16, 14).cuda()
                     for g in row])
    model = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=d, scale=1.2), mode="sample", sampler=sampler,
                         n_samples=n_samples, device="cuda")
    positive_tables(model, seed + 100)
    return model


def _nonlinear(golden, sampler=None, n_samples=1000):
    g = golden("multipole")
    matrix = t32(g["nl_matrix"]).cuda()
    tfs = [CompositeTransform(MultipoleTransform(order=int(g["nl_order"]), strength=float(st)), LinearTransform(matrix))
           for st in g["nl_strengths"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=t32(g["nl_edges"]), bandwidth=0.5).to("cuda")
    return mf.ment.MENT(ndim=2, transforms=tfs, diagnostics=[[diag] for _ in tfs],
                        measurements=[[m.cuda()] for m in t32(g["nl_meas"])],
                        prior=mf.prior.Gaussian(ndim=2, scale=1.5), mode="sample", sampler=sampler,
                        n_samples=n_samples, device="cuda")


def _gaussian_model(d, sampler=None, n_samples=1000):
    """Identity maps onto 1-D screens of ones on [-30, 30]: rho is exactly the prior N(0, I) wherever a chain goes."""
    e = torch.linspace(-30.0, 30.0, 61)
    tfs = [LinearTransform(torch.eye(d).cuda()) for _ in range(d)]
    diags = [[mf.diagnostics.Histogram1D(axis=i, edges=e, bandwidth=0.5).to("cuda")] for i in range(d)]
    return mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=[[torch.ones(60).cuda()] for _ in tfs],
                        prior=mf.prior.Gaussian(ndim=d, scale=1.0), mode="sample", sampler=sampler,
                        n_samples=n_samples, device="cuda")


# ---------------------------------------------------------------------------------------------- replay against float64
def _replay(model, d, n=100_000, seed=1234, start_scale=1.0, offset=0):
    """Start draws (burnin 0) and one step (burnin 1) of n chains against the numpy replay.  Returns the number of
    accept decisions within the 1e-5 margin."""
    chains = np.uint64(offset) + np.arange(n, dtype=np.uint64)
    x0 = MH(d, burnin=0, start_scale=start_scale)(model.prob, n, seed=seed, offset=offset).cpu()
    xi0, _ = mh_draw64(chains, 0, seed, d)
    want0 = start_scale * xi0
    assert np.all(np.abs(x0.double().numpy() - want0) <= 1e-6 * np.maximum(1.0, np.abs(want0)))

    s1 = MH(d, burnin=1, start_scale=start_scale)
    x1 = s1(model.prob, n, seed=seed, offset=offset).cpu()
    xi, u = mh_draw64(chains, 1, seed, d)
    chol = s1.chol.double().numpy()
    x0d = x0.double().numpy()
    step = xi @ chol.T
    prop = x0d + step
    scale = np.maximum(1.0, np.abs(x0d) + np.abs(xi) @ np.abs(chol).T)     # magnitudes of the proposal's terms
    moved = (x1 != x0).any(dim=1).numpy()
    assert np.all(np.abs(x1.double().numpy()[moved] - prop[moved]) <= 1e-6 * scale[moved])
    assert torch.equal(x1[~torch.from_numpy(moved)], x0[~torch.from_numpy(moved)])
    assert int(s1.acceptance_rate.mul(n).round().item()) == int(moved.sum())

    rho0 = oracle_prob(model, x0.double()).double().numpy()
    rhop = oracle_prob(model, torch.from_numpy(prop)).double().numpy()
    lhs, rhs = rhop, u * rho0
    zero = (lhs == 0) & (rhs == 0)           # both sides exactly 0: the rule accepts
    clear = (np.abs(lhs - rhs) > 1e-5 * np.maximum(lhs, rhs)) | zero
    want = np.isfinite(rhop) & (lhs >= rhs)
    miss_zero = int((moved[zero] != want[zero]).sum())   # fp32 and float64 on either side of a table's last centre
    assert miss_zero <= 1e-3 * n
    clear &= ~(zero & (moved != want))
    assert np.array_equal(moved[clear], want[clear])
    assert (rho0 > 0).mean() > 0.2 and 0.05 < moved.mean() < 0.95      # the decisions are not vacuous
    inside = int((~clear).sum())
    print(f"D={d}: {inside} of {n} decisions inside the 1e-5 margin ({miss_zero} at zero density), "
          f"acceptance {moved.mean():.3f}")
    return inside


@pytest.mark.parametrize("d", range(1, 9))
def test_start_points_proposals_and_decisions_replay_in_float64(d):
    model = _model(d, seed=d, two_d=d >= 2)
    assert _replay(model, d) <= 1e-3 * 100_000


def test_replay_of_2d_screens_only_and_chains_past_2_32():
    model = _model(3, seed=31, one_d=False)
    assert model._groups(torch.device("cuda"))[0] is None
    assert _replay(model, 3, n=20_000, offset=2**33 + 5, start_scale=0.8) <= 20


def test_replay_of_kicked_chains(golden):
    nl = _nonlinear(golden, n_samples=10)
    positive_tables(nl, 6)
    assert _replay(nl, 2, start_scale=1.5) <= 100
    model = _model(4, seed=44, one_d=False, kick=True)          # 2-D screens behind a kick
    assert model._pack(torch.device("cuda"))["kicked"]
    assert _replay(model, 4) <= 100


# ---------------------------------------------------------------------------------------------- fused = step by step
_RUNS = [(0, 1, 1, 1001), (3, 4, 2, 777), (5, 3, 1, 1000), (0, 5, 3, 64), (2, 2, 4, 3)]


@pytest.mark.parametrize("kind", ["linear", "kick"])
@pytest.mark.parametrize("burnin,steps,thin,n", _RUNS)
def test_fused_kernel_equals_the_step_kernels_bit_for_bit(kind, burnin, steps, thin, n):
    model = _model(4 if kind == "kick" else 3, seed=7, kick=kind == "kick")
    s = MH(model.ndim, burnin=burnin, steps=steps, thin=thin, start_scale=0.9)
    for offset in (0, 5):
        a = s(model.prob, n, seed=99, offset=offset)
        ra = s.acceptance_rate.clone()
        b = s(lambda x: model.prob(x), n, seed=99, offset=offset)
        assert a.shape == (n, model.ndim) and torch.equal(a, b)
        assert torch.equal(ra, s.acceptance_rate)


def test_fused_equals_step_with_a_start_point_and_a_full_covariance():
    model = _model(5, seed=3)
    cov = torch.tensor(np.diag([0.5, 0.3, 0.8, 0.2, 0.4]) + 0.05, dtype=torch.float64)
    s = MH(5, burnin=4, steps=3, thin=2, proposal_cov=cov, start=torch.full((5,), 0.1))
    a, b = s(model.prob, 5000, seed=4), s(lambda x: model.prob(x), 5000, seed=4)
    assert torch.equal(a, b)
    assert not torch.equal(a[0], a[3])


# ---------------------------------------------------------------------------------------------- shards
@pytest.mark.parametrize("base", [0, 7 * 2**33 + 3])
def test_shards_concatenate_to_one_draw(base):
    model = _model(3, seed=11)
    s = MH(3, burnin=2, steps=7, thin=2)
    for total in (1000, 5):
        full = s(model.prob, total, seed=8, offset=base)
        for world in (2, 3, 8):
            parts = []
            for r in range(world):
                sl = shard_slice(total, r, world)
                parts.append(s(model.prob, sl.stop - sl.start, seed=8, offset=base + sl.start))
            if total == 5 and world == 8:
                assert min(p.shape[0] for p in parts) == 0
            assert torch.equal(torch.cat(parts), full)
    # chains past 2^32: the start draws of base // steps ... replay
    s0 = MH(3, burnin=0, start_scale=1.0)
    x = s0(model.prob, 100, seed=8, offset=base).cpu().double().numpy()
    xi, _ = mh_draw64(np.uint64(base) + np.arange(100, dtype=np.uint64), 0, 8, 3)
    assert np.abs(x - xi).max() <= 1e-6 * max(1.0, float(np.abs(xi).max()))


def test_sharded_ment_draws_are_slices_of_one_stream():
    sampler = MH(3, burnin=3, steps=4, thin=1)
    model = _model(3, seed=12, sampler=sampler, n_samples=100_003)
    torch.manual_seed(17)
    full = model.sample(100_003)
    for world in (2, 3, 8):
        parts = []
        for r in range(world):
            model.shard = (r, world)
            torch.manual_seed(17)
            parts.append(model.sample(100_003))
        model.shard = None
        assert torch.equal(torch.cat(parts), full)


# ---------------------------------------------------------------------------------------------- statistics
def _independent_normal(x):
    x = x.double().cpu()
    n, d = x.shape
    assert (x.mean(dim=0).abs() < 5 / math.sqrt(n)).all()
    cov = torch.cov(x.T).reshape(d, d)
    assert ((cov - torch.eye(d, dtype=torch.float64)).abs() < 6 * math.sqrt(2 / n)).all(), cov
    for i in range(d):
        assert stats.kstest(x[:, i].numpy(), "norm").pvalue > 1e-4


def test_start_draws_in_the_target_are_independent_normal_draws():
    model = _gaussian_model(3)
    s = MH(3, burnin=0, steps=1, start_scale=1.0)
    _independent_normal(s(model.prob, 200_000, seed=21))
    s = MH(3, burnin=50, steps=1, start_scale=1.0)         # chains that start in the target stay there
    _independent_normal(s(model.prob, 200_000, seed=22))


def test_burn_in_forgets_a_wide_start():
    """The fp32 density underflows to 0 beyond |x|^2 ~ 200 (exp(-100)), where a chain random-walks instead of
    drifting in: from start_scale = 4 in 3-D that is 0.6 % of the starts, and they keep the covariance near 2 for
    hundreds of steps.  From start_scale = 2.5 (starts 2.5x wider than the target, none beyond |x|^2 = 200 in
    practice) the burn-in must leave independent N(0, I) draws."""
    model = _gaussian_model(3)
    s = MH(3, burnin=400, steps=1, start_scale=2.5)
    x = s(model.prob, 200_000, seed=23)
    assert 0.2 < float(s.acceptance_rate) < 0.8
    _independent_normal(x)


def _truth_model(d, sampler, n_samples):
    """Screens of a correlated Gaussian truth well inside them, tables after one damped sample-mode sweep with a fine
    GridSampler (undamped sweeps in sample mode grow spikes at the screens' edges, islands a random walk from the
    bulk crosses slowly)."""
    gen = torch.Generator().manual_seed(40 + d)
    a = torch.randn(d, d, generator=gen) * 0.3 + torch.eye(d)
    truth = (torch.randn(400_000, d, generator=gen) @ a.T).cuda()
    tfs = [LinearTransform(_matrix(d, gen).cuda()) for _ in range(4)]
    e = torch.linspace(-6.0, 6.0, 49)
    diags = [[mf.diagnostics.Histogram1D(axis=i % d, edges=e, bandwidth=0.5).to("cuda")] for i in range(4)]
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    res = 256 if d == 2 else 64
    grid = mf.sample.GridSampler(limits=d * [(-6.0, 6.0)], shape=(res,) * d, device="cuda")
    model = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=d, scale=1.5), mode="sample", sampler=grid,
                         n_samples=1_000_000, device="cuda")
    torch.manual_seed(1)
    model.gauss_seidel_update(lr=0.5)
    model.sampler, model.n_samples = sampler, n_samples
    return model, grid


@pytest.mark.parametrize("d", [2, 3])
def test_profiles_agree_with_a_fine_grid_sampler(d):
    mh = MH(d, burnin=1000, steps=1, start_scale=1.0)
    model, grid = _truth_model(d, mh, 1_000_000)
    torch.manual_seed(2)
    x_mh = model.sample(1_000_000)
    p_mh = mf.simulate.forward(x_mh, model.transforms, model.diagnostics)
    x_grid = grid(model.prob, 1_000_000, seed=3)
    p_grid = mf.simulate.forward(x_grid, model.transforms, model.diagnostics)
    for a, b in zip(p_mh, p_grid):
        a, b = a[0].cpu(), b[0].cpu()
        assert float((a - b).abs().max()) < 0.04 * float(b.max()), float((a - b).abs().max() / b.max())


def test_sample_mode_sweeps_with_the_mh_sampler_lower_the_kl():
    mh = MH(2, burnin=200, steps=4, thin=5, start_scale=1.5)
    gen = torch.Generator().manual_seed(5)
    truth = (torch.randn(400_000, 2, generator=gen) @ torch.tensor([[1.0, 0.6], [0.0, 0.7]]).T).cuda()
    tfs = [LinearTransform(_matrix(2, gen).cuda()) for _ in range(4)]
    e = torch.linspace(-4.5, 4.5, 49)
    diags = [[mf.diagnostics.Histogram1D(axis=0, edges=e, bandwidth=0.5).to("cuda")] for _ in tfs]
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    model = mf.ment.MENT(ndim=2, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=2, scale=2.0), mode="sample", sampler=mh,
                         n_samples=1_000_000, device="cuda")
    torch.manual_seed(0)

    def mean_kl():
        pred = model.simulate_all()
        return float(np.mean([float(mf.loss.kl_divergence(p[0], m[0])) for p, m in zip(pred, model.measurements)]))

    kls = [mean_kl()]
    for _ in range(3):
        model.gauss_seidel_update(lr=1.0)
        kls.append(mean_kl())
    assert all(b < a for a, b in zip(kls, kls[1:])), kls
    assert kls[-1] < 0.5 * kls[0], kls


# ---------------------------------------------------------------------------------------------- edges
def test_a_start_outside_every_screen_reaches_the_support():
    """A chain at zero density random-walks: in 1-D it reaches the support at a rate that falls like 1 / sqrt(steps)
    (the share still outside after 5000 steps of sd 2 from 5 away is about 3 %), and never leaves it again."""
    model = _model(1, seed=13)
    start = torch.tensor([8.0])
    assert float(model.prob(start[None].cuda())) == 0.0
    s = MH(1, burnin=5000, steps=1, start=start, proposal_cov=[[4.0]])
    x = s(model.prob, 10_000, seed=5)
    assert float((model.prob(x) > 0).float().mean()) > 0.9
    assert torch.equal(x, s(lambda p: model.prob(p), 10_000, seed=5))


def test_zero_density_proposals_are_never_taken_from_positive_density():
    model = _model(3, seed=14)
    s = MH(3, burnin=0, steps=60, thin=1, start_scale=0.3)
    x = s(model.prob, 60 * 5000, seed=6)
    rho = model.prob(x).reshape(5000, 60)
    positive = rho > 0
    first = torch.where(positive.any(dim=1), positive.float().argmax(dim=1), torch.full((5000,), 60, device="cuda"))
    after = torch.arange(60, device="cuda")[None] >= first[:, None]
    assert bool(positive[after].all()) and float(positive[:, 0].float().mean()) > 0.5
    # a half-plane of zero density, through the step kernels
    half = MH(2, burnin=0, steps=100, start=torch.tensor([-1.0, 0.0]))
    y = half(lambda p: torch.where(p[:, 0] > 0, torch.zeros_like(p[:, 0]), torch.exp(-0.5 * (p * p).sum(dim=1))),
             100 * 2000, seed=7)
    assert float(y[:, 0].max()) <= 0.0 and 0.1 < float(half.acceptance_rate) < 0.9


@pytest.mark.parametrize("bad", [float("nan"), float("inf")])
def test_nan_and_inf_densities_are_rejected(bad):
    def prob(p):
        r = torch.exp(-0.5 * (p * p).sum(dim=1))
        return torch.where(p[:, 0].abs() > 1.0, torch.full_like(r, bad), r)

    s = MH(2, burnin=0, steps=80, start=torch.zeros(2))
    y = s(prob, 80 * 2000, seed=8)
    assert float(y[:, 0].abs().max()) <= 1.0 and torch.isfinite(y).all()
    assert 0.05 < float(s.acceptance_rate) < 0.95


def test_the_same_seed_gives_the_same_bits():
    model = _model(4, seed=15)
    s = MH(4, burnin=10, steps=3, thin=2)
    a, b, c = s(model.prob, 30_000, seed=1), s(model.prob, 30_000, seed=1), s(model.prob, 30_000, seed=2)
    assert torch.equal(a, b) and not torch.equal(a, c)
    torch.manual_seed(3)
    d = s(model.prob, 30_000)
    torch.manual_seed(3)
    assert torch.equal(d, s(model.prob, 30_000))


def test_size_zero_and_cuda_only():
    model = _model(2, seed=16)
    s = MH(2, burnin=3)
    x = s(model.prob, 0, seed=1)
    assert x.shape == (0, 2) and x.is_cuda
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mf.ops.mh_accept(torch.zeros(4, 2), torch.zeros(4), torch.zeros(4, 2).cuda(), torch.zeros(4).cuda(), 0, 1, 1,
                         torch.zeros(1, dtype=torch.int64).cuda())
