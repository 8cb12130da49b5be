"""k-NN entropy on the GPU (ops.knn_kth, entropy.KNNEntropyEstimator) against float64 references: scipy's cKDTree for
the distances, numpy for the tie rule, torch autograd in float64 for the gradient."""
import math

import numpy as np
import pytest
import scipy.spatial
import torch

import mentflow_b200 as mf
from mentflow_b200 import ops
from mentflow_b200.entropy import KNNEntropyEstimator, knn_entropy_constant

pytestmark = pytest.mark.gpu

KS = (1, 2, 5, 16)


def gaussian(n, d, seed):
    """n points of a Gaussian with a random covariance a^T a: scales in [0.5, 2] along random axes."""
    rng = np.random.default_rng(seed)
    rot, _ = np.linalg.qr(rng.normal(size=(d, d)))
    a = np.diag(rng.uniform(0.5, 2.0, size=d)) @ rot
    return (rng.normal(size=(n, d)) @ a).astype(np.float32), a


def scipy_neighbours(x, kmax):
    """float64 distances and indices of the kmax + 1 nearest OTHER particles, self removed by index."""
    n = x.shape[0]
    q = min(kmax + 2, n)
    dist, idx = scipy.spatial.cKDTree(x.astype(np.float64)).query(x.astype(np.float64), k=q, workers=-1)
    order = np.argsort(idx == np.arange(n)[:, None], axis=1, kind="stable")   # self (if listed) to the end
    dist, idx = np.take_along_axis(dist, order, 1)[:, :q - 1], np.take_along_axis(idx, order, 1)[:, :q - 1]
    return dist, idx


def neg_entropy_f64(r, n, d, k, pad=1e-12):
    return -(knn_entropy_constant(n, d, k) + d / n * float(np.sum(np.log(r.astype(np.float64) + pad))))


@pytest.mark.parametrize("n", [2, 3, 6, 17, 127, 128, 129, 1000, 25_000, 100_003])
@pytest.mark.parametrize("d", range(1, 9))
def test_kth_distance_and_index_match_kdtree(n, d):
    x, _ = gaussian(n, d, seed=n * 10 + d)
    dist, idx = scipy_neighbours(x, max(KS))
    xc = torch.from_numpy(x).cuda()
    for k in KS:
        if k >= n:
            continue
        r, nb, logsum = ops.knn_kth(xc, k)
        r, nb = r.cpu().numpy(), nb.cpu().numpy()
        want = dist[:, k - 1]
        np.testing.assert_allclose(r, want, rtol=2e-6, atol=0, err_msg=f"k={k}")
        # the index is pinned wherever the k-th distance is separated from its neighbours in rank
        sep = np.ones(n, dtype=bool)
        if k >= 2:
            sep &= dist[:, k - 1] - dist[:, k - 2] > 1e-5 * dist[:, k - 1]
        if k < dist.shape[1]:
            sep &= dist[:, k] - dist[:, k - 1] > 1e-5 * dist[:, k - 1]
        assert sep.mean() > 0.5
        np.testing.assert_array_equal(nb[sep], idx[sep, k - 1], err_msg=f"k={k}")
        assert abs(float(logsum) - float(np.sum(np.log(want + 1e-12)))) <= 1e-6 * n


@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("k", KS)
def test_lattice_ties_follow_distance_then_index(d, k):
    """Integer points: equal distances are exact, and a third of the points have duplicates."""
    rng = np.random.default_rng(100 + d * 20 + k)
    n = 1500
    x = rng.integers(0, 12 if d == 1 else 6, size=(n, d)).astype(np.int64)
    d2 = ((x[:, None, :] - x[None, :, :]) ** 2).sum(-1)
    key = d2 * n + np.arange(n)[None, :]
    np.fill_diagonal(key, np.iinfo(np.int64).max)
    kth = np.sort(key, axis=1)[:, k - 1]
    want_idx, want_r = kth % n, np.sqrt((kth // n).astype(np.float64)).astype(np.float32)
    r, nb, _ = ops.knn_kth(torch.from_numpy(x.astype(np.float32)).cuda(), k)
    np.testing.assert_array_equal(nb.cpu().numpy(), want_idx)
    np.testing.assert_array_equal(r.cpu().numpy(), want_r)


def grad_reference(x, nb, k, pad=1e-12, weight=1.0):
    """float64 autograd of weight * (-H) with the neighbour indices held fixed; w = 0 where r = 0 (no pair gradient)."""
    xr = torch.from_numpy(x).double().requires_grad_(True)
    n, d = x.shape
    diff = xr - xr[torch.from_numpy(nb).long()]
    r2 = (diff * diff).sum(1)
    zero = r2 == 0
    r = torch.sqrt(torch.where(zero, torch.ones_like(r2), r2))
    logs = torch.where(zero, torch.full_like(r2, math.log(pad)), torch.log(r + pad))
    h = -(knn_entropy_constant(n, d, k) + d / n * logs.sum())
    (weight * h).backward()
    return float(h.detach()), xr.grad.numpy()


def check_gradient(x, k):
    xc = torch.from_numpy(x).cuda().requires_grad_(True)
    h = KNNEntropyEstimator(k=k)(xc)
    assert h.dtype == torch.float32 and h.dim() == 0
    (2.5 * h).backward()
    nb = ops.knn_kth(xc.detach(), k)[1].cpu().numpy()
    href, gref = grad_reference(x, nb, k, weight=2.5)
    g = xc.grad.cpu().numpy().astype(np.float64)
    assert np.isfinite(g).all()
    assert abs(float(h) - href) <= 1e-5
    assert np.abs(g - gref).max() <= 1e-4 * np.abs(gref).max()
    return g, gref


@pytest.mark.parametrize("d", [2, 4, 6])
@pytest.mark.parametrize("k", [1, 5])
def test_gradient_matches_float64_autograd(d, k):
    x, _ = gaussian(5000, d, seed=7 + d + k)
    check_gradient(x, k)


def hubs(k, d, n_hubs, seed):
    """Every point of a hub's spokes has the hub as its k-th neighbour: spokes at distance ~1 along +-e_i, each with
    k - 1 satellites within 0.01, hubs 20 apart."""
    rng = np.random.default_rng(seed)
    pts = []
    for h in range(n_hubs):
        centre = np.zeros(d)
        centre[0] = 20.0 * h
        pts.append(centre)
        for axis in range(d):
            for sign in (1.0, -1.0):
                spoke = centre.copy()
                spoke[axis] += sign * (1.0 + 0.01 * rng.random())
                pts.append(spoke)
                for _ in range(k - 1):
                    pts.append(spoke + 0.005 * rng.normal(size=d) / math.sqrt(d))
    return np.asarray(pts, dtype=np.float32)


@pytest.mark.parametrize("k", [1, 5])
def test_gradient_of_a_hub_that_is_the_kth_neighbour_of_many(k):
    d = 6
    x = hubs(k, d, n_hubs=40, seed=k)
    nb = ops.knn_kth(torch.from_numpy(x).cuda(), k)[1].cpu().numpy()
    per_hub = 1 + 2 * d * k
    hub_of = (np.arange(x.shape[0]) // per_hub) * per_hub
    spokes = np.arange(x.shape[0]) != hub_of
    assert (nb[spokes] == hub_of[spokes]).all()          # each hub is the k-th neighbour of 2 d k particles
    check_gradient(x, k)


def test_duplicates_give_zero_distance_finite_estimate_and_no_pair_gradient():
    x, _ = gaussian(3000, 4, seed=5)
    x[1000:1100] = x[0:100]                              # 100 exact duplicate pairs
    xc = torch.from_numpy(x).cuda()
    r = ops.knn_kth(xc, 1)[0].cpu().numpy()
    assert (r[0:100] == 0).all() and (r[1000:1100] == 0).all() and (r[100:1000] > 0).all()
    check_gradient(x, 1)
    h = KNNEntropyEstimator(k=1)(xc)
    assert torch.isfinite(h)


@pytest.mark.parametrize("n,d,k", [(1000, 3, 1), (25_000, 6, 5), (100_003, 2, 16), (100_003, 8, 5)])
def test_estimate_matches_float64_formula(n, d, k):
    x, _ = gaussian(n, d, seed=3 * n + d)
    dist, _ = scipy_neighbours(x, k)
    h = KNNEntropyEstimator(k=k)(torch.from_numpy(x).cuda())
    assert abs(float(h) - neg_entropy_f64(dist[:, k - 1], n, d, k)) <= 1e-5


@pytest.mark.parametrize("d", [2, 4, 6])
def test_estimate_of_a_gaussian_is_close_to_its_entropy(d):
    x, a = gaussian(100_000, d, seed=40 + d)
    cov = a.T @ a
    analytic = 0.5 * (d * math.log(2.0 * math.pi * math.e) + math.log(np.linalg.det(cov)))
    h = -float(KNNEntropyEstimator(k=5)(torch.from_numpy(x).cuda()))
    assert abs(h - analytic) <= 0.1, (h, analytic)


def test_forward_and_backward_are_bitwise_reproducible():
    x, _ = gaussian(100_003, 6, seed=11)

    def run():
        xc = torch.from_numpy(x).cuda().requires_grad_(True)
        r, nb, logsum = ops.knn_kth(xc, 5)
        (logsum * 0.5).backward()
        return r, nb, logsum.detach(), xc.grad

    a, b = run(), run()
    for u, v in zip(a, b):
        assert torch.equal(u, v)


def _model(ndim, n_meas, k=5):
    from mentflow_b200 import workloads
    dev = torch.device("cuda")
    wl = workloads.isotropic_1d(ndim=ndim, num=n_meas, bins=48, xmax=3.5, seed=2)
    tfs = [mf.simulate.LinearTransform(m.to(dev)) for m in wl["matrices"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to(dev)
    diags = [[diag] for _ in tfs]
    truth = workloads.gaussian_mixture(50_000, ndim=ndim, seed=1, device=dev)
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    torch.manual_seed(5)
    gen = mf.generate.NSFGenerator(ndim).to(dev)
    return mf.MENTFlow(transforms=tfs, diagnostics=diags, measurements=meas, generator=gen, prior=None,
                       entropy_estimator=KNNEntropyEstimator(k=k), discrepancy_function=mf.loss.kl_divergence,
                       penalty_parameter=20.0)


def test_mentflow_loss_with_knn_entropy_reaches_the_flow_parameters():
    model = _model(4, 6)
    L, H, D = model.loss(10_000)
    assert torch.isfinite(L) and torch.isfinite(H)
    L.backward()
    grads = [p.grad for p in model.parameters()]
    assert all(g is not None and torch.isfinite(g).all() for g in grads)
    assert any(float(g.abs().max()) > 0 for g in grads)
    # the entropy term alone moves the parameters too
    model.generator.zero_grad(set_to_none=True)
    x, lq = model.sample_and_log_prob(10_000)
    model.entropy_estimator(x, lq).backward()
    assert any(p.grad is not None and float(p.grad.abs().max()) > 0 for p in model.parameters())


def test_graphed_loss_and_train_step_with_knn_entropy():
    from mentflow_b200.graphs import GraphedLoss, GraphedTrainStep
    model = _model(4, 6)
    gen, n = model.generator, 8192
    g = GraphedLoss(model, n)
    z = torch.randn(n, 4)
    L, H, D = g(z.pin_memory())
    with torch.no_grad():
        x, lq = gen.forward_and_log_prob(z.cuda())
        Le, He, De = model.loss_from_particles(x, lq)
    assert torch.equal(L, Le) and torch.equal(H, He) and torch.equal(torch.stack(D), torch.stack(De))

    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.0, capturable=True)
    step = GraphedTrainStep(model, opt, n)
    losses = [float(step()[0]) for _ in range(4)]
    assert all(math.isfinite(v) for v in losses) and bool(step.finite)
    assert all(torch.isfinite(p).all() for p in model.parameters())
