"""Sliced Wasserstein distance on the GPU (ops.swd_sort, ops.swd_wpp, loss.sliced_wasserstein_distance,
loss.SlicedWassersteinDistance) against float64 references: the fp32 projections replayed with mfb_testutil.fmaf and
numpy's stable argsort for the sort, the interval sum in float64 and scipy's 1-D Wasserstein distance for W_p^p, and
torch autograd in float64 through the interval formula for the gradient."""
import numpy as np
import pytest
import scipy.stats
import torch

from mentflow_b200 import loss, ops
from mfb_testutil import fmaf

pytestmark = pytest.mark.gpu


def directions(d, p, seed):
    return loss.random_projections(d, p, seed).t().float().contiguous().numpy()


def project(x, theta):
    """(P, N) fp32 projections: the kernels' fused multiply-add chain from zero, coordinates in ascending order."""
    u = np.zeros((theta.shape[0], x.shape[0]), np.float32)
    for c in range(x.shape[1]):
        u = fmaf(x[None, :, c], theta[:, c, None], u)
    return u


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def check_sort(x, theta):
    s, perm = ops.swd_sort(torch.from_numpy(x).cuda(), torch.from_numpy(theta).cuda())
    u = project(x, theta)
    want = np.argsort(u, axis=1, kind="stable")
    np.testing.assert_array_equal(perm.cpu().numpy(), want)
    np.testing.assert_array_equal(bits(s.cpu().numpy()), bits(np.take_along_axis(u, want, 1)))
    np.testing.assert_array_equal(s.cpu().numpy(), np.sort(u, axis=1))
    return u


# tiles hold 2048 keys
SORT_SIZES = [1, 2, 255, 256, 257, 2047, 2048, 2049, 4097, 100_003]


@pytest.mark.parametrize("n", SORT_SIZES)
@pytest.mark.parametrize("d", range(1, 9))
def test_sort_is_numpys_stable_sort(n, d):
    rng = np.random.default_rng(n * 10 + d)
    x = rng.normal(size=(n, d)).astype(np.float32)
    nproj = 257 if n <= 4097 else 3
    check_sort(x, directions(d, nproj, seed=d))
    if n <= 257:
        check_sort(x, directions(d, 1, seed=d + 100))


@pytest.mark.parametrize("d", [1, 6])
def test_sort_of_a_million(d):
    x = np.random.default_rng(d).normal(size=(1_000_000, d)).astype(np.float32)
    check_sort(x, directions(d, 1, seed=d))


@pytest.mark.parametrize("d", [1, 2, 3, 6, 8])
def test_sort_of_lattices_with_axis_directions_keeps_ties_in_index_order(d):
    """Integer points along the axes (and their negatives) give heavy exact ties; the points include -0.0 and +0.0."""
    rng = np.random.default_rng(40 + d)
    n = 30_011
    x = rng.integers(-3, 4, size=(n, d)).astype(np.float32)
    x[rng.random((n, d)) < 0.3] = -0.0
    theta = np.concatenate([np.eye(d), -np.eye(d), np.full((1, d), 0.5)]).astype(np.float32)
    u = check_sort(x, theta)
    assert len(np.unique(u[0])) <= 7


def interval_wpp(u, v, p):
    """float64 W_p^p of each row pair of sorted u (P, N) and v (P, M): the exact breakpoints i M and j N, in int64."""
    n, m = u.shape[1], v.shape[1]
    b = np.union1d(np.arange(n + 1, dtype=np.int64) * m, np.arange(m + 1, dtype=np.int64) * n)
    lens = np.diff(b).astype(np.float64)
    i, j = b[:-1] // m, b[:-1] // n
    diff = np.abs(u[:, i].astype(np.float64) - v[:, j].astype(np.float64))
    return (lens * diff ** p).sum(axis=1) / (float(n) * float(m))


WPP_SIZES = [(1, 1), (1, 1000), (1000, 1), (99_991, 100_003), (50_000, 1_000_000), (1_000_000, 50_000),
             (4097, 4097)]


@pytest.mark.parametrize("n,m", WPP_SIZES)
def test_wpp_matches_interval_sum_and_scipy(n, m):
    d, nproj = 3, 3
    rng = np.random.default_rng(n + 7 * m)
    x = rng.normal(size=(n, d)).astype(np.float32)
    y = (rng.normal(size=(m, d)) * 1.3 + 0.4).astype(np.float32)
    theta = torch.from_numpy(directions(d, nproj, seed=1)).cuda()
    xc, yc = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    us, _ = ops.swd_sort(xc, theta)
    vs, _ = ops.swd_sort(yc, theta)
    us, vsn = us.cpu().numpy(), vs.cpu().numpy()
    for p in (1.0, 1.5, 2.0, 3.0):
        got = ops.swd_wpp(xc, theta, vs, p).cpu().numpy()
        want = interval_wpp(us, vsn, p)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0, err_msg=f"p={p}")
        if p == 1.0:
            x64, y64, th64 = x.astype(np.float64), y.astype(np.float64), theta.cpu().double().numpy()
            for k in range(nproj):
                ux, uy = x64 @ th64[k], y64 @ th64[k]
                sp = scipy.stats.wasserstein_distance(ux, uy)
                # the kernels project in fp32: 2^-24 of the largest |u| on top of the relative tolerance
                assert abs(got[k] - sp) <= 1e-6 * sp + 6e-8 * max(abs(ux).max(), abs(uy).max()), (k, got[k], sp)


def swd_autograd_f64(x, y, theta, p):
    """The SWD and its gradient in float64 through the interval formula, with the fp32 projections' values and stable
    ranks (a sort's ranks held fixed: the derivative flows through x theta_k only)."""
    u32, v32 = project(x, theta), project(y, theta)
    pu, pv = np.argsort(u32, axis=1, kind="stable"), np.argsort(v32, axis=1, kind="stable")
    xt = torch.from_numpy(x.astype(np.float64)).requires_grad_(True)
    lin = torch.from_numpy(theta.astype(np.float64)) @ xt.t()                                 # (P, N)
    u = torch.from_numpy(u32.astype(np.float64)) + (lin - lin.detach())
    us = torch.gather(u, 1, torch.from_numpy(pu))
    vs = torch.from_numpy(np.take_along_axis(v32, pv, 1).astype(np.float64))
    n, m = x.shape[0], y.shape[0]
    b = np.union1d(np.arange(n + 1, dtype=np.int64) * m, np.arange(m + 1, dtype=np.int64) * n)
    lens = torch.from_numpy(np.diff(b).astype(np.float64))
    i, j = torch.from_numpy(b[:-1] // m), torch.from_numpy(b[:-1] // n)
    wpp = (lens * (us[:, i] - vs[:, j]).abs() ** p).sum(dim=1) / (float(n) * float(m))
    swd = wpp.mean() ** (1.0 / p)
    swd.backward()
    return float(swd.detach()), xt.grad.numpy()


@pytest.mark.parametrize("case", ["gauss", "ties", "coincide"])
@pytest.mark.parametrize("p", [1.0, 1.5, 2.0, 3.0])
def test_gradient_matches_float64_autograd(case, p):
    rng = np.random.default_rng(["gauss", "ties", "coincide"].index(case) * 10 + int(2 * p))
    d, n, m = 4, 3001, 2500
    if case == "gauss":
        x = rng.normal(size=(n, d)).astype(np.float32)
        y = (rng.normal(size=(m, d)) + 0.3).astype(np.float32)
        theta = directions(d, 7, seed=2)
    else:
        # integer lattices: exact ties inside x; with axis directions u_(i) = v_(j) exactly on many pairs
        x = rng.integers(-3, 4, size=(n, d)).astype(np.float32)
        y = rng.integers(-2, 5, size=(m, d)).astype(np.float32)
        theta = directions(d, 7, seed=2) if case == "ties" else \
            np.concatenate([np.eye(d), -np.eye(d)]).astype(np.float32)
    want_swd, want_g = swd_autograd_f64(x, y, theta, p)
    xc = torch.from_numpy(x).cuda().requires_grad_(True)
    got = loss.sliced_wasserstein_distance(xc, torch.from_numpy(y).cuda(), p=p,
                                           projections=torch.from_numpy(theta).t())
    got.backward()
    assert got.dtype == torch.float32 and got.dim() == 0
    assert abs(float(got.detach()) - want_swd) <= 2e-6 * want_swd
    g = xc.grad.cpu().numpy()
    assert np.abs(g - want_g).max() <= 1e-5 * np.abs(want_g).max()


def test_chunking_and_repeated_calls_are_bitwise_equal(monkeypatch):
    rng = np.random.default_rng(5)
    n, m, d, nproj = 20_011, 7_001, 6, 11
    x = torch.from_numpy(rng.normal(size=(n, d)).astype(np.float32)).cuda()
    y = torch.from_numpy(rng.normal(size=(m, d)).astype(np.float32)).cuda()
    proj = loss.random_projections(d, nproj, seed=3)

    def run():
        xg = x.clone().requires_grad_(True)
        s = loss.sliced_wasserstein_distance(xg, y, p=1.5, projections=proj)
        s.backward()
        theta = proj.t().float().contiguous().cuda()
        srt, perm = ops.swd_sort(y, theta)
        wpp = ops.swd_wpp(x, theta, srt, 2.0)
        return [t.cpu() for t in (s.detach(), xg.grad, srt, perm, wpp)]

    one = run()
    assert all(torch.equal(a, b) for a, b in zip(one, run()))
    lib = ops._lib.load()
    per = int(lib.mfb_swd_workspace_bytes(max(n, m), 1))
    monkeypatch.setattr(ops, "SWD_WORKSPACE_CAP", 3 * per)        # chunks of 3, 3, 3 and 2 directions
    chunked = run()
    for a, b in zip(one, chunked):
        assert torch.equal(a, b) if a.dtype != torch.float32 else torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_shifted_gaussians_approach_the_projected_shift():
    """W_2^2 of N(0, S) and N(delta, S) along theta is (theta . delta)^2; the sampling error of 1e6 samples is ~2e-3."""
    rng = np.random.default_rng(11)
    d, n, nproj = 6, 1_000_000, 50
    a = rng.normal(size=(d, d)) * 0.4 + np.eye(d)
    delta = rng.normal(size=d)
    delta *= 0.8 / np.linalg.norm(delta)
    x = torch.from_numpy((rng.normal(size=(n, d)) @ a).astype(np.float32)).cuda()
    y = torch.from_numpy((rng.normal(size=(n, d)) @ a + delta).astype(np.float32)).cuda()
    proj = loss.random_projections(d, nproj, seed=4)
    want = float(((proj.numpy().T @ delta) ** 2).mean())
    got = float(loss.sliced_wasserstein_distance(x, y, p=2, projections=proj)) ** 2
    assert abs(got - want) <= 5e-3 + 0.01 * want, (got, want)
    # same distribution: a small value that shrinks with N
    same = [float(loss.sliced_wasserstein_distance(x[:k], torch.from_numpy((rng.normal(size=(k, d)) @ a)
                                                                           .astype(np.float32)).cuda(),
                                                   projections=proj)) ** 2 for k in (10_000, n)]
    assert same[1] < same[0] and same[1] < 1e-4, same


def test_class_caches_the_sorted_reference_and_fixes_its_directions():
    rng = np.random.default_rng(12)
    d = 3
    y = torch.from_numpy(rng.normal(size=(20_000, d)).astype(np.float32)).cuda()
    est = loss.SlicedWassersteinDistance(y, n_projections=40, p=2, seed=9)
    assert est.theta.shape == (40, d)
    assert torch.equal(est.y_sorted, ops.swd_sort(y, est.theta)[0])
    assert torch.equal(est.theta, loss.SlicedWassersteinDistance(y, n_projections=40, seed=9).theta)
    assert torch.equal(est.theta.cpu(), loss.random_projections(d, 40, 9).t().float())
    proj = torch.randn(d, 17)
    est2 = loss.SlicedWassersteindDistance(y, projections=proj)
    assert torch.equal(est2.projections.cpu(), proj) and torch.equal(est2.theta.cpu(), proj.t())
    with pytest.raises(ValueError):
        est(torch.randn(100, d + 1, device="cuda"))

    # the class against the function under the same directions, and SGD on the samples lowers it
    x = torch.from_numpy((rng.normal(size=(20_000, d)) + np.array([1.0, -0.5, 0.25])).astype(np.float32)).cuda()
    x.requires_grad_(True)
    first = est(x)
    assert torch.equal(first, loss.sliced_wasserstein_distance(x.detach(), y, projections=est.projections))
    vals = []
    for _ in range(4):
        s = est(x)
        vals.append(float(s))
        x.grad = None
        s.backward()
        with torch.no_grad():
            x -= 0.25 * x.shape[0] * x.grad
    vals.append(float(est(x)))
    assert all(b < a for a, b in zip(vals, vals[1:])), vals
    assert vals[-1] < 0.7 * vals[0], vals


def test_non_finite_samples_give_nan_or_inf_and_leave_the_device_usable():
    rng = np.random.default_rng(13)
    d, n, m = 3, 5000, 4000
    x = rng.normal(size=(n, d)).astype(np.float32)
    y = torch.from_numpy(rng.normal(size=(m, d)).astype(np.float32)).cuda()
    proj = loss.random_projections(d, 5, seed=1)
    theta = proj.t().float().contiguous().cuda()
    ref = loss.sliced_wasserstein_distance(torch.from_numpy(x).cuda(), y, projections=proj)
    xn = x.copy()
    xn[17, 1] = np.nan
    xn[4000, 0] = -np.nan
    srt, perm = ops.swd_sort(torch.from_numpy(xn).cuda(), theta)
    perm = perm.cpu().numpy()
    assert np.array_equal(np.sort(perm, axis=1), np.broadcast_to(np.arange(n), perm.shape))
    assert np.array_equal(perm[:, -2:], np.broadcast_to([17, 4000], (5, 2)))     # NaN last, in index order
    assert np.isnan(srt.cpu().numpy()[:, -2:]).all()
    assert torch.isnan(loss.sliced_wasserstein_distance(torch.from_numpy(xn).cuda(), y, projections=proj))
    xi = x.copy()
    xi[5, :] = [np.inf, 0.0, 0.0]
    assert torch.isinf(loss.sliced_wasserstein_distance(torch.from_numpy(xi).cuda(), y, projections=proj, p=1))
    again = loss.sliced_wasserstein_distance(torch.from_numpy(x).cuda(), y, projections=proj)
    assert torch.equal(again, ref)
