"""k-NN neighbour search at its edges: exact ties across a split candidate axis, and particles without k neighbours at
a finite distance (NaN, inf, or coordinates whose squared distances overflow)."""
import math

import numpy as np
import pytest
import torch

from mentflow_b200 import _lib, ops

pytestmark = pytest.mark.gpu

KS = (1, 2, 5, 16)


def candidate_splits(n, d, k):
    """Number of candidate-axis splits the library plans, read back from the workspace size:
    d Npad floats + two lists of splits * k * n 4-byte entries (each rounded to 16 bytes) + one double per 256 rows."""
    npad = -(-n // 256) * 256
    lists = (int(_lib.load().mfb_knn_workspace_bytes(n, n, d, k)) - d * npad * 4 - (-(-n // 256)) * 8) // 2
    return lists // (k * n * 4)


@pytest.mark.parametrize("d,side", [(1, 2400), (2, 110), (3, 23)])
def test_lattice_ties_across_the_planned_candidate_splits(d, side):
    """12,000 integer points at about one per cell: equal distances are exact and the tied candidates of a query lie
    in every split of the candidate axis, so the merge of the splits decides them."""
    rng = np.random.default_rng(7 + d)
    n = 12_000
    x = rng.integers(0, side, size=(n, d)).astype(np.int64)
    assert all(candidate_splits(n, d, k) >= 2 for k in KS)
    want = {k: np.empty(n, dtype=np.int64) for k in KS}
    cols = np.arange(n)
    for lo in range(0, n, 1000):
        rows = slice(lo, min(lo + 1000, n))
        d2 = sum((x[rows, c, None] - x[None, :, c]) ** 2 for c in range(d))
        key = d2 * n + cols[None, :]
        key[np.arange(key.shape[0]), cols[rows]] = np.iinfo(np.int64).max
        part = np.partition(key, [k - 1 for k in KS], axis=1)
        for k in KS:
            want[k][rows] = part[:, k - 1]
    xc = torch.from_numpy(x.astype(np.float32)).cuda()
    for k in KS:
        r, nb, _ = ops.knn_kth(xc, k)
        np.testing.assert_array_equal(nb.cpu().numpy(), want[k] % n, err_msg=f"k={k}")
        np.testing.assert_array_equal(r.cpu().numpy(), np.sqrt((want[k] // n).astype(np.float64)).astype(np.float32))


def logsum_grad_f64(x, nb, pad=1e-12):
    xr = torch.from_numpy(x).double().requires_grad_(True)
    diff = xr - xr[torch.from_numpy(nb).long()]
    torch.log(torch.sqrt((diff * diff).sum(1)) + pad).sum().backward()
    return xr.grad.numpy()


@pytest.mark.parametrize("k", [1, 5])
def test_particles_without_finite_neighbours_point_at_themselves(k):
    rng = np.random.default_rng(k)
    n, d = 5000, 4
    x = rng.normal(size=(n, d)).astype(np.float32)
    bad = np.array([10, 777, 2500, 4999])
    x[10] = np.nan
    x[777, 2] = np.nan
    x[2500, 0] = np.inf
    x[4999] = 1e30                                   # finite, but every squared distance overflows
    xc = torch.from_numpy(x).cuda().requires_grad_(True)
    r, nb, logsum = ops.knn_kth(xc, k)
    logsum.backward()
    r, nb, g = r.cpu().numpy(), nb.cpu().numpy(), xc.grad.cpu().numpy().astype(np.float64)
    assert ((nb >= 0) & (nb < n)).all()
    np.testing.assert_array_equal(nb[bad], bad)
    assert np.isposinf(r[bad]).all() and math.isinf(float(logsum.detach()))
    assert (g[4999] == 0).all()
    # the finite particles see exactly the search over the finite ones, and get their gradient
    good = np.setdiff1d(np.arange(n), bad)
    rf, nbf, _ = ops.knn_kth(torch.from_numpy(x[good]).cuda(), k)
    np.testing.assert_array_equal(r[good], rf.cpu().numpy())
    np.testing.assert_array_equal(nb[good], good[nbf.cpu().numpy()])
    gref = logsum_grad_f64(x[good], nbf.cpu().numpy())
    assert np.isfinite(g[good]).all()
    assert np.abs(g[good] - gref).max() <= 1e-4 * np.abs(gref).max()
