"""k-NN entropy on sharded particles, with R ranks emulated on one device: the row-range search, the log sum of the
gathered r, the row-range backward and the sharded estimator must reproduce the whole-batch results bit for bit.

A rank's rows are searched against the union batch, so its neighbours, distances and gradient rows are those of one
GPU, whatever the shard boundaries; the log sum of the gathered r is added in the single-GPU order."""
import numpy as np
import pytest
import torch

from mentflow_b200 import ops
from mentflow_b200.distributed import shard_slice, shard_sizes
from mentflow_b200.entropy import KNNEntropyEstimator

pytestmark = pytest.mark.gpu


def gaussian(n, d, seed):
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.normal(size=(n, d)).astype(np.float32)).cuda()


def cuts_of(n, world):
    return [shard_slice(n, r, world) for r in range(world)]


def slices_at(n, bounds):
    edges = [0] + list(bounds) + [n]
    return [slice(a, b) for a, b in zip(edges[:-1], edges[1:])]


def check_rows(x, k, slices, pad=1e-12):
    """r, idx of every row range, concatenated, and the log sum of the concatenated r: bitwise the whole batch"""
    r, idx, logsum = ops.knn_kth(x, k, pad)
    parts = [ops.knn_kth(x, k, pad, rows=sl) for sl in slices]
    for sl, (rp, ip, none) in zip(slices, parts):
        assert none is None and rp.shape == (sl.stop - sl.start,) and ip.dtype == torch.int32
    rc = torch.cat([p[0] for p in parts])
    ic = torch.cat([p[1] for p in parts])
    assert torch.equal(rc, r) and torch.equal(ic, idx)
    ls = ops.knn_logsum(rc, pad)
    assert ls.dtype == torch.float64 and torch.equal(ls, logsum)
    return r, idx, logsum


@pytest.mark.parametrize("d", [1, 2, 6, 8])
@pytest.mark.parametrize("k", [1, 5, 16])
def test_rows_concatenate_to_the_whole_batch(d, k):
    for n in (k + 1, 1000, 25_000, 100_003):
        x = gaussian(n, d, seed=n + 10 * d + k)
        for world in (2, 3, 8):
            check_rows(x, k, cuts_of(n, world))


def test_boundaries_inside_a_query_block_and_a_candidate_tile():
    n = 3000
    x = gaussian(n, 6, seed=1)
    # 300: inside the first 512-query block and the second 256-candidate tile; 700, 1111: inside later ones;
    # 1024: on a block boundary; 2999: one row left
    for bounds in ([300], [128, 300, 700], [700, 1111, 1900], [1024, 2999], [1, 2, 3, 511, 513]):
        for k in (1, 5, 16):
            check_rows(x, k, slices_at(n, bounds))


def test_empty_shards():
    n = 10
    x = gaussian(n, 3, seed=2)
    slices = cuts_of(n, 16)
    assert shard_sizes(n, 16).count(0) == 6
    for k in (1, 5, 9):
        check_rows(x, k, slices)
    r, idx, none = ops.knn_kth(x, 5, rows=slice(10, 10))
    assert r.numel() == 0 and idx.numel() == 0 and none is None
    gx = ops.knn_kth_bwd(x, *ops.knn_kth(x, 5)[:2], torch.ones((), dtype=torch.float64, device="cuda"),
                         rows=slice(4, 4))
    assert gx.shape == (0, 3)


@pytest.mark.parametrize("d", [1, 2, 3])
def test_lattice_ties_decided_across_shards(d):
    """Integer points: equal distances are exact, so the (r^2, j) tie rule decides between neighbours that sit in
    other shards than the query."""
    rng = np.random.default_rng(300 + d)
    n = 1500
    xi = rng.integers(0, 12 if d == 1 else 6, size=(n, d)).astype(np.int64)
    x = torch.from_numpy(xi.astype(np.float32)).cuda()
    d2 = ((xi[:, None, :] - xi[None, :, :]) ** 2).sum(-1)
    key = d2 * n + np.arange(n)[None, :]
    np.fill_diagonal(key, np.iinfo(np.int64).max)
    for k in (1, 5, 16):
        kth = np.sort(key, axis=1)[:, k - 1]
        for slices in (cuts_of(n, 3), cuts_of(n, 8), slices_at(n, [137, 800])):
            r, idx, _ = check_rows(x, k, slices)
            np.testing.assert_array_equal(idx.cpu().numpy(), kth % n)
            np.testing.assert_array_equal(r.cpu().numpy(), np.sqrt((kth // n).astype(np.float64)).astype(np.float32))


def test_duplicates_split_across_shards():
    x = gaussian(3000, 4, seed=5)
    x[1000:1100] = x[0:100]
    for slices in (cuts_of(3000, 2), cuts_of(3000, 8), slices_at(3000, [50, 1050])):
        r, idx, _ = check_rows(x, 1, slices)
        assert (r[0:100] == 0).all() and (r[1000:1100] == 0).all()


def test_nan_and_inf_rows_in_one_shard():
    n = 4000
    x = gaussian(n, 3, seed=6)
    bad = [2100, 2101, 2500, 2999]
    x[2100, 0] = float("nan")
    x[2101] = float("inf")
    x[2500, 2] = -float("inf")
    x[2999, 1] = float("nan")
    for world in (2, 4):
        for k in (1, 5):
            r, idx, logsum = check_rows(x, k, cuts_of(n, world))
            assert torch.isinf(r[bad]).all()
            assert torch.equal(idx[bad].long().cpu(), torch.tensor(bad))


def whole_batch_grad(x, k, g, pad=1e-12):
    xc = x.clone().requires_grad_(True)
    r, idx, logsum = ops.knn_kth(xc, k, pad)
    logsum.backward(torch.tensor(g, dtype=torch.float64, device=x.device))
    return r, idx, xc.grad


@pytest.mark.parametrize("d", [1, 3, 6, 8])
@pytest.mark.parametrize("k", [1, 5, 16])
def test_backward_rows_equal_the_whole_batch_gradient(d, k):
    n = 25_000
    x = gaussian(n, d, seed=50 + d + k)
    x[7000:7050] = x[100:150]                     # pairs at distance 0: no pair gradient
    for g in (1.0, 2.0 ** -7, 0.7368421052631579):
        r, idx, gx = whole_batch_grad(x, k, g)
        gt = torch.tensor(g, dtype=torch.float64, device="cuda")
        assert torch.equal(ops.knn_kth_bwd(x, r, idx, gt), gx)          # the full range
        for slices in (cuts_of(n, 3), cuts_of(n, 8), slices_at(n, [300, 701, 24_999])):
            got = torch.cat([ops.knn_kth_bwd(x, r, idx, gt, rows=sl) for sl in slices])
            assert torch.equal(got, gx), (g, slices)


def test_backward_refuses_r_or_idx_off_the_device_of_x():
    x = gaussian(1000, 3, seed=12)
    r, idx, _ = ops.knn_kth(x, 5)
    g = torch.ones((), dtype=torch.float64, device="cuda")
    for rr, ii in [(r, idx.cpu()), (r.cpu(), idx), (r.cpu(), idx.cpu())]:
        with pytest.raises(ValueError, match="one device"):
            ops.knn_kth_bwd(x, rr, ii, g, rows=slice(0, 500))


def test_full_range_equals_knn_kth():
    x = gaussian(100_003, 6, seed=9)
    r, idx, _ = ops.knn_kth(x, 5)
    for rows in (slice(None), slice(0, 100_003), slice(0, None)):
        rr, ii, none = ops.knn_kth(x, 5, rows=rows)
        assert none is None and torch.equal(rr, r) and torch.equal(ii, idx)


class EmulatedReducer:
    """One rank of a group whose other ranks' gathers were computed beforehand: all_gather returns the precomputed
    pieces with this rank's live tensor in its slot.  The estimator gathers x, then r, then idx."""

    def __init__(self, rank, pieces, equal_shards):
        self.rank, self.world_size, self.equal_shards = rank, len(pieces["x"]), equal_shards
        self.pieces = pieces
        self.calls = []

    def shard_counts(self, n_local, device=None):
        counts = [p.shape[0] for p in self.pieces["x"]]
        assert counts[self.rank] == n_local
        return counts

    def all_gather(self, tensor, counts=None):
        key = "x" if tensor.dim() == 2 else ("idx" if tensor.dtype == torch.int32 else "r")
        self.calls.append(key)
        parts = list(self.pieces[key])
        assert parts[self.rank].shape == tensor.shape and parts[self.rank].dtype == tensor.dtype
        parts[self.rank] = tensor
        return torch.cat(parts)


@pytest.mark.parametrize("n,d,k,world", [(24_000, 6, 5, 2), (24_000, 6, 5, 3), (24_000, 6, 5, 8), (1000, 2, 1, 4),
                                         (100_003, 6, 5, 3), (25_000, 8, 16, 8), (6, 3, 5, 2), (10, 2, 5, 16)])
def test_estimator_on_emulated_ranks_is_the_single_gpu_estimator(n, d, k, world):
    x = gaussian(n, d, seed=n + d)
    equal = n % world == 0
    xg = x.clone().requires_grad_(True)
    est = KNNEntropyEstimator(k=k)
    h_ref = est(xg)
    (3.0 * h_ref).backward()
    g_ref = xg.grad
    slices = cuts_of(n, world)
    rows = [ops.knn_kth(x, k, rows=sl) for sl in slices]
    pieces = {"x": [x[sl] for sl in slices], "r": [p[0] for p in rows], "idx": [p[1] for p in rows]}
    for rank, sl in enumerate(slices):
        est = KNNEntropyEstimator(k=k)
        est.reducer = EmulatedReducer(rank, pieces, equal_shards=equal)
        xl = x[sl].clone().requires_grad_(True)
        if equal:
            torch.cuda.synchronize()
            torch.cuda.set_sync_debug_mode("error")       # the equal-shard forward never waits for the device
            try:
                h = est(xl)
            finally:
                torch.cuda.set_sync_debug_mode("default")
        else:
            h = est(xl)
        assert est.reducer.calls == ["x", "r", "idx"]
        assert h.dtype == torch.float32 and torch.equal(h, h_ref), (rank, float(h), float(h_ref))
        (3.0 * h).backward()
        if xl.shape[0]:
            assert torch.equal(xl.grad, g_ref[sl]), rank
        else:
            assert xl.grad is None or xl.grad.numel() == 0
