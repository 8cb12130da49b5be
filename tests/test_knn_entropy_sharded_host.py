"""k-NN entropy on sharded particles, the parts that need no GPU: the row-range C entry points and ops functions refuse
bad arguments before any launch, the estimator validates the union batch before it gathers anything, and a world-size-2
gloo run of ShardReducer.all_gather returns every rank's rows in rank order, for equal and unequal shards."""
import ctypes
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from mentflow_b200 import _lib, ops
from mentflow_b200 import distributed as mfd
from mentflow_b200.entropy import KNNEntropyEstimator

MFB_E_BADARG, MFB_E_UNSUPPORTED, MFB_E_WORKSPACE = -1, -2, -3


def test_c_entry_points_refuse_bad_arguments_before_any_launch():
    lib = _lib.load()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)

    def kth(n=100, d=3, k=5, row0=0, nrows=10, r=p, idx=p, ws=p):
        return lib.mfb_knn_kth_rows(p, n, d, k, row0, nrows, r, idx, ws, 0, None)

    def bwd(n=100, d=3, row0=0, nrows=10, gx=p):
        return lib.mfb_knn_kth_bwd_rows(p, n, d, p, p, p, p, row0, nrows, 1e-12, p, gx, None)

    for row0, nrows in [(-1, 10), (95, 10), (101, 0), (0, -1), (0, 101), (100, 1)]:
        assert kth(row0=row0, nrows=nrows) == MFB_E_BADARG, (row0, nrows)
        assert bwd(row0=row0, nrows=nrows) == MFB_E_BADARG, (row0, nrows)
    assert kth(n=16, k=16, nrows=2) == MFB_E_BADARG   # k >= n of the union
    assert kth(n=5, k=5, nrows=2) == MFB_E_BADARG
    assert kth(k=0) == MFB_E_BADARG
    assert kth(d=9) == MFB_E_UNSUPPORTED
    assert kth(k=17) == MFB_E_UNSUPPORTED
    assert kth(n=2 ** 31, nrows=0) == MFB_E_BADARG
    assert bwd(d=9) == MFB_E_UNSUPPORTED
    assert bwd(d=0) == MFB_E_BADARG
    assert bwd(n=2 ** 31, nrows=0) == MFB_E_BADARG
    assert kth(r=None) == MFB_E_BADARG and kth(idx=None) == MFB_E_BADARG and kth(ws=None) == MFB_E_BADARG
    assert bwd(gx=None) == MFB_E_BADARG
    assert lib.mfb_knn_kth_rows(None, 100, 3, 5, 0, 10, p, p, p, 0, None) == MFB_E_BADARG
    # an empty range (a rank without particles) launches nothing and succeeds, without outputs or a workspace
    for row0 in (0, 37, 100):
        assert kth(row0=row0, nrows=0, r=None, idx=None, ws=None) == 0
        assert bwd(row0=row0, nrows=0, gx=None) == 0
    assert lib.mfb_knn_rows_workspace_bytes(100, 0, 3, 5) == 0
    for bad in [(100, 10, 9, 5), (100, 10, 3, 17), (100, 10, 3, 100), (100, 101, 3, 5), (100, -1, 3, 5)]:
        assert lib.mfb_knn_rows_workspace_bytes(*bad) == 0, bad
    # the log sum: pointers, n and the workspace size are checked before the launch
    assert lib.mfb_knn_logsum(None, 100, 1e-12, p, p, 64, None) == MFB_E_BADARG
    assert lib.mfb_knn_logsum(p, 100, 1e-12, None, p, 64, None) == MFB_E_BADARG
    assert lib.mfb_knn_logsum(p, 100, 1e-12, p, None, 64, None) == MFB_E_BADARG
    assert lib.mfb_knn_logsum(p, 0, 1e-12, p, p, 64, None) == MFB_E_BADARG
    assert lib.mfb_knn_logsum(p, 2 ** 31, 1e-12, p, p, 2 ** 40, None) == MFB_E_BADARG
    assert lib.mfb_knn_logsum(p, 257, 1e-12, p, p, 8, None) == MFB_E_WORKSPACE      # needs two partials


@pytest.mark.parametrize("n,d,k,rows", [(100, 3, 5, slice(-1, 10)), (100, 3, 5, slice(95, 105)),
                                        (100, 3, 5, slice(0, 101)), (100, 3, 5, slice(10, 5)),
                                        (100, 3, 5, slice(0, 10, 2)), (16, 3, 16, slice(0, 10)),
                                        (100, 9, 5, slice(0, 10)), (100, 3, 17, slice(0, 10)),
                                        (100, 3, 0, slice(0, 10))])
def test_ops_refuse_bad_ranges_and_shapes_with_value_error(n, d, k, rows):
    x = torch.randn(n, d)          # a CPU tensor: reaching the library would raise RuntimeError instead
    with pytest.raises(ValueError):
        ops.knn_kth(x, k, rows=rows)
    if 1 <= d <= ops.KNN_MAX_DIM and not (rows.step is None and 0 <= rows.start <= rows.stop <= n):
        with pytest.raises(ValueError):
            ops.knn_kth_bwd(x, torch.zeros(n), torch.zeros(n, dtype=torch.int32), torch.ones((), dtype=torch.float64),
                            rows=rows)


def test_ops_log_sum_and_backward_refuse_bad_shapes():
    with pytest.raises(ValueError):
        ops.knn_logsum(torch.zeros(10, 2))
    with pytest.raises(ValueError):
        ops.knn_logsum(torch.zeros(0))
    g = torch.ones((), dtype=torch.float64)
    with pytest.raises(ValueError):
        ops.knn_kth_bwd(torch.zeros(10, 9), torch.zeros(10), torch.zeros(10, dtype=torch.int32), g)
    with pytest.raises(ValueError):
        ops.knn_kth_bwd(torch.zeros(10, 3), torch.zeros(9), torch.zeros(10, dtype=torch.int32), g)
    with pytest.raises(ValueError):
        ops.knn_kth_bwd(torch.zeros(10, 3), torch.zeros(10), torch.zeros(10, dtype=torch.int64), g)
    with pytest.raises(RuntimeError, match="no CPU fallback"):      # valid arguments reach the device check
        ops.knn_kth(torch.randn(100, 3), 5, rows=slice(10, 20))


def test_backward_refuses_tensors_on_different_devices():
    # a meta-device x stands for a CUDA x here: the check compares devices before anything is launched or sorted
    x = torch.empty(10, 3, device="meta")
    g = torch.ones((), dtype=torch.float64)
    r, idx = torch.zeros(10), torch.zeros(10, dtype=torch.int32)
    for rr, ii in [(r, idx), (r.to("meta"), idx), (r, idx.to("meta"))]:
        with pytest.raises(ValueError, match="one device"):
            ops.knn_kth_bwd(x, rr, ii, g)
        with pytest.raises(ValueError, match="one device"):
            ops.knn_kth_bwd(x, rr, ii, g, rows=slice(2, 5))


class _GatherReducer:
    """A reducer of `world` equal shards that records what it is asked to do."""

    def __init__(self, world, rank=0, equal_shards=True):
        self.world_size, self.rank, self.equal_shards = world, rank, equal_shards
        self.gathers = 0

    def shard_counts(self, n_local, device=None):
        return [int(n_local)] * self.world_size

    def all_gather(self, tensor, counts=None):
        self.gathers += 1
        return torch.cat([tensor] * self.world_size)


def test_sharded_estimator_validates_the_union_before_gathering():
    est = KNNEntropyEstimator(k=5)
    est.reducer = _GatherReducer(world=2)
    # 3 + 3 particles: k = 5 < 6 is valid for the union although each shard alone is too small
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        est(torch.randn(3, 3))
    for x, k in [(torch.randn(2, 3), 5), (torch.randn(50, 9), 5), (torch.randn(50, 3), 17)]:
        est = KNNEntropyEstimator(k=k)
        est.reducer = _GatherReducer(world=2)
        with pytest.raises(ValueError):
            est(x)
        assert est.reducer.gathers == 0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rows(rank, n, d=0):
    """rank-tagged rows: entry (i, c) = 1000 rank + 10 i + c"""
    base = 1000.0 * rank + 10.0 * torch.arange(n, dtype=torch.float64)
    return base if d == 0 else base[:, None] + torch.arange(d, dtype=torch.float64)[None, :]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ok = []
        # equal shards: one all_gather_into_tensor, rank-major
        red = mfd.ShardReducer(equal_shards=True)
        ok.append(red.rank == rank and red.shard_counts(4) == [4, 4])
        for d, dtype in [(3, torch.float32), (0, torch.float32), (0, torch.int32)]:
            got = red.all_gather(_rows(rank, 4, d).to(dtype))
            want = torch.cat([_rows(q, 4, d) for q in range(world)]).to(dtype)
            ok.append(got.dtype == dtype and torch.equal(got, want))
        # unequal shards: counts gathered (or given), rows padded to the largest count, padding dropped
        red = mfd.ShardReducer(equal_shards=False)
        sizes = [5, 2]
        ok.append(red.shard_counts(sizes[rank]) == sizes)
        for d, dtype in [(3, torch.float32), (0, torch.int32)]:
            want = torch.cat([_rows(q, sizes[q], d) for q in range(world)]).to(dtype)
            ok.append(torch.equal(red.all_gather(_rows(rank, sizes[rank], d).to(dtype)), want))
            ok.append(torch.equal(red.all_gather(_rows(rank, sizes[rank], d).to(dtype), sizes), want))
        empty = [3, 0]                     # a rank without particles
        want = torch.cat([_rows(q, empty[q], 2) for q in range(world)]).float()
        ok.append(torch.equal(red.all_gather(_rows(rank, empty[rank], 2).float()), want))
        out.put((rank, ok))
    finally:
        dist.destroy_process_group()


def test_all_gather_is_rank_major_for_equal_and_unequal_shards():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    results = dict(out.get(timeout=10) for _ in procs)
    for rank in range(2):
        assert all(results[rank]), (rank, results[rank])


def test_one_rank_gathers_nothing():
    red = mfd.ShardReducer()
    x = torch.randn(7, 3)
    assert red.all_gather(x) is x
    assert red.shard_counts(7) == [7] and red.rank == 0
