"""k-NN entropy estimator: refusals raised before anything needs a GPU, and the estimator's constants."""
import math

import numpy as np
import pytest
import scipy.special
import torch

import mentflow_b200 as mf
from mentflow_b200 import ops
from mentflow_b200.entropy import KNNEntropyEstimator, knn_entropy_constant


def test_cpu_tensors_are_refused_without_fallback():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.knn_kth(torch.randn(100, 3), 5)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        KNNEntropyEstimator(k=5)(torch.randn(100, 3))


@pytest.mark.parametrize("n,d,k", [(100, 3, 0), (100, 3, -1), (100, 3, 17), (5, 3, 5), (5, 3, 6), (2, 1, 2),
                                   (100, 9, 5), (100, 0, 5)])
def test_bad_shapes_and_k_are_refused(n, d, k):
    x = torch.randn(n, d)
    with pytest.raises(ValueError):
        ops.knn_kth(x, k)
    with pytest.raises(ValueError):
        KNNEntropyEstimator(k=k)(x)


def test_non_matrix_input_is_refused():
    with pytest.raises(ValueError):
        ops.knn_kth(torch.randn(100), 5)


def test_prior_is_refused():
    with pytest.raises(ValueError):
        KNNEntropyEstimator(prior=mf.prior.Gaussian(ndim=2, scale=1.0))


class _Reducer:
    def __init__(self, world_size):
        self.world_size = world_size
        self.calls = 0

    def __call__(self, sums, n_local, **kw):
        self.calls += 1
        return n_local * self.world_size


def test_sharded_particles_are_refused_before_any_launch():
    est = KNNEntropyEstimator(k=5)
    est.reducer = _Reducer(world_size=2)
    # a CPU tensor: if the estimator reached ops, it would raise RuntimeError instead
    with pytest.raises(NotImplementedError, match="sharded"):
        est(torch.randn(100, 3))
    assert est.reducer.calls == 0
    est.reducer = _Reducer(world_size=1)       # one rank holds the whole batch: not refused for sharding
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        est(torch.randn(100, 3))


@pytest.mark.parametrize("n,k", [(n, k) for n in (2, 3, 9, 10, 11, 127, 1000, 25_000, 100_003, 10 ** 6)
                                 for k in (1, 2, 5, 16) if k < n])
def test_constant_matches_scipy(n, k):
    for d in range(1, 9):
        want = (scipy.special.digamma(n) - scipy.special.digamma(k)
                + 0.5 * d * np.log(np.pi) - scipy.special.gammaln(0.5 * d + 1.0))
        got = knn_entropy_constant(n, d, k)
        assert abs(got - want) <= 1e-13 * max(1.0, abs(want)), (n, d, k, got, want)


def test_unit_ball_volumes():
    for d, v in [(1, 2.0), (2, math.pi), (3, 4.0 * math.pi / 3.0), (6, math.pi ** 3 / 6.0)]:
        assert abs(knn_entropy_constant(7, d, 7 - 1) - (scipy.special.digamma(7) - scipy.special.digamma(6))
                   - math.log(v)) < 1e-14
