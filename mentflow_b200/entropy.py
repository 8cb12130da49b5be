"""Negative-entropy estimators (mentflow/entropy.py).

``MonteCarloEntropyEstimator`` is one fused, deterministic double-precision reduction over
the particles (sum log q and sum |x|^2 in one pass) instead of a MultivariateNormal
triangular solve plus two means."""
import math
from typing import Any

import numpy as np
import torch

from . import ops
from .prior import Gaussian


class _MCEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, log_prob, inv_s2, log_norm, reducer):
        m = ops.moments(x.detach(), log_prob.detach(), with_cov=False)
        n = float(x.shape[0])
        if reducer is not None:
            n = reducer(m, n)
        ctx.save_for_backward(x)
        ctx.inv_s2, ctx.n = inv_s2, n
        # H = mean(log q) - mean(log prior),  log prior = -0.5 |x|^2 / s^2 + log_norm
        return ops.mc_entropy(m, 1.0 / n, 0.5 * inv_s2 / n, log_norm)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        gl = (g / ctx.n).expand(x.shape[0])
        gx = x * (g * (ctx.inv_s2 / ctx.n)) if ctx.inv_s2 != 0.0 else None
        return gx, gl, None, None, None


class _MCEntropyFromSums(torch.autograd.Function):
    """the same estimator from moment sums that were reduced elsewhere (packed all-reduce)"""

    @staticmethod
    def forward(ctx, x, log_prob, m, inv_s2, log_norm, n):
        ctx.save_for_backward(x)
        ctx.inv_s2, ctx.n = inv_s2, n
        return ops.mc_entropy(m, 1.0 / n, 0.5 * inv_s2 / n, log_norm)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        gl = (g / ctx.n).expand(x.shape[0])
        gx = x * (g * (ctx.inv_s2 / ctx.n)) if ctx.inv_s2 != 0.0 else None
        return gx, gl, None, None, None, None


class EntropyEstimator(torch.nn.Module):
    """Estimates negative entropy from samples and/or log probability (entropy.py:8-15)."""

    def __init__(self, prior: Any = None) -> None:
        super().__init__()
        self.prior = prior
        self.reducer = None

    def forward(self, x: torch.Tensor, log_prob: torch.Tensor = None) -> torch.Tensor:
        raise NotImplementedError


class EmptyEntropyEstimator(EntropyEstimator):
    def forward(self, x: torch.Tensor, log_prob: torch.Tensor = None) -> torch.Tensor:
        return 0.0


class MonteCarloEntropyEstimator(EntropyEstimator):
    """H = mean(log q) - mean(log prior(x))  (entropy.py:53-62)."""

    def forward(self, x: torch.Tensor, log_prob: torch.Tensor) -> torch.Tensor:
        if log_prob is None:
            raise ValueError("MonteCarloEntropyEstimator needs the generator's log-density, and this generator has "
                             "none (log_prob is None): use CovarianceEntropyEstimator, KNNEntropyEstimator or "
                             "EmptyEntropyEstimator, which work from the particles alone")
        if self.prior is None:
            return _MCEntropy.apply(x, log_prob, 0.0, 0.0, self.reducer)
        if isinstance(self.prior, Gaussian):
            return _MCEntropy.apply(x, log_prob, 1.0 / self.prior.scale ** 2, self.prior.log_norm, self.reducer)
        # arbitrary prior object: same estimator, prior evaluated by the caller's code
        h = _MCEntropy.apply(x, log_prob, 0.0, 0.0, self.reducer)
        return h - torch.mean(self.prior.log_prob(x))

    # ---- sharded particles: the two moment sums ride on the all-reduce of the profile sums ------------
    def begin(self, x: torch.Tensor, log_prob: torch.Tensor):
        """Compute the local sums and leave them on the reducer; None if this configuration cannot defer
        (no reducer, unequal shards, a prior evaluated by foreign code)."""
        red = self.reducer
        if (log_prob is None or red is None or not hasattr(red, "stash") or red.world_size == 1
                or red.global_count(x.shape[0]) is None
                or not (self.prior is None or isinstance(self.prior, Gaussian))):
            return None
        m = ops.moments(x.detach(), log_prob.detach(), with_cov=False)
        red.stash(m)
        return (x, log_prob, m)

    def finish(self, pending) -> torch.Tensor:
        x, log_prob, m = pending
        red = self.reducer
        n = red.global_count(x.shape[0])
        reduced = red.pop_result()
        if reduced is None:            # nothing carried the sums: reduce them now
            red._stash = None
            red(m, float(x.shape[0]))
            reduced = m
        inv_s2, log_norm = (0.0, 0.0) if self.prior is None else (1.0 / self.prior.scale ** 2, self.prior.log_norm)
        return _MCEntropyFromSums.apply(x, log_prob, reduced, inv_s2, log_norm, n)


class _CovEntropy(torch.autograd.Function):
    """H = c - log(sqrt(det S) + pad), S = unbiased covariance of the particles (entropy.py:27-38).

    Forward: one pass of the moments kernel (float64 sums of x_i and x_i x_j), a D x D determinant.
    Backward in closed form: d log det S / dx_n = 2 S^-1 (x_n - mean) / (n - 1), hence
    dH/dx_n = -eps / (eps + pad) * S^-1 (x_n - mean) / (n - 1), eps = sqrt(det S) -- what torch autograd
    derives through torch.cov / torch.det in the reference."""

    @staticmethod
    def forward(ctx, x, pad, const, reducer):
        n_local, d = x.shape
        m = ops.moments(x.detach(), None, with_cov=True)
        n = float(n_local)
        if reducer is not None:
            n = reducer(m, n)
        mean = m[2:2 + d] / n
        second = m[2 + d:].reshape(d, d) / n
        cov = (second - torch.outer(mean, mean)) * (n / (n - 1.0))
        eps = torch.sqrt(torch.det(cov))
        ctx.save_for_backward(x, mean, cov, eps)
        ctx.pad, ctx.n = pad, n
        return (const - torch.log(eps + pad)).to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        x, mean, cov, eps = ctx.saved_tensors
        scale = -(eps / (eps + ctx.pad)) / (ctx.n - 1.0) * g.double()
        # inv_ex: the same inverse without the error check's host sync, so a CUDA graph can capture the backward
        a = (torch.linalg.inv_ex(cov)[0] * scale).to(torch.float32)    # symmetric D x D
        gx = torch.addmm(-(mean.to(torch.float32) @ a)[None, :], x, a)  # (x - mean) @ a
        return gx, None, None, None


class CovarianceEntropyEstimator(EntropyEstimator):
    """-3 log(2 pi e) - log(sqrt(det cov) + pad)  (entropy.py:27-38; the constant is the
    reference's, hard-coded for six dimensions).  The covariance comes from the moments kernel
    (all-reduced over ranks when the model is sharded); differentiable w.r.t. the particles like the
    reference's torch.cov / torch.det expression."""

    def __init__(self, prior: Any = None, pad: float = 1.0e-12) -> None:
        if prior is not None:
            raise ValueError("This class cannot estimate relative entropy (prior != None).")
        super().__init__(prior=prior)
        self.pad = pad

    def forward(self, x: torch.Tensor, log_prob: torch.Tensor = None) -> torch.Tensor:
        return _CovEntropy.apply(x, float(self.pad), -3.0 * float(np.log(2.0 * np.pi * np.e)), self.reducer)


def _digamma_int(n: int) -> float:
    """psi(n) for an integer n >= 1: the harmonic sum below 10, the asymptotic series (error < 1e-16) above."""
    if n < 10:
        return -0.5772156649015329 + sum(1.0 / m for m in range(1, n))
    x = float(n)
    x2 = 1.0 / (x * x)
    return math.log(x) - 0.5 / x - x2 * (1.0 / 12 - x2 * (1.0 / 120 - x2 * (1.0 / 252 - x2 * (1.0 / 240 - x2 / 132))))


def knn_entropy_constant(n: int, d: int, k: int) -> float:
    """psi(N) - psi(k) + log V_d, V_d = pi^(d/2) / Gamma(d/2 + 1) the volume of the unit d-ball."""
    log_vd = 0.5 * d * math.log(math.pi) - math.lgamma(0.5 * d + 1.0)
    return _digamma_int(n) - _digamma_int(k) + log_vd


class _ShardedKNNLogsum(torch.autograd.Function):
    """sum log(r_i + pad) over the union batch of a sharded model, from this rank's particles ``x``: all-gather the
    particles, search this rank's rows against the union, all-gather r and idx, and add the logs over the union in the
    single-GPU order.  Every rank gets the log sum one GPU computes on the union, bit for bit.  The backward needs no
    exchange: a particle's gradient is its own term plus those of the particles whose k-th neighbour it is, and all of
    them are in the gathered tensors, so each rank runs the gradient kernel for its own rows."""

    @staticmethod
    def forward(ctx, x, k, pad, reducer, counts, row0):
        rows = slice(row0, row0 + x.shape[0])
        xu = reducer.all_gather(x.detach(), counts)
        r_rows, idx_rows, _ = ops.knn_kth(xu, k, pad, rows=rows)
        r = reducer.all_gather(r_rows, counts)
        idx = reducer.all_gather(idx_rows, counts)
        ctx.save_for_backward(xu, r, idx)
        ctx.pad, ctx.rows = pad, rows
        return ops.knn_logsum(r, pad)

    @staticmethod
    def backward(ctx, glogsum):
        xu, r, idx = ctx.saved_tensors
        return ops.knn_kth_bwd(xu, r, idx, glogsum, ctx.pad, rows=ctx.rows), None, None, None, None, None


class KNNEntropyEstimator(EntropyEstimator):
    """-H, H = psi(N) - psi(k) + log V_d + (d/N) sum_i log(r_i + pad), r_i the distance from x_i to its k-th nearest
    other particle (Kozachenko-Leonenko).  Works from the particles alone: ``log_prob`` is ignored.  The distances come
    from an all-pairs CUDA kernel (O(N^2 d), ops.knn_kth); the gradient holds the neighbours fixed, as autograd
    through cdist + topk would.

    Sharded particles (``distributed.shard_model``): N is the union of all ranks' particles, and every rank returns
    the -H one GPU computes on the union, bit for bit.  Each rank all-gathers the particles, searches its own rows
    against the union (a 1 / ranks share of the pair work), and all-gathers r and the neighbour indices; its backward
    gives the gradient of its own particles without further exchange.  With equal shards nothing synchronises with the
    host, so ``GraphedLoss`` captures it.  The reducer must offer ``all_gather``, ``shard_counts`` and ``rank`` (as
    ``distributed.ShardReducer`` does); a reducer without ``all_gather`` is refused, because the neighbours within one
    shard are not those within the union."""

    def __init__(self, prior: Any = None, k: int = 5, pad: float = 1.0e-12) -> None:
        if prior is not None:
            raise ValueError("This class cannot estimate relative entropy (prior != None).")
        super().__init__(prior=prior)
        self.k = k
        self.pad = pad

    def forward(self, x: torch.Tensor, log_prob: torch.Tensor = None) -> torch.Tensor:
        red = self.reducer
        if red is not None and getattr(red, "world_size", 1) > 1:
            if not hasattr(red, "all_gather"):
                raise NotImplementedError("KNNEntropyEstimator needs a reducer with all_gather for sharded particles: "
                                          "the nearest neighbours within one rank's shard are not those within the "
                                          "whole batch")
            logsum, n, d = self._sharded_logsum(x)
        else:
            _, _, logsum = ops.knn_kth(x, self.k, self.pad)
            n, d = x.shape
        return (-(knn_entropy_constant(n, d, self.k) + (d / n) * logsum)).to(torch.float32)

    def _sharded_logsum(self, x: torch.Tensor):
        red = self.reducer
        if not isinstance(x, torch.Tensor) or x.dim() != 2:
            raise ValueError("KNNEntropyEstimator: x must be a (N, d) tensor")
        n_local, d = x.shape
        k = int(self.k)
        counts = red.shard_counts(n_local, x.device)
        n = sum(counts)
        ops.knn_check(n, d, k)
        ops._check_f32("x", x)
        row0 = sum(counts[:red.rank])
        return _ShardedKNNLogsum.apply(x, k, float(self.pad), red, counts, row0), n, d
