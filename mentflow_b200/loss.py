"""Discrepancies between predicted and measured profiles (mentflow/loss.py:7-17).

These act on (B,) or (Bx, By) tensors -- O(K*B) work per step, after the particle
reduction -- and stay differentiable torch expressions so that any user-supplied
discrepancy function works unchanged.  The sliced Wasserstein distance between two sample
sets (the reference's sample-space accuracy check) runs on the CUDA kernels of ``ops``."""
import torch

from . import ops


def mean_absolute_error(pred: torch.Tensor, targ: torch.Tensor) -> torch.Tensor:
    return torch.mean(torch.abs(pred - targ))


def mean_square_error(pred: torch.Tensor, targ: torch.Tensor) -> torch.Tensor:
    return torch.mean(torch.square(pred - targ))


def kl_divergence(pred: torch.Tensor, targ: torch.Tensor, pad: float = 1.0e-12) -> torch.Tensor:
    """sum targ * (log targ - log(pred + pad)) / pred.shape[0]  with 0 log 0 = 0
    (= F.kl_div(log(pred+pad), targ, 'batchmean'), loss.py:15-17)."""
    return torch.sum(torch.xlogy(targ, targ) - targ * torch.log(pred + pad)) / pred.shape[0]


def kl_divergence_batched(pred: torch.Tensor, targ: torch.Tensor, pad: float = 1.0e-12) -> torch.Tensor:
    """(K,) KL of K stacked profiles in one expression (first axis = profile index)."""
    k = pred.shape[0]
    terms = torch.xlogy(targ, targ) - targ * torch.log(pred + pad)
    return terms.reshape(k, -1).sum(dim=1) / pred.shape[1]


# --------------------------------------------------------------------------------------
# sliced Wasserstein distance between sample sets (mentflow/loss.py:20-42 through POT)
# --------------------------------------------------------------------------------------
def random_projections(d: int, n_projections: int, seed=None) -> torch.Tensor:
    """(d, n_projections) float64 directions: standard normal columns drawn on the host from
    ``torch.Generator().manual_seed(seed)`` (the global CPU generator when ``seed`` is None), each divided by its
    Euclidean norm, as POT's ``get_random_projections`` does.  This is not POT's random stream: the same seed gives
    other directions than POT's numpy generator."""
    if int(n_projections) < 1:
        raise ValueError(f"n_projections = {n_projections} must be >= 1")
    gen = torch.Generator().manual_seed(int(seed)) if seed is not None else None
    proj = torch.randn(int(d), int(n_projections), generator=gen, dtype=torch.float64)
    return proj / torch.linalg.vector_norm(proj, dim=0, keepdim=True)


def _swd_directions(d: int, n_projections: int, projections, seed) -> torch.Tensor:
    """(P, d) float32 directions, one per row, as the kernels take them."""
    if projections is None:
        projections = random_projections(d, n_projections, seed)
    elif not isinstance(projections, torch.Tensor) or projections.dim() != 2 or projections.shape[0] != d \
            or projections.shape[1] < 1:
        raise ValueError(f"projections must be a (d, P) = ({d}, P) tensor with P >= 1")
    if projections.requires_grad:
        raise ValueError("projections require grad, but the sliced Wasserstein distance differentiates only x")
    return projections.detach().t().to(torch.float32).contiguous()


def _swd_from_wpp(wpp: torch.Tensor, p: float) -> torch.Tensor:
    mean = wpp.sum() / wpp.shape[0]
    swd = mean if p == 1.0 else (torch.sqrt(mean) if p == 2.0 else mean ** (1.0 / p))
    return swd.to(torch.float32)


def _swd_reference(y: torch.Tensor, d: int) -> None:
    ops.check_swd_points("y", y, d)
    if y.requires_grad:
        raise ValueError("the reference samples require grad, but the sliced Wasserstein distance differentiates "
                         "only x: detach them")


def sliced_wasserstein_distance(x: torch.Tensor, y: torch.Tensor, *, n_projections: int = 50, p: float = 2,
                                projections: torch.Tensor = None, seed=None) -> torch.Tensor:
    """Sliced p-Wasserstein distance between the uniformly weighted samples x (N, d) and y (M, d), as POT's
    ``ot.sliced_wasserstein_distance`` defines it: ((1/P) sum_k W_p^p(x theta_k, y theta_k))^(1/p), W_p^p the 1-D
    p-Wasserstein distance to the p-th power.  ``projections`` ((d, P)) is used as given (in float32); otherwise P =
    ``n_projections`` directions come from ``random_projections(d, n_projections, seed)``, which is not POT's random
    stream.  Returns a float32 0-dim tensor, differentiable w.r.t. x (ranks held fixed, as autograd through a sort).
    The projections are sorted by a CUDA radix sort and the quantile integral runs in the same kernel; there is no
    CPU fallback, and sample weights (POT's ``a``, ``b``) are not accepted."""
    ops.check_swd_points("x", x)
    d = x.shape[1]
    _swd_reference(y, d)
    p = ops.check_swd_p(p)
    theta = _swd_directions(d, n_projections, projections, seed).to(x.device)
    y_sorted, _ = ops.swd_sort(y, theta)
    return _swd_from_wpp(ops.swd_wpp(x, theta, y_sorted, p), p)


class SlicedWassersteinDistance:
    """Sliced p-Wasserstein distance to fixed ground-truth samples ``x_true`` (M, d).  The directions are fixed at
    construction (``projections`` (d, P) as given, else ``random_projections(d, n_projections, seed)``) and the
    projections of ``x_true`` are sorted once; ``self(x)`` then returns ``sliced_wasserstein_distance(x, x_true)``
    under those directions as a float32 0-dim tensor, differentiable w.r.t. x."""

    def __init__(self, x_true: torch.Tensor, n_projections: int = 50, p: float = 2, seed=None,
                 projections: torch.Tensor = None) -> None:
        ops.check_swd_points("x_true", x_true)
        d = x_true.shape[1]
        _swd_reference(x_true, d)
        self.p = ops.check_swd_p(p)
        self.theta = _swd_directions(d, n_projections, projections, seed).to(x_true.device)
        self.projections = self.theta.t()
        self.y_sorted, _ = ops.swd_sort(x_true, self.theta)

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        ops.check_swd_points("x", x, self.theta.shape[1])
        return _swd_from_wpp(ops.swd_wpp(x, self.theta, self.y_sorted, self.p), self.p)


# The survey of the reference records this attribute as ``SlicedWassersteindDistance``; the reference tree is not
# part of this repository, so the spelling cannot be checked and both names are exported.
SlicedWassersteindDistance = SlicedWassersteinDistance
