"""Grid sampling of a density (mentflow/sample.py): evaluate the density on the cell centres of
a regular grid, draw cells from the resulting pmf, jitter uniformly inside each cell.

The reference materialises the res^D x D grid points, calls ``prob_func`` on them and uses
``torch.multinomial`` (limited to 2^24 categories).  Here the density of a ``MENT`` model is
evaluated straight from the grid index, the pmf is turned into a float64 CDF by a scan kernel
and particles are drawn by inverse-CDF search with an in-kernel Philox stream -- no category
limit.  The random stream necessarily differs from torch's CPU generator; parity is statistical.

``MetropolisHastingsSampler`` draws without a grid: random-walk Metropolis chains, one per GPU thread, whose cost
does not grow with the dimension's grid resolution.
"""
import math
from typing import Callable, List, Optional, Sequence, Tuple

import torch

from . import ops
from .utils import coords_from_edges, get_grid_points


def _draw_seed() -> int:
    """A fresh 63-bit seed from torch's global generator, so torch.manual_seed reproduces runs."""
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def sample_hist(hist: torch.Tensor, edges: Sequence[torch.Tensor], size: int, noise: float = 0.0,
                device=None, seed: Optional[int] = None) -> torch.Tensor:
    """Particles from a histogram (sample.py:34-57).  ``edges`` must be equally spaced."""
    if hist.ndim == 1 and isinstance(edges, torch.Tensor):
        edges = [edges]
    shape = list(hist.shape)
    first = [float(e[0]) for e in edges]
    cell = [float((e[-1].double() - e[0].double()) / (len(e) - 1)) for e in edges]
    x = ops.cdf_sample(hist, shape, first, cell, int(size), _draw_seed() if seed is None else seed,
                       jitter=bool(noise))
    return torch.squeeze(x)


class GridSampler:
    def __init__(self, limits: List[Tuple[float]], shape: Tuple[int], noise: float = 0.0, device=None,
                 store: bool = True) -> None:
        self.device = device
        self.shape = tuple(int(s) for s in shape)
        self.limits = limits
        self.ndim = len(limits)
        self.noise = noise
        self.store = store
        self.edges = [torch.linspace(limits[a][0], limits[a][1], self.shape[a] + 1) for a in range(self.ndim)]
        self.coords = [coords_from_edges(e) for e in self.edges]
        self.points = None
        self.calls = 0

    def send(self, x: torch.Tensor) -> torch.Tensor:
        return x.type(torch.float32).to(self.device)

    # geometry handed to the kernels (python floats, float64 arithmetic)
    def cell_sizes(self):
        return [(float(self.limits[a][1]) - float(self.limits[a][0])) / self.shape[a] for a in range(self.ndim)]

    def first_centres(self):
        return [float(self.limits[a][0]) + 0.5 * c for a, c in enumerate(self.cell_sizes())]

    def get_grid_points(self) -> torch.Tensor:
        if self.points is not None:
            return self.points
        points = self.send(get_grid_points(*self.coords))
        if self.store:
            self.points = points
        return points

    supports_offset = True    # __call__ takes the index of the first particle to draw (sharded MENT)

    def __call__(self, prob_func: Callable, size: int, seed: Optional[int] = None, offset: int = 0) -> torch.Tensor:
        """``size`` particles; particle s of the call uses Philox counter ``offset + s``, so ranks that pass the
        same seed (torch.manual_seed on every rank) and disjoint offsets draw disjoint slices of one stream."""
        owner = getattr(prob_func, "__self__", None)
        if owner is not None and hasattr(owner, "prob_on_grid") and getattr(prob_func, "__name__", "") == "prob":
            prob = owner.prob_on_grid(self)           # density from the grid index, nothing materialised
        else:
            prob = prob_func(self.get_grid_points())
        self.calls += 1
        first = [float(self.limits[a][0]) for a in range(self.ndim)]
        x = ops.cdf_sample(prob, list(self.shape), first, self.cell_sizes(), int(size),
                           _draw_seed() if seed is None else seed, offset=int(offset), jitter=bool(self.noise))
        return x

    def to(self, device):
        self.device = device
        self.edges = [self.send(e) for e in self.edges]
        self.coords = [self.send(c) for c in self.coords]
        self.points = None
        return self


class MetropolisHastingsSampler:
    """Random-walk Metropolis chains over a density, one chain per GPU thread, with no sampling grid.

    Every call runs ``ceil(size / steps)`` chains (more when ``offset`` splits one) and returns, row by row, the states
    ``x_{burnin + r thin}``, r = 0 .. steps - 1, of chain 0, then chain 1, ...; row s of a call with ``offset = o`` is
    row o + s of that layout.  A chain starts at ``start`` or at ``start_scale * N(0, I)`` and proposes
    ``x + L xi``, L the Cholesky factor of ``proposal_cov`` (default (2.38^2 / D) I); it moves iff the proposal's
    density is finite and at least ``u`` times the current one, u ~ U(0, 1].  A chain is a pure function of the seed,
    its global index, the start and the density (Philox layout: ``mfb_ment_mh`` in the C header), so the draws do not
    depend on the launch shape or on how the rows are split between ranks.

    Called with a ``MENT`` model's bound ``prob``, the whole run is one fused kernel (``MENT.mh_chains``); with any
    other callable, a propose kernel and an accept kernel run the same chains step by step around ``prob_func``, which
    takes (n, D) float32 points and returns (n,) densities on the same CUDA device.  After a call,
    ``acceptance_rate`` is the fraction of proposals taken, as a device tensor (reading it synchronises)."""

    supports_offset = True    # __call__ takes the index of the first row to draw (sharded MENT)

    def __init__(self, ndim: int, burnin: int, steps: int = 1, thin: int = 1, proposal_cov=None, start=None,
                 start_scale: float = 1.0, device=None) -> None:
        ndim, burnin, steps, thin = int(ndim), int(burnin), int(steps), int(thin)
        if not 1 <= ndim <= 8:
            raise ValueError(f"MetropolisHastingsSampler: ndim must be in 1 .. 8, got {ndim}")
        if burnin < 0 or steps < 1 or thin < 1:
            raise ValueError(f"MetropolisHastingsSampler: burnin >= 0, steps >= 1 and thin >= 1 needed, got "
                             f"burnin={burnin}, steps={steps}, thin={thin}")
        if burnin + (steps - 1) * thin >= 2 ** 32:
            raise ValueError("MetropolisHastingsSampler: a chain runs fewer than 2^32 steps (burnin + (steps-1) thin)")
        if proposal_cov is None:
            cov = torch.eye(ndim, dtype=torch.float64) * (2.38 ** 2 / ndim)
        else:
            cov = torch.as_tensor(proposal_cov).detach().to("cpu", torch.float64)
        if tuple(cov.shape) != (ndim, ndim):
            raise ValueError(f"proposal_cov must have shape ({ndim}, {ndim}), got {tuple(cov.shape)}")
        chol, info = torch.linalg.cholesky_ex(cov)
        if not bool(torch.isfinite(cov).all()) or not torch.allclose(cov, cov.T, rtol=1e-12, atol=0.0) or int(info):
            raise ValueError("proposal_cov must be symmetric positive definite")
        if start is not None:
            start = torch.as_tensor(start).detach().to("cpu", torch.float32).contiguous()
            if tuple(start.shape) != (ndim,):
                raise ValueError(f"start must have shape ({ndim},), got {tuple(start.shape)}")
        if not math.isfinite(float(start_scale)):
            raise ValueError("start_scale must be finite")
        self.ndim, self.burnin, self.steps, self.thin = ndim, burnin, steps, thin
        self.chol = chol.to(torch.float32)
        self.start = start
        self.start_scale = float(start_scale)
        self.device = device
        self.acceptance_rate = None

    def proposals(self) -> int:
        """proposals per chain and call"""
        return self.burnin + (self.steps - 1) * self.thin

    def chain_args(self, device):
        """(chol, start) on ``device``, float32"""
        start = None if self.start is None else self.start.to(device)
        return self.chol.to(device), start

    def _device(self):
        return torch.device(self.device if self.device is not None else "cuda")

    def __call__(self, prob_func: Callable, size: int, seed: Optional[int] = None, offset: int = 0) -> torch.Tensor:
        """Rows ``offset .. offset + size - 1`` of the chains' recorded states; ranks that pass the same seed
        (torch.manual_seed on every rank) and disjoint offsets return disjoint slices of one draw."""
        size, offset = int(size), int(offset)
        seed = _draw_seed() if seed is None else int(seed)   # drawn even for size 0: every rank's generator moves alike
        if size < 0 or offset < 0:
            raise ValueError("size and offset must be non-negative")
        if size == 0:
            return torch.empty((0, self.ndim), dtype=torch.float32, device=self._device())
        c0 = offset // self.steps
        nc = (offset + size - 1) // self.steps - c0 + 1
        owner = getattr(prob_func, "__self__", None)
        if owner is not None and hasattr(owner, "mh_chains") and getattr(prob_func, "__name__", "") == "prob":
            rows, accepted = owner.mh_chains(self, c0, nc, seed)
        else:
            rows, accepted = self._step_chains(prob_func, c0, nc, seed)
        self.acceptance_rate = accepted.double() / max(1, nc * self.proposals())
        lo = offset - c0 * self.steps
        return rows[lo:lo + size]

    def _step_chains(self, prob_func: Callable, c0: int, nc: int, seed: int):
        """The fused kernel's chains, one propose / prob_func / accept round per step."""
        device = ops._cuda_device(self._device(), "MetropolisHastingsSampler")
        chol, start = self.chain_args(device)
        d = self.ndim
        rows = torch.empty((nc, self.steps, d), dtype=torch.float32, device=device)
        accepted = torch.zeros(1, dtype=torch.int64, device=device)
        x = ops.mh_propose(None, nc, d, c0, None, 0, seed, device, start=start, start_scale=self.start_scale)
        rho = self._density(prob_func, x, nc)
        for t in range(self.proposals() + 1):
            if t > 0:
                xp = ops.mh_propose(x, nc, d, c0, chol, t, seed, device)
                ops.mh_accept(x, rho, xp, self._density(prob_func, xp, nc), c0, t, seed, accepted)
            if t >= self.burnin and (t - self.burnin) % self.thin == 0:
                rows[:, (t - self.burnin) // self.thin] = x
        return rows.view(nc * self.steps, d), accepted

    @staticmethod
    def _density(prob_func: Callable, x: torch.Tensor, n: int) -> torch.Tensor:
        rho = prob_func(x)
        if not isinstance(rho, torch.Tensor) or rho.numel() != n:
            raise ValueError(f"prob_func must return {n} densities for {n} points")
        return ops._check_f32("prob_func(x)", rho.reshape(-1)).clone()

    def to(self, device):
        self.device = device
        return self
