"""Classical MENT (mentflow/ment.py): rho(x) = prior(x) * prod_k h_k(M_k x) with one Lagrange
table per measured profile, updated by Gauss-Seidel sweeps.

Interface of the reference's ``MENT`` / ``LagrangeFunction``; the arithmetic runs in the CUDA
library: ``prob`` is one fused kernel over all measurements (the reference does a device->numpy
->scipy->device round trip per measurement), sampling is a scan + inverse-CDF kernel, the
predicted profile of the sampled particles is the fused projection+KDE kernel, and the table
update is one elementwise kernel.  One- and two-dimensional screens (Histogram1D / Histogram2D:
experiments/config/rec_nd_1d_ment.yaml, rec_nd_2d_ment.yaml) of any size may be mixed, as in the reference: a
family whose screens all have the same bins is passed as stacked tables, one whose sizes differ as concatenated
tables with offsets (``ops.RaggedTables1D`` / ``ops.RaggedTables2D``), which the same kernels read in their ragged
layout.

Transfer maps are linear (``LinearTransform``, or a ``CompositeTransform`` of them) or a chain
linear* -> MultipoleTransform (order 3, 4 or 5, normal or skew) -> linear* (experiments/rec_2d/nonlinear), in
any mix.  Behind a kick the projection of a screen is ``w . x + a Re(z^m) + b Im(z^m)``
(``simulate.multipole_terms``), evaluated inside the density kernels; integrate mode maps the screen back
with the chain's folded inverse (``simulate.multipole_inverse_terms``), and sample mode predicts profiles
through ``simulate.forward`` (1-D screens behind a kick fused, 2-D ones object by object).  Other maps
raise ``NotImplementedError``.

Sharded over GPUs (``mentflow_b200.distributed.shard_model``; BASELINE config 5): every rank evaluates
the same density, draws ITS slice of the ``n_samples`` particles from the same Philox stream (particle s
always uses counter s, whichever rank draws it), and the unnormalised profile sums are all-reduced before
the normalisation -- so every rank applies the identical table update and the union of the particles is
the set one GPU would have drawn.
"""
import math
from typing import Any, Callable, List, Optional, Tuple

import torch

from . import ops
from .diagnostics import Histogram1D, Histogram2D
from .loss import kl_divergence
from .prior import Gaussian, Uniform
from .simulate import forward as simulate_forward
from .simulate.simulate import _linear_matrix, _multipole_chain, multipole_inverse_terms, multipole_terms
from .simulate.transform import LinearTransform
from .utils import coords_from_edges, get_grid_points, unravel


class LagrangeFunction:
    """One h_k: values on the bin centres (1-D) or on the grid of bin centres (2-D), multilinear
    interpolation in between, zero outside (ment.py:20-52; scipy RegularGridInterpolator(method="linear",
    bounds_error=False, fill_value=0), evaluated in double)."""

    def __init__(self, coords, values: torch.Tensor, **interpolation_kws) -> None:
        method = interpolation_kws.get("method", "linear")
        if method != "linear":
            raise NotImplementedError("only linear interpolation of the Lagrange functions is implemented")
        self.coords = coords
        self.values = values

    def set_values(self, values: torch.Tensor) -> None:
        self.values = values

    def __call__(self, u: torch.Tensor) -> torch.Tensor:
        if self.values.ndim == 1:
            u = u.reshape(-1, 1).to(torch.float32)
            one = torch.ones((1, 1), dtype=torch.float32, device=u.device)
            coords, values = (t.reshape(1, -1).to(u.device) for t in (self.coords, self.values))
            return ops.ment_prob(u, (one, coords, values), None, 0.0, 0.0)
        u = u.reshape(-1, 2).to(torch.float32)
        eye = torch.eye(2, dtype=torch.float32, device=u.device).reshape(1, 2, 2)
        cx, cy = (c.reshape(1, -1).to(u.device) for c in self.coords)
        return ops.ment_prob(u, None, (eye, cx, cy, self.values.to(u.device)[None]), 0.0, 0.0)


class MENT:
    def __init__(self, ndim: int, transforms: List[Callable], diagnostics: List[List[Callable]],
                 measurements: List[List[torch.Tensor]], discrepancy_function: Callable = kl_divergence,
                 prior: Any = None, interpolation: str = "linear", mode: str = "integrate",
                 integration_limits=None, integration_shape=None, sampler: Optional[Callable] = None,
                 n_samples: int = 1000000, device=None, verbose: bool = False) -> None:
        self.device = device
        self.verbose = verbose
        self.mode = mode
        self.ndim = ndim
        self.epoch = 0
        self.transforms = transforms
        self.diagnostics = [[]] if diagnostics is None else diagnostics
        self.measurements = [[]] if measurements is None else measurements
        self.discrepancy_function = discrepancy_function
        # the reference's default refers to an undefined `UniformPrior` (ment.py:143)
        self.prior = prior if prior is not None else Uniform(ndim=ndim, scale=100.0)
        self.integration_limits = integration_limits
        self.integration_shape = integration_shape
        self.sampler = sampler
        self.n_samples = int(n_samples)
        self.interpolation = interpolation
        self.reducer = None
        self._packed = None
        self.shard = None     # (rank, world_size) when the particles are sharded over GPUs
        for row in self.diagnostics:
            for d in row:
                if not isinstance(d, (Histogram1D, Histogram2D)):
                    raise NotImplementedError("MENT on the CUDA path supports Histogram1D / Histogram2D screens")
        self.lagrange_functions = self.initialize_lagrange_functions()

    # ------------------------------------------------------------------ bookkeeping
    def send(self, x: torch.Tensor) -> torch.Tensor:
        return x.type(torch.float32).to(self.device)

    def set_diagnostics(self, diagnostics):
        self.diagnostics = [[]] if diagnostics is None else diagnostics
        self._packed = None
        return self.diagnostics

    def set_measurements(self, measurements):
        self.measurements = [[]] if measurements is None else measurements
        return self.measurements

    def initialize_lagrange_functions(self):
        """h_k = 1 where the measurement is positive, else 0 (ment.py:169-182)."""
        self.lagrange_functions = []
        for index in range(len(self.measurements)):
            row = []
            for measurement, diagnostic in zip(self.measurements[index], self.diagnostics[index]):
                if measurement.ndim == 1:
                    coords = coords_from_edges(diagnostic.edges)
                else:
                    coords = [coords_from_edges(e) for e in diagnostic.edges]
                values = (measurement > 0.0).float()
                row.append(LagrangeFunction(coords, values, method=self.interpolation))
            self.lagrange_functions.append(row)
        self._packed = None
        return self.lagrange_functions

    def _slots(self):
        return [(i, j) for i in range(len(self.diagnostics)) for j in range(len(self.diagnostics[i]))]

    def _transfer(self, index: int):
        """(matrix, chain) of transform ``index``: the matrix of a linear map (None for the identity) and no chain, or
        no matrix and the (pre, kick, post) of a linear* -> MultipoleTransform -> linear* chain."""
        transform = self.transforms[index]
        matrix = _linear_matrix(transform)
        if matrix is not NotImplemented:
            return matrix, None
        chain = _multipole_chain(transform)
        if chain is None or self.ndim == 3:
            raise NotImplementedError(
                "MENT on the CUDA path supports linear transfer maps (LinearTransform or a CompositeTransform of them) "
                "and chains linear* -> MultipoleTransform(order 3, 4 or 5) -> linear* in D = 2 or D >= 4; "
                f"transform {index} is {type(transform).__name__}")
        return None, chain

    def _pack(self, device):
        """Static part of the kernel arguments: projection rows and bin centres of every table, the 1-D and
        the 2-D screens as two families; with a multipole kick anywhere in the model, the multipole rows of every
        screen as well (order 0 behind linear maps).  A family of equal sizes stacks its centres; one whose sizes
        differ concatenates them and keeps the offsets of the ragged layout ("offsets", "offsets2")."""
        if self._packed is not None and self._packed["device"] == device:
            return self._packed
        slots1, proj1, coords1, mp1 = [], [], [], []
        slots2, proj2, cx2, cy2, mp2 = [], [], [], [], []
        nd = self.ndim
        for i, j in self._slots():
            d = self.diagnostics[i][j]
            matrix, chain = self._transfer(i)
            if chain is not None:
                # measured rows of the linear part after the kick, folded through the kick and the part before it
                pre, kick, post = chain
                post32 = post.to(torch.float32) if post is not None else None
                rows = (d.projection_vectors(post32, nd, "cpu") if isinstance(d, Histogram2D)
                        else d.projection_vector(post32, nd, "cpu")[None])
                terms = [multipole_terms(r, pre, kick, nd) for r in rows]
                vec = torch.stack([w for w, _ in terms]).to(device)
                mp = torch.stack([m for _, m in terms]).to(device)
            if isinstance(d, Histogram2D):
                slots2.append((i, j))
                proj2.append(d.projection_vectors(matrix, nd, device) if chain is None else vec)
                mp2.append(mp if chain is not None else None)
                cx2.append(coords_from_edges(d.edges_x.to(torch.float32)).to(device))
                cy2.append(coords_from_edges(d.edges_y.to(torch.float32)).to(device))
            else:
                slots1.append((i, j))
                proj1.append(d.projection_vector(matrix, nd, device) if chain is None else vec[0])
                mp1.append(mp[0] if chain is not None else None)
                coords1.append(coords_from_edges(d.edges.to(torch.float32)).to(device))
        kicked = any(m is not None for m in mp1 + mp2)

        def starts(sizes):
            out = [0]
            for n in sizes:
                out.append(out[-1] + n)
            return out

        bins1 = [int(c.shape[0]) for c in coords1]
        bins2 = [(int(x.shape[0]), int(y.shape[0])) for x, y in zip(cx2, cy2)]
        offsets = starts(bins1) if len(set(bins1)) > 1 else None
        offsets2 = ([starts(bx for bx, _ in bins2), starts(by for _, by in bins2), starts(bx * by for bx, by in bins2)]
                    if len(set(bins2)) > 1 else None)

        def stack_mp(rows, shape):
            if not kicked or not rows:
                return None
            return torch.stack([m if m is not None else torch.zeros(shape, dtype=torch.float32, device=device)
                                for m in rows]).contiguous()

        def pack(family, ragged):
            if not family:
                return None
            return (torch.cat(family) if ragged else torch.stack(family)).contiguous()

        self._packed = {"device": device, "slots1": slots1, "slots2": slots2,
                        "proj": torch.stack(proj1).contiguous() if proj1 else None,
                        "coords": pack(coords1, offsets is not None), "offsets": offsets,
                        "proj2": torch.stack(proj2).contiguous() if proj2 else None,
                        "cx2": pack(cx2, offsets2 is not None), "cy2": pack(cy2, offsets2 is not None),
                        "offsets2": offsets2,
                        "mp": stack_mp(mp1, (2 * nd + 4,)), "mp2": stack_mp(mp2, (2, 2 * nd + 4)),
                        "kicked": kicked, "inverse": {}}
        return self._packed

    def _groups(self, device):
        """(g1, g2) for ``ops.ment_prob``: the current tables of the two screen families, followed by their
        multipole rows when the model has a kick; a family whose sizes differ as ``ops.RaggedTables1D`` /
        ``ops.RaggedTables2D`` of the concatenated tables."""
        pk = self._pack(device)

        def tables(slots, ragged):
            values = [self.lagrange_functions[i][j].values.to(device=device, dtype=torch.float32) for i, j in slots]
            return (torch.cat([v.reshape(-1) for v in values]) if ragged else torch.stack(values)).contiguous()

        g1 = g2 = None
        if pk["slots1"]:
            h = tables(pk["slots1"], pk["offsets"] is not None)
            if pk["offsets"] is not None:
                g1 = ops.RaggedTables1D(pk["proj"], pk["coords"], h, pk["offsets"], pk["mp"])
            else:
                g1 = (pk["proj"], pk["coords"], h) + ((pk["mp"],) if pk["kicked"] else ())
        if pk["slots2"]:
            h = tables(pk["slots2"], pk["offsets2"] is not None)
            if pk["offsets2"] is not None:
                g2 = ops.RaggedTables2D(pk["proj2"], pk["cx2"], pk["cy2"], h, pk["offsets2"], pk["mp2"])
            else:
                g2 = (pk["proj2"], pk["cx2"], pk["cy2"], h) + ((pk["mp2"],) if pk["kicked"] else ())
        return g1, g2

    def _inverse(self, index: int, device):
        """(minv, inv_mp) mapping screen coordinates of transform ``index`` back to x: the inverse matrix of a linear
        map (``matrix_inv`` of a LinearTransform, the inverse of the product of a linear CompositeTransform) and no
        kick, or L and the kick terms of a multipole chain (``multipole_inverse_terms``, kept with the packed rows)."""
        matrix, chain = self._transfer(index)
        if chain is None:
            transform = self.transforms[index]
            if isinstance(transform, LinearTransform):
                minv = transform.matrix_inv
            elif matrix is None:
                minv = torch.eye(self.ndim)
            else:
                minv = torch.linalg.inv(matrix)
            return minv.to(device=device, dtype=torch.float32).contiguous(), None
        cache = self._pack(device)["inverse"]
        if index not in cache:
            lin, imp = multipole_inverse_terms(*chain, self.ndim)
            cache[index] = (lin.to(device).contiguous(), imp.to(device).contiguous())
        return cache[index]

    def _prior_args(self) -> Tuple[float, float]:
        if isinstance(self.prior, Gaussian):
            return -0.5 / self.prior.scale ** 2, self.prior.log_norm
        if isinstance(self.prior, Uniform):
            return 0.0, -math.log(self.prior.volume)
        raise NotImplementedError("MENT on the CUDA path supports the Gaussian and Uniform priors")

    # ------------------------------------------------------------------ density
    def prob(self, x: torch.Tensor) -> torch.Tensor:
        """rho(x) (ment.py:239-249)."""
        g1, g2 = self._groups(x.device)
        a, b = self._prior_args()
        return ops.ment_prob(x, g1, g2, a, b)

    def prob_on_grid(self, sampler) -> torch.Tensor:
        """rho on the cell centres of a GridSampler grid, straight from the grid index."""
        device = torch.device(self.device if self.device is not None else "cuda")
        g1, g2 = self._groups(device)
        a, b = self._prior_args()
        return ops.ment_prob_grid(list(sampler.shape), sampler.first_centres(), sampler.cell_sizes(), g1, g2, a, b,
                                  device)

    def mh_chains(self, sampler, chain0: int, nchains: int, seed: int):
        """Metropolis-Hastings chains chain0 .. chain0 + nchains - 1 of a MetropolisHastingsSampler over rho, in one
        fused kernel: (recorded states (nchains * steps, D), proposals taken (1,) int64)."""
        device = torch.device(self.device if self.device is not None else "cuda")
        g1, g2 = self._groups(device)
        a, b = self._prior_args()
        chol, start = sampler.chain_args(device)
        return ops.ment_mh(g1, g2, a, b, self.ndim, chain0, nchains, chol, sampler.burnin, sampler.steps, sampler.thin,
                           seed, start=start, start_scale=sampler.start_scale)

    def log_prob(self, x: torch.Tensor, pad: float = 1.0e-12) -> torch.Tensor:
        return torch.log(self.prob(x) + pad)

    def evaluate_lagrange_function(self, u: torch.Tensor, index: int, diag_index: int) -> torch.Tensor:
        diagnostic = self.diagnostics[index][diag_index]
        return self.lagrange_functions[index][diag_index](diagnostic.project(u))

    def sample(self, size: int) -> torch.Tensor:
        """``size`` particles from rho.  Sharded (``self.shard``): this rank's slice of them -- the sampler draws
        particle s with Philox counter s, so the slices of all ranks together are the particles of one draw."""
        size = int(size)
        if self.shard is not None and self.shard[1] > 1 and getattr(self.sampler, "supports_offset", False):
            from .distributed import shard_slice
            sl = shard_slice(size, self.shard[0], self.shard[1])
            return self.send(self.sampler(self.prob, sl.stop - sl.start, offset=sl.start))
        return self.send(self.sampler(self.prob, size))

    def sample_and_log_prob(self, size: int):
        x = self.sample(size)
        return x, self.log_prob(x)

    def discrepancy_vector(self, predictions) -> List[torch.Tensor]:
        return [self.discrepancy_function(pred, meas)
                for pred, meas in zip(unravel(predictions), unravel(self.measurements))]

    # ------------------------------------------------------------------ simulation of one profile
    def normalize_projection(self, projection: torch.Tensor, index: int, diag_index: int) -> torch.Tensor:
        diagnostic = self.diagnostics[index][diag_index]
        if isinstance(diagnostic, Histogram2D):
            bin_volume = math.prod(float(e[1] - e[0]) for e in diagnostic.edges)
        else:
            bin_volume = diagnostic.edges[1] - diagnostic.edges[0]
        return projection / projection.sum() / bin_volume

    def get_meas_points(self, index: int, diag_index: int) -> torch.Tensor:
        diagnostic = self.diagnostics[index][diag_index]
        if isinstance(diagnostic, Histogram2D):
            return get_grid_points(*[coords_from_edges(e) for e in diagnostic.edges])
        return coords_from_edges(diagnostic.edges)

    def get_integration_points(self, index: int, diag_index: int) -> torch.Tensor:
        limits = self.integration_limits[index][diag_index]
        shape = self.integration_shape[index][diag_index]
        coords = [self.send(torch.linspace(limits[k][0], limits[k][1], shape[k])) for k in range(len(shape))]
        return coords[0] if len(coords) == 1 else self.send(get_grid_points(*coords))

    def _simulate_integrate(self, index: int, diag_index: int) -> torch.Tensor:
        """pred[b] = sum over the integration grid of rho(T^-1 [pixel; grid]) (ment.py:267-317)."""
        limits = self.integration_limits[index][diag_index]
        shape = [int(s) for s in self.integration_shape[index][diag_index]]
        diagnostic = self.diagnostics[index][diag_index]
        device = torch.device(self.device if self.device is not None else "cuda")
        g1, g2 = self._groups(device)
        a, b = self._prior_args()
        first = [float(limits[k][0]) for k in range(len(shape))]
        step = [(float(limits[k][1]) - float(limits[k][0])) / max(shape[k] - 1, 1) for k in range(len(shape))]
        minv, inv_mp = self._inverse(index, device)
        if isinstance(diagnostic, Histogram2D):
            cx = coords_from_edges(diagnostic.edges_x.to(torch.float32)).to(device)
            cy = coords_from_edges(diagnostic.edges_y.to(torch.float32)).to(device)
            ax, ay = diagnostic.axis
            pred = ops.ment_integrate(self.ndim, cx, ax, cy, ay, shape, first, step, minv, g1, g2, a, b,
                                      inv_mp=inv_mp)
        else:
            meas_coords = coords_from_edges(diagnostic.edges.to(torch.float32)).to(device)
            pred = ops.ment_integrate(self.ndim, meas_coords, diagnostic.axis, None, -1, shape, first, step, minv,
                                      g1, g2, a, b, inv_mp=inv_mp)
        return self.normalize_projection(pred, index, diag_index)

    def _simulate_sample(self, index: int, diag_index: int) -> torch.Tensor:
        """sample -> transform -> KDE profile -> normalise (ment.py:319-326)."""
        x = self.sample(int(self.n_samples))
        pred = simulate_forward(x, [self.transforms[index]], [[self.diagnostics[index][diag_index]]],
                                reducer=self.reducer)[0][0]
        return self.normalize_projection(pred, index, diag_index)

    def simulate(self, index: int, diag_index: int, **kws) -> torch.Tensor:
        if self.mode == "integrate":
            return self._simulate_integrate(index, diag_index, **kws)
        if self.mode == "sample":
            return self._simulate_sample(index, diag_index, **kws)
        raise ValueError(f"Invalid mode {self.mode}")

    def simulate_all(self, **kws):
        if self.mode == "integrate":
            return [[self._simulate_integrate(i, j, **kws) for j in range(len(self.diagnostics[i]))]
                    for i in range(len(self.diagnostics))]
        x = self.sample(self.n_samples)
        return simulate_forward(x, self.transforms, self.diagnostics, reducer=self.reducer)

    # ------------------------------------------------------------------ Gauss-Seidel relaxation
    def gauss_seidel_update(self, lr: float = 1.0, thresh: float = 1.0e-10, **kws) -> None:
        """h <- h * (1 + lr * (g / g* - 1)) where g != 0 and g* >= thresh, one measurement after the
        other, each update feeding the next simulation (ment.py:336-371)."""
        for index in range(len(self.transforms)):
            if self.verbose:
                print(f"index={index}")
            for diag_index in range(len(self.diagnostics[index])):
                lf = self.lagrange_functions[index][diag_index]
                measurement = self.measurements[index][diag_index]
                prediction = self.simulate(index, diag_index, **kws)
                values = lf.values.to(device=prediction.device, dtype=torch.float32).contiguous().clone()
                ops.gs_update(values.view(-1), measurement.to(prediction.device).reshape(-1), prediction.reshape(-1),
                              lr, thresh)
                lf.set_values(values)
        self.epoch += 1

    gauss_seidel_step = gauss_seidel_update   # name used by BASELINE.json's north_star

    # ------------------------------------------------------------------ persistence
    def save(self, path: str) -> None:
        state = {"lagrange_functions": self.lagrange_functions, "epoch": self.epoch, "transforms": self.transforms,
                 "diagnostics": self.diagnostics, "measurements": self.measurements, "prior": self.prior,
                 "ndim": self.ndim, "sampler": self.sampler}
        torch.save(state, path)

    def load(self, path: str, device=None) -> None:
        state = torch.load(path, map_location=device, weights_only=False)
        for key in ("lagrange_functions", "epoch", "transforms", "diagnostics", "measurements", "prior", "ndim",
                    "sampler"):
            setattr(self, key, state[key])
        self._packed = None
        self.to(device)

    def to(self, device):
        self.device = device
        self._packed = None
        if self.transforms is not None:
            self.transforms = [t.to(device) for t in self.transforms]
        if self.diagnostics is not None:
            self.diagnostics = [[d.to(device) for d in row] for row in self.diagnostics]
        if self.measurements is not None:
            self.measurements = [[m.to(device) for m in row] for row in self.measurements]
        if self.sampler is not None:
            self.sampler = self.sampler.to(device)
        if self.prior is not None:
            self.prior = self.prior.to(device)
        for row in self.lagrange_functions:
            for lf in row:
                lf.values = self.send(lf.values)
                # a 2-D screen's centres are one tensor per axis
                lf.coords = ([self.send(c) for c in lf.coords] if isinstance(lf.coords, (list, tuple))
                             else self.send(lf.coords))
        return self
