"""Forward simulation: particles -> predicted profiles on every screen.

``forward(x, transforms, diagnostics)`` has the signature and return structure of
``mentflow/simulate/simulate.py:8-33`` (``predictions[i][j]`` = diagnostic j after transform i).
Where the reference loops in Python (K clones, K full D x D matmuls, K dense (N, B) kernel
matrices), this builds a *plan* -- one projection row per linear (transform, screen) pair --
and launches the fused projection+binning kernel once per group of equally shaped screens.
Pairs that cannot be fused (a non-linear transform, a custom diagnostic) fall back to calling
the objects one by one, exactly like the reference; the screen itself still bins with the
CUDA kernel.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Callable, List, Optional, Sequence

import torch
import torch.nn as nn

from .. import ops
from ..diagnostics.diagnostics import Histogram1D, Histogram2D
from .transform import CompositeTransform, LinearTransform, MultipoleTransform

# set by mentflow_b200.distributed when particles are sharded across ranks: a callable
# reducer(sums_tensor, n_local) -> n_global that all-reduces in place
_default_reducer: Optional[Callable] = None


def set_default_reducer(reducer: Optional[Callable]) -> None:
    global _default_reducer
    _default_reducer = reducer


def _geom_tensor(rows, device):
    return torch.tensor([[c0, spacing, sigma, delta, 0.0, 0.0, 0.0, 0.0] for c0, spacing, sigma, delta in rows],
                        dtype=torch.float32, device=device)


def _density_from_counts(counts: torch.Tensor, widths: torch.Tensor) -> torch.Tensor:
    """torch.histogram(density=True) from integer counts: counts / total / bin widths, all in
    fp32 like the reference's CPU op (SURVEY App. B.3)."""
    c = counts.to(torch.float32)
    total = c.sum(dim=tuple(range(1, c.ndim)), keepdim=True)
    return c / total / widths


def profiles_1d(x: torch.Tensor, proj: torch.Tensor, diags: Sequence[Histogram1D], kde: bool = True,
                reducer: Optional[Callable] = None, cache: Optional[dict] = None,
                kl_targets: Optional[torch.Tensor] = None, mp: Optional[torch.Tensor] = None):
    """(K, B) profiles of K one-dimensional screens sharing the same number of bins.
    proj is (K, D): x_proj_k = x . proj_k.  ``cache`` keeps the device-side geometry between
    calls (filled on first use).  With ``kl_targets`` (K, B) and KDE screens the result is a pair
    (profiles, kl[K]): the KL of loss.py:15-17 comes out of the normalisation kernel.  ``mp`` (K, 2D+4):
    multipole terms of the transfer maps (``multipole_terms``)."""
    reducer = reducer if reducer is not None else _default_reducer
    cache = {} if cache is None else cache
    nb = diags[0].nbins
    if kde:
        if "geom" not in cache:
            rows = [d.geometry() for d in diags]
            cache["geom"] = _geom_tensor(rows, x.device)
            cache["ratio"] = max(s / sp for _, sp, s, _ in rows)
        return ops.project_kde1d(x, proj, cache["geom"], cache["ratio"], nb, reducer, kl_targets, mp)
    if "edges" not in cache:
        cache["edges"] = torch.stack([d.edges.to(x.device) for d in diags]).contiguous()
        cache["widths"] = torch.diff(cache["edges"], dim=1)
    counts = ops.project_hist1d(x.detach(), proj, cache["edges"], mp=mp)
    if reducer is not None:
        reducer(counts, 0.0)
    return _density_from_counts(counts, cache["widths"])


def profiles_2d(x: torch.Tensor, proj: torch.Tensor, diags: Sequence[Histogram2D], kde: bool = True,
                reducer: Optional[Callable] = None, cache: Optional[dict] = None) -> torch.Tensor:
    """(K, Bx, By) profiles of K two-dimensional screens of equal shape; proj is (K, 2, D)."""
    reducer = reducer if reducer is not None else _default_reducer
    cache = {} if cache is None else cache
    bx, by = diags[0].shape
    if kde:
        if "geom" not in cache:
            rows = []
            for d in diags:
                gx, gy = d.geometry()
                rows += [gx, gy]
            cache["geom"] = _geom_tensor(rows, x.device).reshape(len(diags), 2, -1)
            cache["ratio"] = max(s / sp for _, sp, s, _ in rows)
        return ops.project_kde2d(x, proj, cache["geom"], cache["ratio"], bx, by, reducer)
    if "ex" not in cache:
        cache["ex"] = torch.stack([d.edges_x.to(x.device) for d in diags]).contiguous()
        cache["ey"] = torch.stack([d.edges_y.to(x.device) for d in diags]).contiguous()
        cache["area"] = torch.diff(cache["ex"], dim=1)[:, :, None] * torch.diff(cache["ey"], dim=1)[:, None, :]
    counts = ops.project_hist2d(x.detach(), proj, cache["ex"], cache["ey"])
    if reducer is not None:
        reducer(counts, 0.0)
    return _density_from_counts(counts, cache["area"])


# --------------------------------------------------------------------------------------
# plan: which (transform, screen) pairs fuse, grouped by screen shape
# --------------------------------------------------------------------------------------
class _Group:
    __slots__ = ("kind", "kde", "slots", "diags", "proj", "cache", "mp")

    def __init__(self, kind, kde):
        self.kind, self.kde = kind, kde
        self.slots, self.diags, self.proj = [], [], []
        self.cache = {}
        self.mp = None      # list of multipole rows (1-D groups behind a MultipoleTransform), else None


class _Plan:
    def __init__(self):
        self.groups: "OrderedDict[tuple, _Group]" = OrderedDict()
        self.fallback: List[tuple] = []
        self.shape: List[int] = []
        self.refs: list = []     # keeps the objects the cache key identifies alive (see _plan_key)


def _linear_matrix(transform) -> Optional[torch.Tensor]:
    if isinstance(transform, LinearTransform):
        return transform.matrix
    if isinstance(transform, CompositeTransform):
        m = transform.as_matrix()
        return NotImplemented if m is None and len(transform.transforms) > 0 else m
    if transform is None or isinstance(transform, nn.Identity):
        return None
    return NotImplemented


def _multipole_chain(transform):
    """(pre, multipole, post) if ``transform`` is linear* -> MultipoleTransform -> linear* (pre / post are
    product matrices or None for the identity), else None."""
    stages = [transform] if isinstance(transform, MultipoleTransform) else (
        list(transform.transforms) if isinstance(transform, CompositeTransform) else None)
    if stages is None:
        return None
    pre = post = kick = None
    for t in stages:
        if isinstance(t, MultipoleTransform):
            if kick is not None:
                return None
            kick = t
        elif isinstance(t, LinearTransform):
            m = t.matrix.detach().to("cpu", torch.float64)
            if kick is None:
                pre = m if pre is None else m @ pre
            else:
                post = m if post is None else m @ post
        else:
            return None
    if kick is None or kick.order not in (3, 4, 5):
        return None
    return pre, kick, post


def multipole_terms(row: torch.Tensor, pre: Optional[torch.Tensor], kick: MultipoleTransform, ndim: int):
    """(w, mp): the measured coordinate of ``post-row . kick(pre x)`` as
    ``w . x + a Re(z^m) + b Im(z^m)``, z = wa . x + i wb . x, m = order - 1, mp = [wa | wb | a | b | order | 0].

    ``row`` (D,) is the measured row of the linear part after the kick.  Follows
    MultipoleTransform.forward (simulate/transform.py:107-143): normal kick U1 = X1 - k Re, U3 = X1 + k Im
    (the reference reads column 1 there: a linear term, folded into w); skew kick U1 = X1 + k Im,
    U3 = X3 + k Re; columns 2.. exist only for D > 2.  Evaluated in float64 on the host."""
    row = row.detach().to("cpu", torch.float64)
    pre = torch.eye(ndim, dtype=torch.float64) if pre is None else pre
    k = kick.coefficient()
    w = row @ pre
    wa = pre[0].clone()
    wb = pre[2].clone() if ndim > 2 else torch.zeros(ndim, dtype=torch.float64)
    r1 = float(row[1])
    r3 = float(row[3]) if ndim > 2 else 0.0
    if kick.skew:
        a, b = k * r3, k * r1
    else:
        a, b = -k * r1, k * r3
        if ndim > 2:
            w = w + r3 * (pre[1] - pre[3])
    mp = torch.cat([wa, wb, torch.tensor([a, b, float(kick.order), 0.0], dtype=torch.float64)])
    return w.to(torch.float32), mp.to(torch.float32)


def multipole_inverse_terms(pre: Optional[torch.Tensor], kick: MultipoleTransform, post: Optional[torch.Tensor],
                            ndim: int, dtype=torch.float32):
    """(L, imp): the inverse of ``post . kick . pre`` as ``x = L u + p Re(z^m) + q Im(z^m)``, z = r0 . u + i r2 . u,
    m = order - 1, imp = [r0 | r2 | p | q | order | 0] (the integrate mode of classical MENT).

    Follows CompositeTransform.inverse: post^-1, then the kick's inverse (momentum reversal, kick, momentum reversal:
    simulate/transform.py:145-146), then pre^-1.  With A = pre^-1 and B = post^-1, r0 / r2 are rows 0 / 2 of B; the
    normal kick gives p = k A[:, 1], q = -k A[:, 3] and L = A Q B, where Q is the identity except that row 3 is e1 for
    D > 2 (the reference's U[:, 3] = X[:, 1] + ... quirk); the skew kick gives p = -k A[:, 3], q = -k A[:, 1] and L = A B.
    Columns 3.. are absent for D = 2.  Evaluated in float64 on the host, returned as ``dtype``."""
    eye = torch.eye(ndim, dtype=torch.float64)
    a_inv = eye if pre is None else torch.linalg.inv(pre.to(torch.float64))
    b_inv = eye if post is None else torch.linalg.inv(post.to(torch.float64))
    k = kick.coefficient()
    zero = torch.zeros(ndim, dtype=torch.float64)
    r0 = b_inv[0]
    r2 = b_inv[2] if ndim > 2 else zero
    c1 = a_inv[:, 1]
    c3 = a_inv[:, 3] if ndim > 2 else zero
    if kick.skew:
        p, q = -k * c3, -k * c1
        lin = a_inv @ b_inv
    else:
        p, q = k * c1, -k * c3
        quirk = eye.clone()
        if ndim > 2:
            quirk[3] = eye[1]
        lin = a_inv @ quirk @ b_inv
    imp = torch.cat([r0, r2, p, q, torch.tensor([float(kick.order), 0.0], dtype=torch.float64)])
    return lin.to(dtype), imp.to(dtype)


def _tensor_key(t):
    """identity + in-place version of a tensor (None-safe)"""
    return (id(t), getattr(t, "_version", 0)) if t is not None else None


def _plan_key(transforms, diagnostics):
    """(key, refs): the key is built from object identities and tensor version counters; ``refs`` lists
    every object whose id() went into it.  The cached plan keeps ``refs`` alive, so that CPython cannot
    hand a recycled id to a new transform / matrix / screen while the plan that was built for the old one
    is still in the cache (a fresh ``LinearTransform`` per call would otherwise silently reuse stale
    projection rows).  Screen geometry (edges, bandwidth) is part of the key through the buffers' version
    counters, so editing ``diag.bandwidth`` or the edges in place rebuilds the plan."""
    key, refs = [], []
    for t, row in zip(transforms, diagnostics):
        m = getattr(t, "matrix", None)
        key.append((id(t), _tensor_key(m)))
        refs += [t, m]
        for st in (getattr(t, "transforms", None) or [t]):      # stages of a composite map
            sm = getattr(st, "matrix", None)
            key.append((id(st), _tensor_key(sm), getattr(st, "order", None),
                        getattr(st, "strength", None), getattr(st, "skew", None)))
            refs += [st, sm]
        for d in row:
            direction = getattr(d, "direction", None)
            geom = []
            for name in ("edges", "edges_x", "edges_y", "bandwidth", "bandwidth_x", "bandwidth_y"):
                v = getattr(d, name, None)
                if torch.is_tensor(v):
                    geom.append(_tensor_key(v))
                    refs.append(v)
                elif isinstance(v, (int, float)):
                    geom.append(float(v))
                elif isinstance(v, (tuple, list)) and all(isinstance(q, (int, float)) for q in v):
                    geom.append(tuple(float(q) for q in v))
            key.append((id(d), getattr(d, "kde", None), getattr(d, "axis", None), _tensor_key(direction), tuple(geom)))
            refs += [d, direction]
    return tuple(key), refs


_plan_cache: "OrderedDict[tuple, _Plan]" = OrderedDict()
_PLAN_CACHE_SIZE = 16


def _build_plan(x, transforms, diagnostics) -> _Plan:
    plan = _Plan()
    ndim, device = x.shape[1], x.device
    for i, (t, row) in enumerate(zip(transforms, diagnostics)):
        plan.shape.append(len(row))
        matrix = _linear_matrix(t)
        chain = _multipole_chain(t) if matrix is NotImplemented else None
        for j, d in enumerate(row):
            if chain is not None and type(d) is Histogram1D and ndim <= 8:
                # thin multipole between linear sections: folded into the projection kernel
                pre, kick, post = chain
                row_post = d.projection_vector(post.to(torch.float32) if post is not None else None, ndim, "cpu")
                vec, mp_row = multipole_terms(row_post, pre, kick, ndim)
                gkey = ("1d-mp", bool(d.kde), d.nbins)
                grp = plan.groups.get(gkey)
                if grp is None:
                    grp = plan.groups[gkey] = _Group("1d", bool(d.kde))
                    grp.mp = []
                grp.slots.append((i, j))
                grp.diags.append(d)
                grp.proj.append(vec.to(device))
                grp.mp.append(mp_row.to(device))
                continue
            if matrix is NotImplemented or type(d) not in (Histogram1D, Histogram2D):
                plan.fallback.append((i, j))
                continue
            if type(d) is Histogram1D:
                gkey = ("1d", bool(d.kde), d.nbins)
                vec = d.projection_vector(matrix, ndim, device)
            else:
                gkey = ("2d", bool(d.kde), d.shape)
                vec = d.projection_vectors(matrix, ndim, device)
            grp = plan.groups.get(gkey)
            if grp is None:
                grp = plan.groups[gkey] = _Group(gkey[0], gkey[1])
            grp.slots.append((i, j))
            grp.diags.append(d)
            grp.proj.append(vec)
    for grp in plan.groups.values():
        grp.proj = torch.stack(grp.proj).contiguous()
        if grp.mp is not None:
            grp.mp = torch.stack(grp.mp).contiguous()
    return plan


def _stacked_targets(grp: "_Group", targets, device) -> Optional[torch.Tensor]:
    """(K, B) stack of the measurements of a group's slots, cached on the identity of the tensors."""
    try:
        rows = [targets[i][j] for i, j in grp.slots]
    except (IndexError, TypeError):
        return None
    if not all(torch.is_tensor(m) and m.ndim == 1 and m.shape[0] == grp.diags[0].nbins for m in rows):
        return None
    key = tuple((id(m), m._version) for m in rows)
    hit = grp.cache.get("targets")
    if hit is None or hit[0] != key or hit[1].device != device:
        # `rows` is kept with the entry: the ids in the key stay owned by these very tensors
        hit = grp.cache["targets"] = (key, torch.stack([m.detach().to(device=device, dtype=torch.float32)
                                                        for m in rows]).contiguous(), rows)
    return hit[1]


def forward(x: torch.Tensor, transforms: List[nn.Module], diagnostics: List[List[nn.Module]],
            reducer: Optional[Callable] = None, stacked: Optional[list] = None,
            kl_targets=None) -> List[List[torch.Tensor]]:
    """Predicted profiles for every transform / diagnostic pair (simulate/simulate.py:8-33).

    ``stacked`` (optional list) receives one ``(slots, profiles)`` pair per fused group, where
    ``profiles`` is the (K, ...) tensor the returned rows are views of and ``slots`` the (i, j)
    positions they fill -- callers that reduce all profiles at once (MENTFlow.loss) use it to
    avoid K small kernels.  It is left empty if any pair needed the object-by-object path.
    ``kl_targets`` (optional, nested like the result): measured profiles; one-dimensional KDE
    groups then also evaluate KL(target || profile) inside the normalisation kernel and the
    ``stacked`` entries become ``(slots, profiles, kl)`` (kl is None for the other groups)."""
    pkey, refs = _plan_key(transforms, diagnostics)
    key = (pkey, x.shape[1], str(x.device))
    plan = _plan_cache.get(key)
    if plan is None:
        plan = _build_plan(x, transforms, diagnostics)
        plan.refs = refs
        _plan_cache[key] = plan
        while len(_plan_cache) > _PLAN_CACHE_SIZE:
            _plan_cache.popitem(last=False)
    else:
        _plan_cache.move_to_end(key)
    out: List[List[Optional[torch.Tensor]]] = [[None] * n for n in plan.shape]
    for grp in plan.groups.values():
        noisy = any(d.noise and d.noise_scale > 0.0 for d in grp.diags)
        kl = None
        if grp.kind == "1d":
            targ = None
            if kl_targets is not None and stacked is not None and grp.kde and not noisy and not plan.fallback:
                targ = _stacked_targets(grp, kl_targets, x.device)
            prof = profiles_1d(x, grp.proj, grp.diags, kde=grp.kde, reducer=reducer, cache=grp.cache,
                               kl_targets=targ, mp=grp.mp)
            if targ is not None:
                prof, kl = prof
        else:
            prof = profiles_2d(x, grp.proj, grp.diags, kde=grp.kde, reducer=reducer, cache=grp.cache)
        if stacked is not None and not noisy and not plan.fallback:
            stacked.append((grp.slots, prof, kl) if kl_targets is not None else (grp.slots, prof))
        for row, (i, j), d in zip(prof.unbind(0), grp.slots, grp.diags):
            out[i][j] = d.apply_noise(row) if noisy else row
    if plan.fallback:
        cache = {}
        for i, j in plan.fallback:
            if i not in cache:
                cache[i] = transforms[i](x.clone())
            out[i][j] = diagnostics[i][j](cache[i])
    return out


class Simulator:
    """simulate/simulate.py:36-47."""

    def __init__(self, transforms, diagnostics) -> None:
        self.transforms = transforms
        self.diagnostics = diagnostics

    def forward(self, x: torch.Tensor) -> List[List[torch.Tensor]]:
        return forward(x, self.transforms, self.diagnostics)
