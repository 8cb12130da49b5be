"""Thin torch layer over the C ABI: device pointers in, device pointers out.

Each function validates its tensors (CUDA, fp32, contiguous), allocates outputs/workspaces
with torch, and launches on torch's *current* stream (autograd runs backward on a worker
thread, so nothing here caches streams or keeps global state).  Differentiable ops are
``torch.autograd.Function`` s whose backward is again a hand-written kernel.
"""
from __future__ import annotations

import ctypes
import math
from typing import Optional

import torch

from . import _lib

GEOM_STRIDE = 8
FLAG_NO_TENSOR_CORES = 1            # MFB_FLAG_NO_TENSOR_CORES of the C ABI (per call; the library keeps no switches)
# Python-side choices between two implementations of the same result, read at call time (A/B tests)
KDE2D_USE_TENSOR_CORES = True
NSF_BWD_USE_TENSOR_CORES = True


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check_f32(name: str, t: torch.Tensor) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: mentflow_b200 kernels need CUDA tensors (got {t.device}); "
                           "there is no CPU fallback")
    if t.dtype != torch.float32:
        raise TypeError(f"{name}: expected float32, got {t.dtype}")
    if not t.is_contiguous() or t.data_ptr() % 16:
        t = t.contiguous()
        if t.data_ptr() % 16:
            t = t.clone()
    return t


# --------------------------------------------------------------------------------------
# supported bandwidths
# --------------------------------------------------------------------------------------
# A KDE kernel deposits a particle into the R bins on either side of its nearest bin, R = the smallest integer
# >= 8.85 sigma / delta - 1/2 (kde1d.cu window_radius): the taps it drops are below 1e-17 of the centre.  The windows are
# compiled for R = 4, 9 and 13 in 1-D, R = 4 and 9 for the 2-D fixed-point deposit and the 2-D backward; the 2-D
# tensor-core forward evaluates dense kernel rows and takes any bandwidth.  Wider kernels are refused here, before
# anything is launched, instead of failing inside the library with a generic error code.
KDE1D_MAX_RADIUS = 13
KDE2D_MAX_RADIUS = 9


def kde_window_radius(ratio: float) -> int:
    """Window radius the kernels use for sigma / bin spacing = ``ratio`` (<= 0 stands for the default 0.5)."""
    r = ctypes.c_float(ratio).value          # the C ABI takes the ratio as a float
    if r <= 0.0:
        r = 0.5
    return max(1, math.ceil(8.85 * r - 0.5))


def kde_max_ratio(radius: int) -> float:
    """Largest sigma / bin spacing whose window fits ``radius`` bins."""
    return (radius + 0.5) / 8.85


def check_kde_ratio(ratio: float, max_radius: int, what: str) -> None:
    """ValueError unless a kernel compiled up to ``max_radius`` covers sigma / bin spacing = ``ratio``."""
    if kde_window_radius(ratio) > max_radius:
        raise ValueError(f"{what}: KDE bandwidth too wide: sigma / bin spacing = {float(ratio):.4g}, the supported limit "
                         f"is {kde_max_ratio(max_radius):.4f} (a window of {max_radius} bins on either side); "
                         "use a smaller bandwidth or wider bins")


# --------------------------------------------------------------------------------------
# projection + KDE, 1-D screens
# --------------------------------------------------------------------------------------
def _check_mp(mp: torch.Tensor, k: int, d: int) -> torch.Tensor:
    mp = _check_f32("mp", mp)
    if mp.shape != (k, 2 * d + 4):
        raise ValueError(f"multipole terms must have shape ({k}, {2 * d + 4}), got {tuple(mp.shape)}")
    return mp


KL_PAD = 1.0e-12   # loss.py:15-17


def _kde1d_fwd(x, proj, geom, ratio, mp, sums, n_total=1.0, meas=None, prof=None, kl=None):
    """Deposit + merge into ``sums`` (K, B); with ``prof`` also normalise by ``n_total`` (+ KL against ``meas``)."""
    lib = _lib.load()
    check_kde_ratio(ratio, KDE1D_MAX_RADIUS, "1-D KDE")
    x, proj, geom = _check_f32("x", x), _check_f32("proj", proj), _check_f32("geom", geom)
    n, d = x.shape
    k, nbins = sums.shape
    if mp is not None:
        mp = _check_mp(mp, k, d)
    with torch.cuda.device(x.device):
        wbytes = lib.mfb_kde1d_workspace_bytes(n, d, k, nbins)
        work = torch.empty(max(wbytes, 16), dtype=torch.uint8, device=x.device)
        _lib.check(lib.mfb_project_kde1d_fwd(_ptr(x), n, d, _ptr(proj), _ptr(mp), _ptr(geom), k, nbins, float(ratio),
                                             float(n_total), _ptr(meas), KL_PAD, _ptr(sums), _ptr(prof), _ptr(kl),
                                             _ptr(work), wbytes, _stream()), "project_kde1d_fwd")


def kde1d_sums(x: torch.Tensor, proj: torch.Tensor, geom: torch.Tensor, ratio: float, nbins: int,
               mp: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """S[k, b] = sum_n exp(-0.5 ((u_kn - c_b) / sigma_k)^2)  (unnormalised), u_kn = proj_k . x_n, plus the
    multipole terms of ``mp`` (K, 2D+4) when given (see ``simulate.multipole_terms``)."""
    sums = out if out is not None else torch.empty((proj.shape[0], nbins), dtype=torch.float32, device=x.device)
    _kde1d_fwd(x, proj, geom, ratio, mp, sums)
    return sums


def kde1d_grad_x(x, proj, geom, ratio, gsums, mp: Optional[torch.Tensor] = None):
    lib = _lib.load()
    check_kde_ratio(ratio, KDE1D_MAX_RADIUS, "1-D KDE backward")
    n, d = x.shape
    k, b = gsums.shape
    if mp is not None:
        mp = _check_mp(mp, k, d)
    gx = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(lib.mfb_project_kde1d_bwd(_ptr(x), n, d, _ptr(proj), _ptr(mp), _ptr(geom), k, b, float(ratio),
                                             _ptr(gsums), _ptr(gx), 0, _stream()), "project_kde1d_bwd")
    return gx


def kde1d_loss_forward(x, proj, geom, ratio, nbins, n_total, meas, mp=None):
    """Deposit + merge + normalise (+ KL against ``meas``) in two launches: (sums, profiles, kl)."""
    sums = torch.empty((proj.shape[0], nbins), dtype=torch.float32, device=x.device)
    prof = torch.empty_like(sums)
    kl = torch.empty(proj.shape[0], dtype=torch.float32, device=x.device) if meas is not None else None
    _kde1d_fwd(x, proj, geom, ratio, mp, sums, n_total, meas, prof, kl)
    return sums, prof, kl


def kde1d_finish(sums, n_total, geom, meas):
    """Normalise merged sums (+ KL against ``meas``): (profiles, kl)."""
    lib = _lib.load()
    k, b = sums.shape
    prof = torch.empty_like(sums)
    kl = torch.empty(k, dtype=torch.float32, device=sums.device) if meas is not None else None
    with torch.cuda.device(sums.device):
        _lib.check(lib.mfb_kde1d_finish(_ptr(sums), float(n_total), _ptr(geom), k, b, _ptr(meas), KL_PAD,
                                        _ptr(prof), _ptr(kl), _stream()), "kde1d_finish")
    return prof, kl


def kde1d_finish_bwd(sums, n_total, geom, meas, gprof, gkl):
    lib = _lib.load()
    k, b = sums.shape
    gprof = _check_f32("gprof", gprof) if gprof is not None else None
    gkl = _check_f32("gkl", gkl) if gkl is not None else None
    gsums = torch.empty_like(sums)
    with torch.cuda.device(sums.device):
        _lib.check(lib.mfb_kde1d_finish_bwd(_ptr(sums), float(n_total), _ptr(geom), k, b, _ptr(meas), KL_PAD,
                                            _ptr(gprof), _ptr(gkl), _ptr(gsums), _stream()), "kde1d_finish_bwd")
    return gsums


def kde1d_loss_forward_p2p(peer, x, proj, geom, ratio, nbins, tail, n_total, meas):
    """Sharded forward tail in two launches: deposit, then merge + cross-rank sum over NVLink peer memory +
    normalisation (+ KL).  Returns (sums, profiles, kl, tail_sum)."""
    lib = _lib.load()
    check_kde_ratio(ratio, KDE1D_MAX_RADIUS, "1-D KDE")
    x, proj, geom = _check_f32("x", x), _check_f32("proj", proj), _check_f32("geom", geom)
    n, d = x.shape
    k = proj.shape[0]
    nt = 0 if tail is None else int(tail.numel())
    block, handle, ptrs, state = peer.block_for(k, nbins, nt, x.device)
    sums = torch.empty((k, nbins), dtype=torch.float32, device=x.device)
    prof = torch.empty_like(sums)
    kl = torch.empty(k, dtype=torch.float32, device=x.device) if meas is not None else None
    tail_out = torch.empty(nt, dtype=torch.float64, device=x.device) if nt else None
    arr = (ctypes.c_uint64 * len(ptrs))(*ptrs)
    with torch.cuda.device(x.device):
        wbytes = lib.mfb_kde1d_workspace_bytes(n, d, k, nbins)
        work = torch.empty(max(wbytes, 16), dtype=torch.uint8, device=x.device)
        _lib.check(lib.mfb_project_kde1d_loss_fwd_p2p(_ptr(x), n, d, _ptr(proj), _ptr(geom), k, nbins, float(ratio),
                                                      float(n_total), _ptr(meas), KL_PAD, ctypes.cast(arr, ctypes.c_void_p),
                                                      peer.rank, peer.world, _ptr(state), _ptr(tail), nt, _ptr(sums),
                                                      _ptr(prof), _ptr(kl), _ptr(tail_out), _ptr(work), wbytes, _stream()),
                   "project_kde1d_loss_fwd_p2p")
    return sums, prof, kl, tail_out


def kde1d_finish_p2p(peer, sums_local, tail, n_total, geom, meas):
    """Cross-rank sum over NVLink peer memory + normalisation (+ KL) in one kernel: (sums, profiles, kl, tail_sum).
    ``peer``: ``distributed.PeerExchange``; ``tail``: float64 vector reduced alongside (or None)."""
    lib = _lib.load()
    k, b = sums_local.shape
    nt = 0 if tail is None else int(tail.numel())
    block, handle, ptrs, state = peer.block_for(k, b, nt, sums_local.device)
    sums = torch.empty_like(sums_local)
    prof = torch.empty_like(sums_local)
    kl = torch.empty(k, dtype=torch.float32, device=sums_local.device) if meas is not None else None
    tail_out = torch.empty(nt, dtype=torch.float64, device=sums_local.device) if nt else None
    arr = (ctypes.c_uint64 * len(ptrs))(*ptrs)
    with torch.cuda.device(sums_local.device):
        _lib.check(lib.mfb_kde1d_finish_p2p(ctypes.cast(arr, ctypes.c_void_p), peer.rank, peer.world, _ptr(state),
                                            _ptr(sums_local), _ptr(tail), nt, float(n_total), _ptr(geom), k, b, _ptr(meas),
                                            KL_PAD, _ptr(sums), _ptr(prof), _ptr(kl), _ptr(tail_out), _stream()),
                   "kde1d_finish_p2p")
    return sums, prof, kl, tail_out


class ProjectKDE1D(torch.autograd.Function):
    """profiles[k, b] of K one-dimensional screens, differentiable w.r.t. the particles.

    ``reducer`` (optional) all-reduces the unnormalised sums across ranks *before* the
    non-linear normalisation and returns the global particle count (SURVEY.md 8e).
    ``meas`` (optional, (K, B)): also return kl[k] = KL(meas_k || profile_k) of loss.py:15-17,
    evaluated by the same kernel that normalises.
    """

    @staticmethod
    def forward(ctx, x, proj, geom, ratio, nbins, reducer, meas, mp=None):
        ctx.set_materialize_grads(False)
        check_kde_ratio(ratio, KDE1D_MAX_RADIUS, "1-D KDE")      # before any launch or cross-rank exchange
        x = _check_f32("x", x)
        n_total = float(x.shape[0])
        if meas is not None:
            meas = _check_f32("meas", meas)
        peer = getattr(reducer, "peer", None)
        if reducer is None and x.shape[0] > 0:
            sums, prof, kl = kde1d_loss_forward(x, proj, geom, ratio, nbins, n_total, meas, mp)
        elif (peer is not None and mp is None and x.shape[0] > 0 and proj.shape[0] <= 1024 and nbins <= 4096
                and (proj.shape[0] * nbins) % 2 == 0):
            # sharded: the cross-rank sum happens inside the tail kernel, over NVLink peer memory
            n_total = reducer.global_count(n_total)
            stash = reducer.take_stash()
            sums, prof, kl, tail_sum = kde1d_loss_forward_p2p(peer, x, proj, geom, ratio, nbins, stash, n_total, meas)
            if stash is not None:
                reducer.set_stash_result(tail_sum)
            reducer.calls += 1
        else:
            # sharded: the unnormalised sums are all-reduced before the non-linear tail; float64 partial sums
            # another op stashed on the reducer (the entropy moments) ride at the end of the same buffer
            tail = reducer.tail_floats() if hasattr(reducer, "tail_floats") else 0
            if tail:
                flat = torch.empty(proj.shape[0] * nbins + tail, dtype=torch.float32, device=x.device)
                sums = kde1d_sums(x, proj, geom, ratio, nbins, mp, out=flat[: proj.shape[0] * nbins].view(-1, nbins))
                n_total = reducer(sums, n_total, flat=flat)
            else:
                sums = kde1d_sums(x, proj, geom, ratio, nbins, mp)
                if reducer is not None:
                    n_total = reducer(sums, n_total)
            prof, kl = kde1d_finish(sums, n_total, geom, meas)
        ctx.save_for_backward(x, proj, geom, sums, meas, mp)
        ctx.ratio, ctx.n_total = ratio, n_total
        if meas is None:
            return prof
        return prof, kl

    @staticmethod
    def backward(ctx, gprof, gkl=None):
        x, proj, geom, sums, meas, mp = ctx.saved_tensors
        if gprof is None and gkl is None:
            return None, None, None, None, None, None, None, None
        gsums = kde1d_finish_bwd(sums, ctx.n_total, geom, meas, gprof, gkl if meas is not None else None)
        gx = kde1d_grad_x(x, proj, geom, ctx.ratio, gsums, mp=mp)
        return gx, None, None, None, None, None, None, None


def project_kde1d(x, proj, geom, ratio, nbins, reducer=None, meas=None, mp=None):
    """(K, B) profiles; with ``meas`` a pair (profiles, kl[K]); ``mp``: multipole terms (K, 2D+4)."""
    return ProjectKDE1D.apply(x, proj, geom, ratio, nbins, reducer, meas, mp)


# --------------------------------------------------------------------------------------
# projection + exact histogram, 1-D screens
# --------------------------------------------------------------------------------------
def project_hist1d(x: torch.Tensor, proj: torch.Tensor, edges: torch.Tensor,
                   counts: Optional[torch.Tensor] = None, mp: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int64 counts[k, b]; edges is (K, B+1).  Adds into ``counts`` when given.  ``mp``: multipole
    terms (K, 2D+4) of the transfer maps, see ``simulate.multipole_terms``."""
    lib = _lib.load()
    x, proj, edges = _check_f32("x", x), _check_f32("proj", proj), _check_f32("edges", edges)
    n, d = x.shape
    k, b = proj.shape[0], edges.shape[1] - 1
    if counts is None:
        counts = torch.zeros((k, b), dtype=torch.int64, device=x.device)
    if n == 0:              # nothing to count
        return counts
    if mp is not None:
        mp = _check_mp(mp, k, d)
    with torch.cuda.device(x.device):
        _lib.check(lib.mfb_project_hist1d(_ptr(x), n, d, _ptr(proj), _ptr(mp), _ptr(edges), k, b, _ptr(counts),
                                          _stream()), "project_hist1d")
    return counts


# --------------------------------------------------------------------------------------
# 2-D screens
# --------------------------------------------------------------------------------------
def kde2d_sums(x, proj, geom, ratio, bx, by):
    """(sums float32 [K,bx,by], acc int64 [2,K,bx,by]): acc holds the exact fixed-point
    accumulators (plane 0: value * 2^22, plane 1: remainder * 2^44) that ranks all-reduce."""
    lib = _lib.load()
    x, proj, geom = _check_f32("x", x), _check_f32("proj", proj), _check_f32("geom", geom)
    n, d = x.shape
    k = proj.shape[0]
    flags = 0 if KDE2D_USE_TENSOR_CORES else FLAG_NO_TENSOR_CORES
    if not lib.mfb_kde2d_uses_tensor_cores(n, d, bx, by, flags):     # the windowed fixed-point deposit
        check_kde_ratio(ratio, KDE2D_MAX_RADIUS, "2-D KDE (fixed-point deposit)")
    sums = torch.empty((k, bx, by), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        # workspace = the two int64 planes, then the per-CTA partial screens of the tensor-core path
        wbytes = int(lib.mfb_kde2d_workspace_bytes(n, d, k, bx, by))
        work = torch.empty((wbytes + 7) // 8, dtype=torch.int64, device=x.device)
        _lib.check(lib.mfb_project_kde2d_fwd(_ptr(x), n, d, _ptr(proj), _ptr(geom), k, bx, by, float(ratio),
                                             _ptr(sums), _ptr(work), wbytes, flags, _stream()),
                   "project_kde2d_fwd")
    acc = work[: 2 * k * bx * by].view(2, k, bx, by)
    return sums, acc


def kde2d_normalize(sums, geom):
    lib = _lib.load()
    k, bx, by = sums.shape
    prof = torch.empty_like(sums)
    with torch.cuda.device(sums.device):
        _lib.check(lib.mfb_kde2d_normalize(_ptr(sums), _ptr(geom), k, bx, by, _ptr(prof), _stream()),
                   "kde2d_normalize")
    return prof


class ProjectKDE2D(torch.autograd.Function):
    """profiles[k, a, b] of K two-dimensional screens, differentiable w.r.t. the particles."""

    @staticmethod
    def forward(ctx, x, proj, geom, ratio, bx, by, reducer):
        x = _check_f32("x", x)
        sums, acc = kde2d_sums(x, proj, geom, ratio, bx, by)
        if reducer is not None:
            reducer(acc, float(x.shape[0]))          # exact integer all-reduce
            sums = (acc[0].to(torch.float64) * 2.0 ** -22 + acc[1].to(torch.float64) * 2.0 ** -44).to(torch.float32)
        prof = kde2d_normalize(sums, geom)
        ctx.save_for_backward(x, proj, geom, sums)
        ctx.ratio = ratio
        return prof

    @staticmethod
    def backward(ctx, gprof):
        lib = _lib.load()
        check_kde_ratio(ctx.ratio, KDE2D_MAX_RADIUS, "2-D KDE backward")
        x, proj, geom, sums = ctx.saved_tensors
        k, bx, by = sums.shape
        gprof = _check_f32("gprof", gprof)
        gsums = torch.empty_like(sums)
        gx = torch.empty_like(x)
        n, d = x.shape
        with torch.cuda.device(x.device):
            _lib.check(lib.mfb_kde2d_normalize_bwd(_ptr(sums), _ptr(geom), k, bx, by, _ptr(gprof), _ptr(gsums),
                                                   _stream()), "kde2d_normalize_bwd")
            _lib.check(lib.mfb_project_kde2d_bwd(_ptr(x), n, d, _ptr(proj), _ptr(geom), k, bx, by,
                                                 float(ctx.ratio), _ptr(gsums), _ptr(gx), 0, _stream()),
                       "project_kde2d_bwd")
        return gx, None, None, None, None, None, None


def project_kde2d(x, proj, geom, ratio, bx, by, reducer=None):
    if torch.is_grad_enabled() and x.requires_grad:
        # the backward is windowed at any batch size: refuse now rather than in backward()
        check_kde_ratio(ratio, KDE2D_MAX_RADIUS, "2-D KDE backward (x requires grad)")
    return ProjectKDE2D.apply(x, proj, geom, ratio, bx, by, reducer)


def project_hist2d(x, proj, edges_x, edges_y, counts=None):
    """int64 counts[k, a, b]; edges_x (K, bx+1), edges_y (K, by+1)."""
    lib = _lib.load()
    x, proj = _check_f32("x", x), _check_f32("proj", proj)
    edges_x, edges_y = _check_f32("edges_x", edges_x), _check_f32("edges_y", edges_y)
    n, d = x.shape
    k, bx, by = proj.shape[0], edges_x.shape[1] - 1, edges_y.shape[1] - 1
    if counts is None:
        counts = torch.zeros((k, bx, by), dtype=torch.int64, device=x.device)
    if n == 0:              # nothing to count
        return counts
    with torch.cuda.device(x.device):
        _lib.check(lib.mfb_project_hist2d(_ptr(x), n, d, _ptr(proj), _ptr(edges_x), _ptr(edges_y), k, bx, by,
                                          _ptr(counts), _stream()), "project_hist2d")
    return counts


# --------------------------------------------------------------------------------------
# neural spline flow
# --------------------------------------------------------------------------------------
def nsf_layer_param_floats(d: int, hidden_units: int, hidden_layers: int, bins: int) -> int:
    return int(_lib.load().mfb_nsf_layer_param_floats(d, hidden_units, hidden_layers, bins))


NSF_USE_TENSOR_CORES = True   # tcgen05 conditioner where the configuration is compiled; False = fp32 CUDA-core kernel


def orders_autoregressive(orders) -> bool:
    """every layer's order is a permutation (strict autoregressive ordering; coupling layers repeat values)"""
    return all(sorted(int(v) for v in o) == list(range(len(o))) for o in orders)


def nsf_tc_supported(d: int, hidden_units: int, hidden_layers: int, bins: int, orders=None) -> bool:
    """the tcgen05 layer kernels are compiled for this shape (and, when ``orders`` is given, these orderings)"""
    if orders is not None and not orders_autoregressive(orders):
        return False
    return bool(NSF_USE_TENSOR_CORES and _lib.load().mfb_nsf_tc_supported(d, hidden_units, hidden_layers, bins))


def nsf_tc_images(packed, orders, hidden_units, hidden_layers, bins):
    """fp16 (hi, lo) SWIZZLE_128B operand images of every layer's masked weights, (T, bytes) uint8;
    built on the device from the packed fp32 parameters (one small launch per forward call)."""
    lib = _lib.load()
    packed = _check_f32("packed", packed)
    t_layers, d = len(orders), len(orders[0])
    nbytes = int(lib.mfb_nsf_tc_image_bytes(d, hidden_layers))
    images = torch.empty((t_layers, nbytes), dtype=torch.uint8, device=packed.device)
    order_arr = (ctypes.c_int32 * (t_layers * d))(*[int(o) for order in orders for o in order])
    with torch.cuda.device(packed.device):
        _lib.check(lib.mfb_nsf_tc_prepare(_ptr(packed), packed.stride(0), t_layers, d, hidden_units, hidden_layers,
                                          bins, ctypes.cast(order_arr, ctypes.c_void_p), _ptr(images), _stream()),
                   "nsf_tc_prepare")
    return images


def nsf_direction_images(use, packed, orders, hidden_units, hidden_layers, bins, images=None):
    """The operand images one direction of the flow runs its layers from, or None for the fp32 CUDA-core kernels.
    None unless ``use`` (the direction's switch) is set and the tcgen05 kernels are compiled for this shape and
    these orders; then ``images`` when the caller has them for these weights, else built here."""
    d = len(orders[0])
    if not (use and orders_autoregressive(orders) and _lib.load().mfb_nsf_tc_supported(d, hidden_units, hidden_layers,
                                                                                        bins)):
        return None
    return images if images is not None else nsf_tc_images(packed, orders, hidden_units, hidden_layers, bins)


def nsf_layer_forward(v, params, order, hidden_units, hidden_layers, bins, logq_in, first_layer,
                      want_logq=True, image=None):
    """One autoregressive spline layer: returns (y, logq_out).  With ``image`` (one row of
    ``nsf_tc_images``) the tensor-core kernel runs, otherwise the fp32 CUDA-core kernel."""
    lib = _lib.load()
    v = _check_f32("v", v)
    params = _check_f32("params", params)
    n, d = v.shape
    y = torch.empty_like(v)
    logq_out = torch.empty(n, dtype=torch.float32, device=v.device) if want_logq else None
    if n == 0:          # an empty batch has no storage to point at: nothing to launch
        return y, logq_out
    order_arr = (ctypes.c_int32 * d)(*[int(o) for o in order])
    with torch.cuda.device(v.device):
        _lib.check(lib.mfb_nsf_layer_fwd(_ptr(v), n, d, hidden_units, hidden_layers, bins, _ptr(params), _ptr(image),
                                         ctypes.cast(order_arr, ctypes.c_void_p), _ptr(logq_in),
                                         1 if first_layer else 0, _ptr(y), _ptr(logq_out), _stream()),
                   "nsf_layer_fwd")
    return y, logq_out


def _nsf_run_layers(z, packed, orders, hidden_units, hidden_layers, bins, want_logq, images):
    """All layers in sampling order; returns ([z, y_1, ..., x], log q).  ``images``: the forward's
    operand images (``nsf_direction_images``), None for the CUDA-core kernel."""
    steps, logq = [z], None
    for t, order in enumerate(orders):
        y, logq = nsf_layer_forward(steps[-1], packed[t], order, hidden_units, hidden_layers, bins, logq,
                                    first_layer=(t == 0), want_logq=want_logq,
                                    image=None if images is None else images[t])
        steps.append(y)
    return steps, logq


# --------------------------------------------------------------------------------------
# moments
# --------------------------------------------------------------------------------------
def moments(x: torch.Tensor, logq: Optional[torch.Tensor], with_cov: bool = False) -> torch.Tensor:
    """float64 vector: [sum logq, sum |x|^2] (+ [sum x_i, sum x_i x_j] with ``with_cov``)."""
    lib = _lib.load()
    x = _check_f32("x", x)
    if logq is not None:
        logq = _check_f32("logq", logq)
    n, d = x.shape
    m = 2 + d + d * d if with_cov else 2      # every entry is written by the kernel
    out = torch.empty(m, dtype=torch.float64, device=x.device)
    with torch.cuda.device(x.device):
        wbytes = lib.mfb_moments_workspace_bytes(n, d)
        work = torch.empty(max(wbytes, 16), dtype=torch.uint8, device=x.device)
        _lib.check(lib.mfb_moments(_ptr(x), _ptr(logq), n, d, 1 if with_cov else 0, _ptr(out), _ptr(work), wbytes,
                                   _stream()), "moments")
    return out


def mc_entropy(sums: torch.Tensor, a: float, b: float, c: float) -> torch.Tensor:
    """float32 scalar a * sums[0] + b * sums[1] - c, evaluated in double by one launch."""
    lib = _lib.load()
    assert sums.dtype == torch.float64 and sums.numel() >= 2 and sums.is_contiguous()
    h = torch.empty((), dtype=torch.float32, device=sums.device)
    with torch.cuda.device(sums.device):
        _lib.check(lib.mfb_mc_entropy(_ptr(sums), float(a), float(b), float(c), _ptr(h), _stream()), "mc_entropy")
    return h


class LossTail(torch.autograd.Function):
    """L = H + mu * mean(D) as one launch (core.py:111-113); dL/dH = 1, dL/dD_k = mu / K."""

    @staticmethod
    def forward(ctx, h, d, mu):
        lib = _lib.load()
        dd = _check_f32("d", d.detach())
        hh = None if h is None else _check_f32("h", h.detach())
        out = torch.empty(2, dtype=torch.float32, device=dd.device)
        with torch.cuda.device(dd.device):
            _lib.check(lib.mfb_loss_tail(_ptr(dd), dd.numel(), _ptr(hh), float(mu), _ptr(out), _stream()), "loss_tail")
        ctx.k, ctx.mu, ctx.shape, ctx.has_h = dd.numel(), float(mu), d.shape, h is not None
        return out[0]

    @staticmethod
    def backward(ctx, g):
        gd = (g * (ctx.mu / ctx.k)).expand(ctx.shape)
        return (g if ctx.has_h else None), gd, None


def f64_split(values: torch.Tensor, out: torch.Tensor) -> None:
    """float64 (n,) -> float32 (2n,) [hi | lo] written into ``out`` (a slice of an all-reduce buffer)."""
    lib = _lib.load()
    n = values.numel()
    assert values.dtype == torch.float64 and out.dtype == torch.float32 and out.numel() == 2 * n and out.is_contiguous()
    with torch.cuda.device(values.device):
        _lib.check(lib.mfb_f64_split(_ptr(values), n, _ptr(out), _stream()), "f64_split")


def f64_join(pairs: torch.Tensor) -> torch.Tensor:
    lib = _lib.load()
    n = pairs.numel() // 2
    out = torch.empty(n, dtype=torch.float64, device=pairs.device)
    with torch.cuda.device(pairs.device):
        _lib.check(lib.mfb_f64_join(_ptr(pairs), n, _ptr(out), _stream()), "f64_join")
    return out


# --------------------------------------------------------------------------------------
# k-th nearest neighbour (k-NN entropy)
# --------------------------------------------------------------------------------------
KNN_MAX_K = 16
KNN_MAX_DIM = 8


class KNNKth(torch.autograd.Function):
    """(r, idx, logsum) of ``knn_kth``; only ``logsum`` carries a gradient, with the neighbours held fixed."""

    @staticmethod
    def forward(ctx, x, k, pad):
        lib = _lib.load()
        x = _check_f32("x", x.detach())
        n, d = x.shape
        r = torch.empty(n, dtype=torch.float32, device=x.device)
        idx = torch.empty(n, dtype=torch.int32, device=x.device)
        logsum = torch.empty((), dtype=torch.float64, device=x.device)
        with torch.cuda.device(x.device):
            wbytes = lib.mfb_knn_workspace_bytes(n, d, k)
            work = torch.empty(max(wbytes, 16), dtype=torch.uint8, device=x.device)
            _lib.check(lib.mfb_knn_kth(_ptr(x), n, d, k, float(pad), _ptr(r), _ptr(idx), _ptr(logsum), _ptr(work),
                                       wbytes, _stream()), "knn_kth")
        ctx.save_for_backward(x, r, idx)
        ctx.pad = float(pad)
        ctx.mark_non_differentiable(r, idx)
        return r, idx, logsum

    @staticmethod
    def backward(ctx, _gr, _gidx, glogsum):
        x, r, idx = ctx.saved_tensors
        return knn_kth_bwd(x, r, idx, glogsum, ctx.pad), None, None


def knn_check(n: int, d: int, k: int, what: str = "knn_kth") -> None:
    """ValueError unless the k-NN kernels take a batch of ``n`` particles in ``d`` dimensions at this ``k``."""
    if not 1 <= k <= KNN_MAX_K:
        raise ValueError(f"{what}: k = {k} is outside [1, {KNN_MAX_K}]")
    if k >= n:
        raise ValueError(f"{what}: k = {k} needs more than k particles (got N = {n})")
    if not 1 <= d <= KNN_MAX_DIM:
        raise ValueError(f"{what}: d = {d} is outside [1, {KNN_MAX_DIM}]")
    if n >= 2 ** 31:
        raise ValueError(f"{what}: N = {n} does not fit the int32 neighbour indices")


def knn_rows(rows: Optional[slice], n: int, what: str = "knn_kth"):
    """(row0, nrows) of a row range given as a slice of the batch, ``None`` for the whole batch; ValueError unless it
    is a contiguous range inside [0, n]."""
    if rows is None:
        return 0, n
    if not isinstance(rows, slice) or rows.step not in (None, 1):
        raise ValueError(f"{what}: rows must be a slice with step 1 (got {rows!r})")
    start = 0 if rows.start is None else int(rows.start)
    stop = n if rows.stop is None else int(rows.stop)
    if not 0 <= start <= stop <= n:
        raise ValueError(f"{what}: rows [{start}, {stop}) is not a range inside [0, {n}]")
    return start, stop - start


def knn_kth(x: torch.Tensor, k: int, pad: float = 1.0e-12, rows: Optional[slice] = None):
    """Distance ``r`` (float32, (N,)) from every particle to its k-th nearest other particle, that neighbour's index
    ``idx`` (int32; ties go to the smaller index) and ``logsum`` = sum log(r + pad) (float64 0-dim tensor, the only
    differentiable output).  A particle without k others at a finite distance (NaN or inf coordinates) gets r = inf and
    idx = its own index, which carries no gradient.  All pairs on the GPU: O(N^2 d).

    ``rows``: a slice of the batch (a rank's ``distributed.shard_slice`` of gathered particles).  Only those rows are
    searched, against every particle of ``x``; the result is ``(r, idx, None)`` for those rows, bit for bit the rows of
    the whole-batch call, with idx indexing ``x``.  There is no log sum (it needs every row: ``knn_logsum`` of the
    concatenated r) and no autograd (``knn_kth_bwd`` gives the gradient of those rows)."""
    if not isinstance(x, torch.Tensor) or x.dim() != 2:
        raise ValueError("knn_kth: x must be a (N, d) tensor")
    n, d = x.shape
    k = int(k)
    knn_check(n, d, k)
    if rows is None:
        _check_f32("x", x)
        return KNNKth.apply(x, k, float(pad))
    row0, nrows = knn_rows(rows, n)
    x = _check_f32("x", x.detach())
    r = torch.empty(nrows, dtype=torch.float32, device=x.device)
    idx = torch.empty(nrows, dtype=torch.int32, device=x.device)
    lib = _lib.load()
    with torch.cuda.device(x.device):
        wbytes = lib.mfb_knn_rows_workspace_bytes(n, nrows, d, k)
        work = torch.empty(max(wbytes, 16), dtype=torch.uint8, device=x.device)
        _lib.check(lib.mfb_knn_kth_rows(_ptr(x), n, d, k, row0, nrows, _ptr(r), _ptr(idx), _ptr(work), wbytes,
                                        _stream()), "knn_kth_rows")
    return r, idx, None


def knn_logsum(r: torch.Tensor, pad: float = 1.0e-12) -> torch.Tensor:
    """sum log(r + pad) over the k-th neighbour distances ``r`` of a whole batch (float64 0-dim tensor), added in the
    order ``knn_kth`` adds them: for r gathered from row ranges it is bit for bit ``knn_kth``'s logsum."""
    if not isinstance(r, torch.Tensor) or r.dim() != 1 or r.numel() < 1:
        raise ValueError("knn_logsum: r must be a non-empty (N,) tensor")
    if r.numel() >= 2 ** 31:
        raise ValueError(f"knn_logsum: N = {r.numel()} does not fit the int32 neighbour indices")
    r = _check_f32("r", r.detach())
    n = r.numel()
    logsum = torch.empty((), dtype=torch.float64, device=r.device)
    wbytes = 8 * (-(-n // 256))
    work = torch.empty(wbytes, dtype=torch.uint8, device=r.device)
    lib = _lib.load()
    with torch.cuda.device(r.device):
        _lib.check(lib.mfb_knn_logsum(_ptr(r), n, float(pad), _ptr(logsum), _ptr(work), wbytes, _stream()),
                   "knn_logsum")
    return logsum


def knn_kth_bwd(x: torch.Tensor, r: torch.Tensor, idx: torch.Tensor, glogsum: torch.Tensor, pad: float = 1.0e-12,
                rows: Optional[slice] = None) -> torch.Tensor:
    """glogsum * d logsum / dx for the rows ``rows`` of the batch (all rows for None), the neighbours held fixed:
    bit for bit those rows of ``knn_kth``'s gradient.  ``x``, ``r`` and ``idx`` are the whole batch's (the gathered
    particles and the concatenated results of the row ranges); ``glogsum`` is a float64 scalar tensor."""
    if not isinstance(x, torch.Tensor) or x.dim() != 2:
        raise ValueError("knn_kth_bwd: x must be a (N, d) tensor")
    n, d = x.shape
    if not 1 <= d <= KNN_MAX_DIM:
        raise ValueError(f"knn_kth_bwd: d = {d} is outside [1, {KNN_MAX_DIM}]")
    if not 2 <= n < 2 ** 31:
        raise ValueError(f"knn_kth_bwd: N = {n} is outside [2, 2^31)")
    if r.shape != (n,) or idx.shape != (n,) or idx.dtype != torch.int32:
        raise ValueError("knn_kth_bwd: r (float32) and idx (int32) must hold one entry per particle of x")
    if r.device != x.device or idx.device != x.device:
        raise ValueError(f"knn_kth_bwd: x, r and idx must be on one device (got {x.device}, {r.device}, {idx.device})")
    row0, nrows = knn_rows(rows, n, "knn_kth_bwd")
    x = _check_f32("x", x.detach())
    gx = torch.empty((nrows, d), dtype=torch.float32, device=x.device)
    if nrows == 0:
        return gx
    r = _check_f32("r", r.detach())
    idx = idx.contiguous()
    sorted_idx, perm = torch.sort(idx, stable=True)     # particle i's incoming neighbours, ascending j
    g = glogsum.detach().to(device=x.device, dtype=torch.float64).reshape(()).contiguous()
    lib = _lib.load()
    with torch.cuda.device(x.device):
        _lib.check(lib.mfb_knn_kth_bwd_rows(_ptr(x), n, d, _ptr(r), _ptr(idx), _ptr(sorted_idx), _ptr(perm), row0,
                                            nrows, float(pad), _ptr(g), _ptr(gx), _stream()), "knn_kth_bwd_rows")
    return gx


# --------------------------------------------------------------------------------------
# sliced Wasserstein distance: projections, stable radix sort, 1-D quantile integral
# --------------------------------------------------------------------------------------
SWD_MAX_DIM = 8
SWD_MAX_CHUNK = 65535               # directions per chunk (the library's grid limit)
SWD_WORKSPACE_CAP = 1 << 30         # bytes of sort workspace per call; the directions are sorted in chunks that fit
                                    # (about 16.5 bytes per particle and direction)


def check_swd_points(name: str, t, d: Optional[int] = None) -> None:
    """Refuse anything but a (N, d) tensor with 1 <= d <= 8, 1 <= N < 2^31 (and d equal to ``d`` when given)."""
    if not isinstance(t, torch.Tensor) or t.dim() != 2:
        raise ValueError(f"{name} must be a (N, d) tensor")
    n, dd = t.shape
    if not 1 <= dd <= SWD_MAX_DIM:
        raise ValueError(f"{name}: d = {dd} is outside [1, {SWD_MAX_DIM}]")
    if d is not None and dd != d:
        raise ValueError(f"{name} has d = {dd}, the samples have d = {d}")
    if not 1 <= n < 2 ** 31:
        raise ValueError(f"{name}: N = {n} is outside [1, 2^31)")


def check_swd_p(p) -> float:
    p = float(p)
    if not (math.isfinite(p) and p >= 1.0):
        raise ValueError(f"p = {p} must be finite and >= 1")
    return p


def _swd_theta(theta, d: int) -> None:
    if not isinstance(theta, torch.Tensor) or theta.dim() != 2 or theta.shape[1] != d or theta.shape[0] < 1:
        raise ValueError(f"theta must be a (P, {d}) tensor of directions with P >= 1")
    if theta.requires_grad:
        raise ValueError("theta requires grad, but the sliced Wasserstein kernels differentiate only x")


def _swd_workspace(lib, n: int, nproj: int, device):
    per = int(lib.mfb_swd_workspace_bytes(n, 1))
    chunk = max(1, min(nproj, SWD_MAX_CHUNK, SWD_WORKSPACE_CAP // per))
    wbytes = int(lib.mfb_swd_workspace_bytes(n, chunk))
    return torch.empty(wbytes, dtype=torch.uint8, device=device), wbytes


def swd_sort(x: torch.Tensor, theta: torch.Tensor):
    """Projections u = x theta_k (fp32 fused multiply-add chains from zero, coordinates in ascending order) of every
    direction (row of ``theta``, (P, d)), sorted stably: returns ``sorted`` ((P, N) float32) and ``perm`` ((P, N)
    int32, the particle index of each entry; ties keep index order, -0 and +0 compare equal, NaN sorts last).  An
    8-bit LSD radix sort on the GPU; not differentiable."""
    check_swd_points("x", x)
    n, d = x.shape
    _swd_theta(theta, d)
    x = _check_f32("x", x.detach())
    theta = _check_f32("theta", theta)
    nproj = theta.shape[0]
    lib = _lib.load()
    sorted_ = torch.empty((nproj, n), dtype=torch.float32, device=x.device)
    perm = torch.empty((nproj, n), dtype=torch.int32, device=x.device)
    with torch.cuda.device(x.device):
        work, wbytes = _swd_workspace(lib, n, nproj, x.device)
        _lib.check(lib.mfb_swd_sort(_ptr(x), n, d, _ptr(theta), nproj, _ptr(sorted_), _ptr(perm), _ptr(work), wbytes,
                                    _stream()), "swd_sort")
    return sorted_, perm


class SWDWpp(torch.autograd.Function):
    """(P,) float64 W_p^p of ``swd_wpp``; only x gets a gradient, with the ranks held fixed."""

    @staticmethod
    def forward(ctx, x, theta, y_sorted, p):
        lib = _lib.load()
        n, d = x.shape
        nproj, m = y_sorted.shape
        wpp = torch.empty(nproj, dtype=torch.float64, device=x.device)
        gcoef = torch.empty((nproj, n), dtype=torch.float32, device=x.device) if ctx.needs_input_grad[0] else None
        with torch.cuda.device(x.device):
            work, wbytes = _swd_workspace(lib, n, nproj, x.device)
            _lib.check(lib.mfb_swd_wpp(_ptr(x), n, d, _ptr(theta), nproj, _ptr(y_sorted), m, p, _ptr(wpp), _ptr(gcoef),
                                       _ptr(work), wbytes, _stream()), "swd_wpp")
        if gcoef is not None:
            ctx.save_for_backward(gcoef, theta)
        return wpp

    @staticmethod
    def backward(ctx, gwpp):
        gcoef, theta = ctx.saved_tensors
        nproj, n = gcoef.shape
        d = theta.shape[1]
        gw = gwpp.to(torch.float64).contiguous()
        gx = torch.empty((n, d), dtype=torch.float32, device=gcoef.device)
        lib = _lib.load()
        with torch.cuda.device(gcoef.device):
            _lib.check(lib.mfb_swd_bwd(_ptr(gcoef), n, d, _ptr(theta), nproj, _ptr(gw), _ptr(gx), _stream()),
                       "swd_bwd")
        return gx, None, None, None


def swd_wpp(x: torch.Tensor, theta: torch.Tensor, y_sorted: torch.Tensor, p: float) -> torch.Tensor:
    """W_p^p (the p-th power, as POT's ``wasserstein_1d``) between the projections of x on every direction (row of
    ``theta``, (P, d)) and the ascending reference projections ``y_sorted`` ((P, M), e.g. ``swd_sort(y, theta)[0]``),
    both sets uniformly weighted: (P,) float64.  Differentiable w.r.t. x only (ranks held fixed, the derivative of
    |0| is 0); the forward keeps a (P, N) float32 coefficient table for the backward when x requires grad."""
    check_swd_points("x", x)
    n, d = x.shape
    _swd_theta(theta, d)
    p = check_swd_p(p)
    if not isinstance(y_sorted, torch.Tensor) or y_sorted.dim() != 2 or y_sorted.shape[0] != theta.shape[0]:
        raise ValueError("y_sorted must be a (P, M) tensor, one sorted row per direction")
    if not 1 <= y_sorted.shape[1] < 2 ** 31:
        raise ValueError(f"y_sorted: M = {y_sorted.shape[1]} is outside [1, 2^31)")
    if y_sorted.requires_grad:
        raise ValueError("y_sorted requires grad, but the sliced Wasserstein kernels differentiate only x")
    x = _check_f32("x", x)                  # a contiguous copy, if one is made, stays on the autograd graph
    theta = _check_f32("theta", theta)
    y_sorted = _check_f32("y_sorted", y_sorted)
    return SWDWpp.apply(x, theta, y_sorted, p)


# --------------------------------------------------------------------------------------
# zuko-layout parameters <-> packed blocks
# --------------------------------------------------------------------------------------
# --------------------------------------------------------------------------------------
# tanh-MLP generator (generate/nn.py): fused forward, recomputing backward
# --------------------------------------------------------------------------------------
def nn_supported(din: int, dout: int, hidden_units: int, hidden_layers: int) -> bool:
    return bool(_lib.load().mfb_nn_supported(int(din), int(dout), int(hidden_units), int(hidden_layers)))


class NNForward(torch.autograd.Function):
    """x = MLP(z) from the six stacked parameter tensors; one library call each way."""

    @staticmethod
    def forward(ctx, z, w_in, b_in, w_hid, b_hid, w_out, b_out):
        lib = _lib.load()
        z = _check_f32("z", z.detach())
        params = [_check_f32(name, t.detach()) for name, t in
                  zip(("w_in", "b_in", "w_hid", "b_hid", "w_out", "b_out"), (w_in, b_in, w_hid, b_hid, w_out, b_out))]
        n, din = z.shape
        hidden, dout, layers = w_in.shape[0], w_out.shape[0], w_hid.shape[0] + 1
        x = torch.empty((n, dout), dtype=torch.float32, device=z.device)
        if n > 0:
            with torch.cuda.device(z.device):
                _lib.check(lib.mfb_nn_fwd(_ptr(z), n, din, dout, hidden, layers, *[_ptr(t) for t in params], _ptr(x),
                                          _stream()), "nn_fwd")
        ctx.save_for_backward(z, *params)
        ctx.dims = (din, dout, hidden, layers)
        return x

    @staticmethod
    def backward(ctx, gx):
        z, *params = ctx.saved_tensors
        din, dout, hidden, layers = ctx.dims
        n = z.shape[0]
        grads = [torch.zeros_like(t) for t in params]
        gz = torch.zeros_like(z) if ctx.needs_input_grad[0] else None
        if n > 0:
            gx = _check_f32("grad_x", gx)
            lib = _lib.load()
            with torch.cuda.device(z.device):
                wbytes = lib.mfb_nn_bwd_workspace_bytes(n, din, dout, hidden, layers)
                work = torch.empty(max(wbytes, 16), dtype=torch.uint8, device=z.device)
                _lib.check(lib.mfb_nn_bwd(_ptr(z), _ptr(gx), n, din, dout, hidden, layers, *[_ptr(t) for t in params],
                                          _ptr(gz), *[_ptr(g) for g in grads], _ptr(work), wbytes, _stream()), "nn_bwd")
        return (gz, *[g if need else None for g, need in zip(grads, ctx.needs_input_grad[1:])])


def nn_forward(z, w_in, b_in, w_hid, b_hid, w_out, b_out) -> torch.Tensor:
    """(N, Dout) particles of the tanh MLP for (N, Din) base noise z; differentiable w.r.t. z and the parameters."""
    if not isinstance(z, torch.Tensor) or z.dim() != 2 or z.shape[1] != w_in.shape[1]:
        raise ValueError(f"nn_forward: z must be a (N, {w_in.shape[1]}) tensor")
    _check_f32("z", z)
    return NNForward.apply(z, w_in, b_in, w_hid, b_hid, w_out, b_out)


class PackParameters(torch.autograd.Function):
    """(packed (T, floats_per_layer), packed_om (T, om_floats)) from the zuko-layout tensors of the whole flow in one
    launch; backward = one launch the other way (masked entries get exactly zero gradient).  ``packed_om`` is the
    same numbers in the backward kernels' out-major layout and carries no gradient of its own."""

    @staticmethod
    def forward(ctx, w_in, b_in, w_hid, b_hid, w_out, b_out, m_in, m_hid, m_out, dims):
        lib = _lib.load()
        T, d, hidden_units, hidden_layers, bins = dims
        ts = [_check_f32(n, t) for n, t in zip(("w_in", "b_in", "w_hid", "b_hid", "w_out", "b_out", "m_in", "m_hid", "m_out"),
                                                (w_in, b_in, w_hid, b_hid, w_out, b_out, m_in, m_hid, m_out))]
        dev = w_in.device
        with torch.cuda.device(dev):
            np_ = int(lib.mfb_nsf_layer_param_floats(d, hidden_units, hidden_layers, bins))
            nom = int(lib.mfb_nsf_layer_param_om_floats(d, hidden_units, hidden_layers))
            packed = torch.empty((T, np_), dtype=torch.float32, device=dev)
            packed_om = torch.empty((T, nom), dtype=torch.float32, device=dev)
            _lib.check(lib.mfb_nsf_pack_params(*[_ptr(t) if t.numel() else None for t in ts], T, d, hidden_units,
                                               hidden_layers, bins, _ptr(packed), _ptr(packed_om), _stream()),
                       "nsf_pack_params")
        ctx.save_for_backward(ts[6], ts[7], ts[8])
        ctx.dims = dims
        ctx.shapes = [t.shape for t in ts[:6]]
        ctx.mark_non_differentiable(packed_om)
        return packed, packed_om

    @staticmethod
    def backward(ctx, gpacked, _gom):
        lib = _lib.load()
        m_in, m_hid, m_out = ctx.saved_tensors
        T, d, hidden_units, hidden_layers, bins = ctx.dims
        gpacked = _check_f32("gpacked", gpacked)
        grads = [torch.empty(sh, dtype=torch.float32, device=gpacked.device) for sh in ctx.shapes]
        with torch.cuda.device(gpacked.device):
            _lib.check(lib.mfb_nsf_unpack_grads(_ptr(gpacked), _ptr(m_in), _ptr(m_hid) if m_hid.numel() else None,
                                                _ptr(m_out), T, d, hidden_units, hidden_layers, bins,
                                                *[_ptr(g) if g.numel() else None for g in grads], _stream()),
                       "nsf_unpack_grads")
        return (*grads, None, None, None, None)


# --------------------------------------------------------------------------------------
# whole flow (all layers), differentiable
# --------------------------------------------------------------------------------------
class NSFForward(torch.autograd.Function):
    """x, log q = flow(z): one kernel launch per autoregressive layer.  Only the layer inputs are
    kept (24 B / particle / layer); backward recomputes the conditioner activations instead of
    storing them (10.9 KB / particle in the reference's autograd graph)."""

    @staticmethod
    def forward(ctx, z, packed, packed_om, meta):
        orders, hidden_units, hidden_layers, bins, want_logq, images = meta
        z = _check_f32("z", z)
        packed = _check_f32("packed", packed)
        steps, logq = _nsf_run_layers(z, packed, orders, hidden_units, hidden_layers, bins, want_logq, images)
        ctx.meta = meta
        ctx.images = images        # the backward kernels read the same operand images (~1 MB, not rebuilt)
        ctx.save_for_backward(packed, packed_om, *steps[:-1])
        if logq is None:
            logq = z.new_empty(0)
        return steps[-1], logq

    @staticmethod
    def backward(ctx, gx, glogq):
        orders, hidden_units, hidden_layers, bins, want_logq, _ = ctx.meta
        images = ctx.images
        packed, packed_om, *inputs = ctx.saved_tensors
        n, d = inputs[0].shape
        gx = _check_f32("gx", gx) if gx is not None else torch.zeros_like(inputs[0])
        gl = _check_f32("glogq", glogq) if (want_logq and glogq is not None and glogq.numel() == n) else None
        gz, gpacked = nsf_backward(inputs, packed, packed_om, orders, hidden_units, hidden_layers, bins, gx, gl,
                                   images=images)
        return gz, gpacked, None, None


NSF_BWD_CHUNK = 1 << 20   # particles per backward pass: bounds the recompute workspace (~2.9 KB/particle)


def nsf_bwd_chunk(n: int) -> int:
    """Particles per backward pass for a batch of ``n``: NSF_BWD_CHUNK rounded down to a multiple of 128 (at least
    128), so that every chunk starts on a 16-byte aligned row for every D (the tcgen05 kernels bulk-copy their rows)."""
    return min(n, max(128, NSF_BWD_CHUNK // 128 * 128))


def nsf_backward(inputs, packed, packed_om, orders, hidden_units, hidden_layers, bins, gx, glogq, images=None):
    """(dL/dz, dL/dpacked) given the per-layer inputs saved by the forward pass.  ``images``: the tcgen05
    operand images of the same packed weights (``nsf_tc_images``), reused instead of being rebuilt."""
    lib = _lib.load()
    n, d = inputs[0].shape
    dev = inputs[0].device
    gpacked = torch.zeros_like(packed)
    gz = torch.empty_like(inputs[0])
    if n == 0:
        return gz, gpacked
    images = nsf_direction_images(NSF_BWD_USE_TENSOR_CORES, packed, orders, hidden_units, hidden_layers, bins, images)
    chunk = nsf_bwd_chunk(n)
    with torch.cuda.device(dev):
        wbytes = lib.mfb_nsf_layer_bwd_workspace_bytes(chunk, d, hidden_layers)
        work = torch.empty(wbytes, dtype=torch.uint8, device=dev)
        for start in range(0, n, chunk):
            m = min(chunk, n - start)
            g = gx[start:start + m]
            gl = None if glogq is None else glogq[start:start + m]
            for t in range(len(orders) - 1, -1, -1):
                order_arr = (ctypes.c_int32 * d)(*[int(o) for o in orders[t]])
                out = gz[start:start + m] if t == 0 else torch.empty((m, d), dtype=torch.float32, device=dev)
                _lib.check(lib.mfb_nsf_layer_bwd(_ptr(inputs[t][start:start + m]), _ptr(g), _ptr(gl), m, d,
                                                 hidden_units, hidden_layers, bins, _ptr(packed[t]), _ptr(packed_om[t]),
                                                 None if images is None else _ptr(images[t]),
                                                 ctypes.cast(order_arr, ctypes.c_void_p), 1 if t == 0 else 0,
                                                 _ptr(out), _ptr(gpacked[t]), 1 if start > 0 else 0, _ptr(work),
                                                 wbytes, _stream()), "nsf_layer_bwd")
                g = out
    return gz, gpacked


def nsf_forward(z, packed, packed_om, orders, hidden_units, hidden_layers, bins, want_logq=True, want_steps=False,
                images=None):
    """Returns (x, logq or None, steps or None)."""
    images = nsf_direction_images(NSF_USE_TENSOR_CORES, packed.detach(), orders, hidden_units, hidden_layers, bins,
                                  images)
    if want_steps or not (torch.is_grad_enabled() and (z.requires_grad or packed.requires_grad)):
        # nothing to differentiate: skip the autograd.Function bookkeeping
        z = _check_f32("z", z.detach())
        steps, logq = _nsf_run_layers(z, _check_f32("packed", packed.detach()), orders, hidden_units, hidden_layers,
                                      bins, want_logq, images)
        return steps[-1], logq, (steps if want_steps else None)
    meta = (tuple(tuple(o) for o in orders), hidden_units, hidden_layers, bins, bool(want_logq), images)
    x, logq = NSFForward.apply(z, packed, packed_om, meta)
    return x, (logq if want_logq else None), None


NSF_INV_USE_TENSOR_CORES = True   # tcgen05 inverse where the forward's operand images exist; False = fp32 CUDA-core kernel


def nsf_inverse(x, packed, orders, hidden_units, hidden_layers, bins, want_logq=True, want_steps=False, images=None):
    """Density direction: returns (z, log q(x) or None, steps or None).  Not differentiable (no
    experiment of the reference trains through log_prob(x); SURVEY.md 3.5).  ``images``: the forward kernel's operand
    images (``nsf_tc_images``): with them each layer is one tensor-core launch (S x 4 GEMM round trips per tile)
    instead of D full sweeps of the CUDA-core kernel."""
    lib = _lib.load()
    x = _check_f32("x", x.detach())
    packed = _check_f32("packed", packed.detach())
    n, d = x.shape
    if images is not None:     # the inverse runs from the forward's images only: it builds none of its own
        images = nsf_direction_images(NSF_INV_USE_TENSOR_CORES, packed, orders, hidden_units, hidden_layers, bins,
                                      images)
    steps = [x]
    acc = None
    with torch.cuda.device(x.device):
        for t in range(len(orders) - 1, -1, -1):
            v = torch.empty_like(x)
            out = torch.empty(n, dtype=torch.float32, device=x.device) if want_logq else None
            order_arr = (ctypes.c_int32 * d)(*[int(o) for o in orders[t]])
            if n == 0:          # empty batch: nothing to launch
                acc = out
                steps.append(v)
                continue
            _lib.check(lib.mfb_nsf_layer_inv(_ptr(steps[-1]), n, d, hidden_units, hidden_layers, bins, _ptr(packed[t]),
                                             None if images is None else _ptr(images[t]),
                                             ctypes.cast(order_arr, ctypes.c_void_p), _ptr(acc), 1 if t == 0 else 0,
                                             _ptr(v), _ptr(out), _stream()), "nsf_layer_inv")
            acc = out
            steps.append(v)
    return steps[-1], acc, (steps if want_steps else None)


# --------------------------------------------------------------------------------------
# classical MENT
# --------------------------------------------------------------------------------------
def _host_i32(values):
    arr = (ctypes.c_int32 * len(values))(*[int(v) for v in values])
    return arr, ctypes.cast(arr, ctypes.c_void_p)


def _host_f32(values):
    arr = (ctypes.c_float * len(values))(*[float(v) for v in values])
    return arr, ctypes.cast(arr, ctypes.c_void_p)


def _ment_tables(g1, g2, d: int, device, kick: bool = False):
    """C-ABI arguments of the two table families in ABI order (proj, coords, tables, k, b, mp, proj2, cx, cy, tables2,
    k2, bx, by, mp2), the tensors they point into, and whether the model has kicks.
    g1 = (proj (K,D), coords (K,B), tables (K,B)[, mp (K,2D+4)]) or None,
    g2 = (proj2 (K2,2,D), cx (K2,Bx), cy (K2,By), tables2 (K2,Bx,By)[, mp2 (K2,2,2D+4)]) or None.
    The optional multipole rows have the layout of ``simulate.multipole_terms``, order 0 for the rows of linear maps.
    The model has kicks when either family carries rows or ``kick`` is set; then a family without rows gets order-0
    rows.  A linear model passes NULL for both."""
    keep = []
    if g1 is not None:
        proj, coords, tables = (_check_f32(n, t) for n, t in zip(("proj", "coords", "tables"), g1))
        keep += [proj, coords, tables]
        a1 = [_ptr(proj), _ptr(coords), _ptr(tables), tables.shape[0], tables.shape[1]]
    else:
        a1 = [None, None, None, 0, 2]
    if g2 is not None:
        proj2, cx, cy, tab2 = (_check_f32(n, t) for n, t in zip(("proj2", "cx", "cy", "tables2"), g2))
        if proj2.ndim != 3 or proj2.shape[1] != 2 or tab2.shape != (proj2.shape[0], cx.shape[1], cy.shape[1]):
            raise ValueError("2-D Lagrange tables: proj2 (K,2,D), cx (K,Bx), cy (K,By), tables2 (K,Bx,By) expected")
        keep += [proj2, cx, cy, tab2]
        a2 = [_ptr(proj2), _ptr(cx), _ptr(cy), _ptr(tab2), tab2.shape[0], tab2.shape[1], tab2.shape[2]]
    else:
        a2 = [None, None, None, None, 0, 0, 0]
    mp1 = g1[3] if g1 is not None and len(g1) > 3 else None
    mp2 = g2[4] if g2 is not None and len(g2) > 4 else None
    kick = kick or mp1 is not None or mp2 is not None
    rows = []
    stride = 2 * d + 4
    for mp, grp, lead, name in ((mp1, g1, (), "mp"), (mp2, g2, (2,), "mp2")):
        if not kick or grp is None:
            rows.append(None)
            continue
        k = int(grp[0].shape[0])
        if mp is None:
            mp = torch.zeros((k,) + lead + (stride,), dtype=torch.float32, device=device)
        mp = _check_f32(name, mp)
        if tuple(mp.shape) != (k,) + lead + (stride,):
            raise ValueError(f"MENT multipole rows {name} must have shape {(k,) + lead + (stride,)}, "
                             f"got {tuple(mp.shape)}")
        keep.append(mp)
        rows.append(_ptr(mp))
    return a1 + [rows[0]] + a2 + [rows[1]], keep, kick


def ment_prob(x, g1, g2, neg_half_inv_s2: float, log_norm: float) -> torch.Tensor:
    """rho at explicit points x (G, D) with one- and two-dimensional Lagrange tables and, when g1 / g2 carry
    multipole rows, the kicks (see ``_ment_tables``)."""
    lib = _lib.load()
    x = _check_f32("x", x)
    g, d = x.shape
    args, keep, _ = _ment_tables(g1, g2, d, x.device)
    out = torch.empty(g, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.mfb_ment_prob(_ptr(x), g, d, *args, float(neg_half_inv_s2), float(log_norm), _ptr(out),
                                     _stream()), "ment_prob")
    return out


def ment_prob_grid(shape, first_centre, step, g1, g2, neg_half_inv_s2, log_norm, device) -> torch.Tensor:
    """rho on the centres of a regular grid (flattened, 'ij' order) without materialising the points."""
    lib = _lib.load()
    d = len(shape)
    g = 1
    for s_ in shape:
        g *= int(s_)
    args, keep, _ = _ment_tables(g1, g2, d, device)
    out = torch.empty(g, dtype=torch.float32, device=device)
    h1, p1 = _host_i32(shape)
    h2, p2 = _host_f32(first_centre)
    h3, p3 = _host_f32(step)
    with torch.cuda.device(device):
        _lib.check(lib.mfb_ment_prob_grid(d, p1, p2, p3, *args, float(neg_half_inv_s2), float(log_norm), _ptr(out),
                                          _stream()), "ment_prob_grid")
    return out


def ment_integrate(d, meas_coords, meas_axis, meas_coords2, meas_axis2, int_shape, int_first, int_step, minv, g1, g2,
                   neg_half_inv_s2, log_norm, inv_mp: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Integration-mode prediction of one screen: 1-D (meas_axis2 = -1) -> (B,), 2-D -> (Bx, By).  The screen is mapped
    back with ``minv``; with ``inv_mp`` (4D+2,) = [r0 | r2 | p | q | order | 0] (``simulate.multipole_inverse_terms``)
    the map back is ``minv u + p Re(z^m) + q Im(z^m)``, z = r0 . u + i r2 . u.  Multipole rows in g1 / g2 or an
    ``inv_mp`` select the kernel with multipole terms."""
    lib = _lib.load()
    meas_coords, minv = _check_f32("meas_coords", meas_coords), _check_f32("minv", minv)
    if tuple(minv.shape) != (d, d):
        raise ValueError(f"minv must have shape ({d}, {d}), got {tuple(minv.shape)}")
    nb = meas_coords.shape[0]
    nb2 = 0
    if meas_axis2 >= 0:
        meas_coords2 = _check_f32("meas_coords2", meas_coords2)
        nb2 = meas_coords2.shape[0]
    args, keep, kick = _ment_tables(g1, g2, d, minv.device, kick=inv_mp is not None)
    if kick:
        if inv_mp is None:
            inv_mp = torch.zeros(4 * d + 2, dtype=torch.float32, device=minv.device)
        inv_mp = _check_f32("inv_mp", inv_mp)
        if tuple(inv_mp.shape) != (4 * d + 2,):
            raise ValueError(f"inv_mp must have shape ({4 * d + 2},), got {tuple(inv_mp.shape)}")
    pred = torch.empty((nb, nb2) if meas_axis2 >= 0 else (nb,), dtype=torch.float32, device=minv.device)
    h1, p1 = _host_i32(int_shape)
    h2, p2 = _host_f32(int_first)
    h3, p3 = _host_f32(int_step)
    mc2 = _ptr(meas_coords2) if meas_axis2 >= 0 else None
    with torch.cuda.device(minv.device):
        _lib.check(lib.mfb_ment_integrate(d, _ptr(meas_coords), nb, int(meas_axis), mc2, nb2, int(meas_axis2),
                                          len(int_shape), p1, p2, p3, _ptr(minv), _ptr(inv_mp), *args,
                                          float(neg_half_inv_s2), float(log_norm), _ptr(pred), _stream()),
                   "ment_integrate")
    return pred


def cdf_sample(rho: torch.Tensor, shape, first_edge, cell, size: int, seed: int, offset: int = 0,
               jitter: bool = False, pad: float = 1.0e-15) -> torch.Tensor:
    """`size` particles from the piecewise-constant density rho (flattened grid, 'ij' order)."""
    lib = _lib.load()
    rho = _check_f32("rho", rho.reshape(-1))
    g = rho.numel()
    d = len(shape)
    cdf = torch.empty(g, dtype=torch.float64, device=rho.device)
    out = torch.empty((int(size), d), dtype=torch.float32, device=rho.device)
    a1, p1 = _host_i32(shape)
    a2, p2 = _host_f32(first_edge)
    a3, p3 = _host_f32(cell)
    with torch.cuda.device(rho.device):
        wbytes = lib.mfb_cdf_workspace_bytes(g)
        work = torch.empty(wbytes, dtype=torch.uint8, device=rho.device)
        _lib.check(lib.mfb_cdf_build(_ptr(rho), g, float(pad), _ptr(cdf), _ptr(work), wbytes, _stream()), "cdf_build")
        _lib.check(lib.mfb_cdf_sample(_ptr(cdf), g, _ptr(work), d, p1, p2, p3, 1 if jitter else 0,
                                      int(seed) & (2 ** 64 - 1), int(offset), int(size), _ptr(out), _stream()),
                   "cdf_sample")
    return out


def gs_update(table: torch.Tensor, meas: torch.Tensor, pred: torch.Tensor, lr: float, thresh: float) -> None:
    """In-place Gauss-Seidel update of one Lagrange table."""
    lib = _lib.load()
    n = table.numel()
    meas, pred = _check_f32("meas", meas), _check_f32("pred", pred)
    if not (table.is_cuda and table.is_contiguous() and table.dtype == torch.float32):
        raise RuntimeError("gs_update: table must be a contiguous CUDA float32 tensor (no CPU fallback)")
    with torch.cuda.device(table.device):
        _lib.check(lib.mfb_gs_update(_ptr(table), _ptr(meas), _ptr(pred), n, float(lr), float(thresh), _stream()),
                   "gs_update")


# --------------------------------------------------------------------------------------
# base noise on the device (generate/flows/zuko.py:15-16 -> torch.randn)
# --------------------------------------------------------------------------------------
class PhiloxStream:
    """torch's CUDA generator, mirrored for the library's randn kernel.

    ``normal_(out)`` fills ``out`` with exactly the values ``torch.randn(out.shape, device=...)`` would
    produce for the generator's current (seed, offset) and moves the generator on by the same amount, so
    library draws and torch draws interleave as if all of them were torch's.  While a CUDA graph is being
    captured the (seed, offset) pair is read from a device tensor instead, and the kernel advances it
    itself; ``sync()`` before a replay re-primes that tensor if the generator was re-seeded or used by
    somebody else in the meantime, ``consumed()`` after it books the replay's draws on the generator.
    """

    def __init__(self, device) -> None:
        self.device = torch.device(device)
        self.state: Optional[torch.Tensor] = None   # int64[2] on the device: seed, offset
        self._mirror = None                          # (seed, offset) the device tensor holds
        self._pinned = None
        self.captured_increment = 0                  # offset consumed by one replay of the captured draws

    def _generator(self):
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        return torch.cuda.default_generators[idx]

    @staticmethod
    def _as_i64(v: int) -> int:
        v &= (1 << 64) - 1
        return v - (1 << 64) if v >= (1 << 63) else v

    def normal_(self, out: torch.Tensor) -> torch.Tensor:
        lib = _lib.load()
        if not out.is_cuda or out.dtype != torch.float32 or not out.is_contiguous():
            raise RuntimeError("PhiloxStream.normal_: contiguous float32 CUDA tensor expected; there is no CPU fallback")
        numel = out.numel()
        if numel == 0:
            return out
        with torch.cuda.device(out.device):
            inc = int(lib.mfb_randn_offset_increment(numel))
            if torch.cuda.is_current_stream_capturing():
                if self.state is None:
                    raise RuntimeError("PhiloxStream: call begin_capture() before capturing a draw")
                _lib.check(lib.mfb_randn_philox_state(_ptr(out), numel, _ptr(self.state), 1, _stream()), "randn_philox_state")
                self.captured_increment += inc
            else:
                g = self._generator()
                seed, off = int(g.initial_seed()), int(g.get_offset())
                _lib.check(lib.mfb_randn_philox(_ptr(out), numel, ctypes.c_uint64(seed & ((1 << 64) - 1)),
                                                ctypes.c_uint64(off), _stream()), "randn_philox")
                g.set_offset(off + inc)
        return out

    def mark(self) -> int:
        """current offset of torch's generator (see ``rewind``)"""
        return int(self._generator().get_offset())

    def rewind(self, mark: int) -> None:
        """put torch's generator back to a marked offset (warm-up passes of a capture must not consume
        the caller's random stream)"""
        self._generator().set_offset(int(mark))

    # ---- graph replay support ---------------------------------------------------------------
    def begin_capture(self) -> None:
        """Allocate / prime the device state; call right before the graph capture starts."""
        if self.state is None:
            self.state = torch.zeros(2, dtype=torch.int64, device=self.device)
            # ring of pinned staging slots, each guarded by an event: a slot is rewritten by the host only after
            # the asynchronous copy that last read it has completed (re-seeding every step without synchronising
            # in between must not let a later state overtake an earlier replay)
            self._pinned = torch.zeros((8, 2), dtype=torch.int64).pin_memory()
            self._pinned_np = self._pinned.numpy()       # the same memory: element writes without a dispatcher trip
            self._slot_events = [None] * 8
            self._slot = 0
        self.captured_increment = 0
        self._mirror = None
        self.sync()

    def sync(self) -> None:
        """Make the device state equal to torch's generator (no-op in steady state)."""
        g = self._generator()
        cur = (int(g.initial_seed()), int(g.get_offset()))
        if self._mirror != cur:
            i = self._slot
            self._slot = (i + 1) % self._pinned.shape[0]
            ev = self._slot_events[i]
            if ev is not None:
                ev.synchronize()
            else:
                ev = self._slot_events[i] = torch.cuda.Event()
            self._pinned_np[i, 0] = self._as_i64(cur[0])
            self._pinned_np[i, 1] = self._as_i64(cur[1])
            self.state.copy_(self._pinned[i], non_blocking=True)
            ev.record()
            self._mirror = cur

    def consumed(self) -> None:
        """Book one replay of the captured draws on torch's generator."""
        if self.captured_increment:
            g = self._generator()
            off = int(g.get_offset()) + self.captured_increment
            g.set_offset(off)
            self._mirror = (self._mirror[0], off)
