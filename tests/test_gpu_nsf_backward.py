"""GPU: both backward implementations of the flow -- the tcgen05 kernels (nsf_tc.cu kBwd, then the dgrad and wgrad
kernels of nsf_tc_bwd.cu; the default) and the fp32 CUDA-core kernels (nsf_bwd.cu) -- at every compiled dimension
against float64 autograd of the oracle.

Metric (as test_gpu_nsf.py's test_backward_matches_oracle_autograd): the error of each gradient tensor relative to
its largest entry.  The flow is only piecewise smooth: d(log q)/dz jumps across spline knots and ReLU kinks, and a
particle within an fp32 ulp of such a boundary takes the other branch than the float64 oracle.  Pass 1 finds those
particles from their dL/dz (at most 2 + n / 100 of them); pass 2 repeats the comparison without them and requires
every gradient tensor to agree: max below 1e-3, median below 2e-5.

A ReLU kink hides from dL/dz: across it the conditioner's output is continuous, so dL/dz barely moves, while the
particle's whole upstream gradient of that unit moves in or out of the unit's bias and weight gradients.  Measured:
at D = 2, n = 3201 one particle has a float64 pre-activation of -1.5e-7 (2.6e-7 of the magnitude of its terms); both
backward paths put it on the active side, and b_hid3.0 then differs from float64 by exactly that particle's
gradient, 1.08e-3 of the largest entry, on both paths alike (torch-fp32 autograd, on the inactive side: 6e-6).
Pass 1 therefore also excludes the particles the float64 oracle itself places within 1e-6 of a kink
(nsf_relu_kink_particles): a property of the inputs, not of the kernels, so they are not counted against the bound
(12 of 3201 particles at D = 2, 29 of 60 001 at D = 6).

Beyond the float64 comparison: chunked batches (every partial sum accumulated into the previous chunk's), one-sided
losses (no dL/dlog q; dL/dx = 0), upstream gradients scaled by powers of two (exact on both paths) or spread over six
decades (the per-row and per-batch operand scaling of the tcgen05 kernels), run-to-run determinism and the empty
batch."""
import pytest
import torch

from mentflow_b200 import _lib, ops
from mfb_testutil import (grad_rel, nsf_case, nsf_kernel_grads, nsf_named_grads, nsf_oracle_grads,
                          nsf_relu_kink_particles, oracle_from_generator)

pytestmark = pytest.mark.gpu
DIMS = [2, 3, 4, 5, 6]
PARAMS = ("w_in", "b_in", "w_hid", "b_hid", "w_out", "b_out")


@pytest.fixture(params=["tcgen05", "cuda_core"])
def bwd_path(request, monkeypatch):
    """Run a test once per backward implementation (ops.NSF_BWD_USE_TENSOR_CORES)."""
    monkeypatch.setattr(ops, "NSF_BWD_USE_TENSOR_CORES", request.param == "tcgen05")
    return request.param


def _case(path, d, n, scale=1.0, hidden_layers=3, transforms=5, bins=20, seed=0):
    """``nsf_case`` with the flow on the GPU; a tcgen05 case first makes sure its kernels are compiled for the shape,
    so that it cannot quietly run on the CUDA-core kernels instead."""
    if path == "tcgen05":
        assert (hidden_layers, bins) == (3, 20) and ops.nsf_tc_supported(d, 64, 3, 20)
    gen, ref, z, a, b = nsf_case(d, n, scale, hidden_layers, transforms, bins, seed)
    return gen.to("cuda"), ref, z, a, b


def _check_vs_oracle(gen, ref, z, a, b, loss="both", per_particle=False, param_tol=None):
    """The two-pass float64 comparison of the module docstring; masked weights must get exactly zero gradient.

    per_particle: dL/dz of each particle relative to that particle's own largest entry instead of the tensor's.
    param_tol: None for the fixed bounds on the parameter gradients, or a factor f: worst entry of each parameter
    gradient at most max(1e-3, f x the oracle's torch-fp32 autograd's worst entry) on the same particles."""
    hl, tr = gen.hidden_layers, gen.transforms
    n = z.shape[0]

    def z_err(got, want):
        if not per_particle:
            return grad_rel(got, want)
        want = want.double().cpu()
        return (got.double().cpu() - want).abs() / want.abs().max(dim=1, keepdim=True).values.clamp_min(1e-30)

    got = nsf_named_grads(nsf_kernel_grads(gen, z, a, b, loss), hl, tr)
    want, masks = nsf_oracle_grads(ref, z, a, b, loss)
    suspects = z_err(got["z"], want["z"]).max(dim=1).values > 1e-4
    assert int(suspects.sum()) <= 2 + n // 100, f"{int(suspects.sum())} of {n} particles disagree in dL/dz"
    suspects |= nsf_relu_kink_particles(ref, z)
    if bool(suspects.any()):
        keep = ~suspects
        assert bool(keep.any())
        z, a, b = z[keep], a[keep], b[keep]
        got = nsf_named_grads(nsf_kernel_grads(gen, z, a, b, loss), hl, tr)
        want, masks = nsf_oracle_grads(ref, z, a, b, loss)
    want32, _ = nsf_oracle_grads(oracle_from_generator(gen, torch.float32), z, a, b, loss)
    for name, w in want.items():
        g = got[name]
        assert g.shape == w.shape and bool(torch.isfinite(g).all()), name
        if name in masks:               # masked weights: exactly zero gradient
            assert bool((g.cpu()[~masks[name]] == 0).all()), name
        e = (z_err if name == "z" else grad_rel)(g, w).flatten()
        e32 = float(grad_rel(want32[name], w).max())
        msg = f"{name}: max {float(e.max()):.2e}, median {float(e.median()):.2e} (torch-fp32 autograd: max {e32:.2e})"
        if name != "z" and param_tol is not None:
            assert float(e.max()) <= max(1e-3, param_tol * e32), msg
        else:
            assert float(e.max()) < 1e-3 and float(e.median()) < 2e-5, msg


# ---------------------------------------------------------------------------------- A. every dimension, both paths
@pytest.mark.parametrize("scale", [1.0, 1.5])
@pytest.mark.parametrize("n", [1, 129, 4097])
@pytest.mark.parametrize("d", DIMS)
def test_every_dimension(d, n, scale, bwd_path):
    """Each D has its own slot arithmetic in the masked conditioner; n = 1 (a single row in a single tile), 129 (a
    second tile holding one row), 4097 (33 tiles, the last with one row)."""
    _check_vs_oracle(*_case(bwd_path, d, n, scale, seed=10 * d + n % 7 + int(4 * scale)))


@pytest.mark.parametrize("d", DIMS)
def test_persistent_multi_tile_loop(d, monkeypatch):
    """More 128-particle tiles than warpgroups on the device (148 SMs x 3 = 444 on a B200): every warpgroup of the
    spline-backward, dgrad and wgrad kernels runs its persistent loop over more than one tile."""
    monkeypatch.setattr(ops, "NSF_BWD_USE_TENSOR_CORES", True)
    n = 60_001
    assert n > _lib.load().mfb_sm_count() * 3 * 128
    _check_vs_oracle(*_case("tcgen05", d, n, 1.0, transforms=2, seed=600 + d))


def test_cuda_core_parameter_block_edge(monkeypatch):
    """bins = 21 fills the CUDA-core kernels' per-feature parameter block (3 x 21 - 1 = 62 of kPP = 64 rows), with two
    hidden layers (a shape the tcgen05 kernels are not compiled for)."""
    monkeypatch.setattr(ops, "NSF_BWD_USE_TENSOR_CORES", False)
    _check_vs_oracle(*_case("cuda_core", 5, 2049, 1.0, hidden_layers=2, bins=21, seed=521))


# ---------------------------------------------------------------------------------- B. chunked accumulation
@pytest.mark.parametrize("d", DIMS)
def test_chunked_backward_matches_one_pass(d, bwd_path, monkeypatch):
    """Backward in chunks of 1024 particles (n = 3 x 1024 + 129: the last chunk has two tiles, the second holding one
    row), every later chunk accumulating into the parameter gradients of the ones before.  dL/dz is bit-identical to
    the single pass (each particle's rows are scaled by their own maximum, wherever the particle sits); the parameter
    gradients differ by the order of summation only; and the chunked result passes the float64 comparison."""
    n = 3 * 1024 + 129
    gen, ref, z, a, b = _case(bwd_path, d, n, 1.0, seed=300 + d)
    assert ops.nsf_bwd_chunk(n) == n
    one = nsf_kernel_grads(gen, z, a, b)
    one = {k: v.clone() for k, v in one.items()}
    monkeypatch.setattr(ops, "NSF_BWD_CHUNK", 1024)
    assert ops.nsf_bwd_chunk(n) == 1024
    chunked = nsf_kernel_grads(gen, z, a, b)
    assert torch.equal(chunked["z"], one["z"])
    for name in PARAMS:
        e = float(grad_rel(chunked[name], one[name]).max())
        assert e <= 1e-6, f"{name}: {e:.2e} of the largest entry"
    _check_vs_oracle(gen, ref, z, a, b)


# ---------------------------------------------------------------------------------- C. one-sided losses
@pytest.mark.parametrize("loss", ["x", "logq"])
@pytest.mark.parametrize("bwd_path,d", [("tcgen05", d) for d in DIMS] + [("cuda_core", 2), ("cuda_core", 6)],
                         indirect=["bwd_path"])
def test_one_sided_loss(d, loss, bwd_path):
    """x only (gen.forward: no log q is computed, the spline backward kernels get no dL/dlog q) and log q only
    (dL/dx arrives as zeros)."""
    _check_vs_oracle(*_case(bwd_path, d, 4097, 1.5, seed=400 + d), loss=loss)


# ---------------------------------------------------------------------------------- D. gradient scale
@pytest.mark.parametrize("d", DIMS)
def test_power_of_two_upstream_scale_is_exact(d, bwd_path):
    """Upstream gradients x 2^-60 and x 2^40: every gradient is the unscaled one x 2^k bit for bit.  Both factors keep
    every fp32 intermediate normal, and the tcgen05 kernels' operand scales are powers of two derived from the
    operands' maxima, so a scale derived wrongly (or one that is not a power of two) shows here.  All-zero upstream
    gradients give exactly zero (and finite) gradients: the scale of a zero maximum."""
    gen, _, z, a, b = _case(bwd_path, d, 4097, 1.5, seed=700 + d)
    base = {k: v.clone() for k, v in nsf_kernel_grads(gen, z, a, b).items()}
    assert all(float(v.abs().max()) > 0 for v in base.values())
    for k in (-60, 40):
        f = 2.0 ** k
        got = nsf_kernel_grads(gen, z, a * f, b * f)
        for name, v in got.items():
            assert torch.equal(v.double(), base[name].double() * f), f"{name}, 2^{k}"
    got = nsf_kernel_grads(gen, z, torch.zeros_like(a), torch.zeros_like(b))
    for name, v in got.items():
        assert bool(torch.isfinite(v).all()) and bool((v == 0).all()), name


@pytest.mark.parametrize("d", DIMS)
def test_heavy_tailed_upstream(d, bwd_path):
    """Per-particle upstream magnitudes 10^U(-6, 0).  dL/dz of each particle against float64 relative to that
    particle's own largest entry (the tcgen05 dgrad scales every row by its own maximum); the parameter gradients,
    sums dominated by the largest particles, within max(1e-3, 3 x torch-fp32 autograd's error) of their largest entry
    (the tcgen05 wgrad scales per batch)."""
    gen, ref, z, a, b = _case(bwd_path, d, 4097, 1.0, seed=800 + d)
    g = torch.Generator().manual_seed(800 + d)
    m = 10.0 ** (-6.0 * torch.rand(z.shape[0], generator=g))
    _check_vs_oracle(gen, ref, z, a * m[:, None], b * m, per_particle=True, param_tol=3.0)


# ---------------------------------------------------------------------------------- E. determinism, empty batch
@pytest.mark.parametrize("d,n,transforms", [(6, 60_001, 2), (3, 4097, 5)])
def test_backward_is_deterministic(d, n, transforms, bwd_path):
    """Two backward passes on the same inputs: bitwise-equal gradients (fixed reduction orders, no atomics in a sum)."""
    gen, _, z, a, b = _case(bwd_path, d, n, 1.0, transforms=transforms, seed=900 + d)
    first = {k: v.clone() for k, v in nsf_kernel_grads(gen, z, a, b).items()}
    second = nsf_kernel_grads(gen, z, a, b)
    for name, v in second.items():
        assert torch.equal(v, first[name]), name


@pytest.mark.parametrize("d", [3, 6])
def test_empty_batch(d, bwd_path):
    """n = 0: an empty dL/dz and zero parameter gradients."""
    gen, _, z, a, b = _case(bwd_path, d, 0, 1.0, seed=1000 + d)
    got = nsf_kernel_grads(gen, z, a, b)
    assert got["z"].shape == (0, d)
    for name in PARAMS:
        assert got[name].shape == getattr(gen, name).shape and bool((got[name] == 0).all()), name
