"""CPU tests of the host layer: C-ABI library loads and exports what include/*.h declares,
mask construction / parameter packing agree with the oracle, API objects behave like the
reference's, and compute entry points refuse CPU tensors (no fallback)."""
import os
import re

import numpy as np
import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200 import _lib, ops
from mfb_testutil import generator_from_golden, oracle_from_generator, t32
from oracle.zuko_nsf import layer_order, masked_mlp_masks

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol_at_the_header_abi_version():
    header = open(os.path.join(ROOT, "include", "mentflow_b200.h")).read()
    declared = set(re.findall(r"\b(mfb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.SIGNATURES), "ctypes table and header disagree"
    version = int(re.search(r"#define MFB_ABI_VERSION (\d+)", header).group(1))
    assert lib.mfb_abi_version() == version == _lib.ABI_VERSION == 5
    assert b"workspace" in lib.mfb_error_string(-3)


@pytest.mark.parametrize("d", [2, 3, 4, 6])
def test_closed_form_masks_equal_zuko_construction(d):
    for layer in (0, 1):
        mine = mf.generate.conditioner_masks(mf.generate.layer_order(d, layer), 59, 64, 3)
        ref = masked_mlp_masks(layer_order(d, layer), 59, [64] * 3)
        assert len(mine) == len(ref)
        for a, b in zip(mine, ref):
            assert torch.equal(a.bool(), b.bool())


@pytest.mark.parametrize("d,passes", [(6, 2), (4, 2), (5, 2), (6, 3), (3, 2)])
def test_coupling_masks_equal_zuko_construction(d, passes):
    """zuko's `passes` option (coupling layers for passes = 2): orders repeat, every hidden unit of a coupling
    layer has the single reachable class, the first half of the features gets bias-only splines."""
    for layer in (0, 1):
        order = mf.generate.layer_order(d, layer, passes)
        assert order == layer_order(d, layer, passes).tolist()
        mine = mf.generate.conditioner_masks(order, 59, 64, 3)
        ref = masked_mlp_masks(layer_order(d, layer, passes), 59, [64] * 3)
        for a, b in zip(mine, ref):
            assert torch.equal(a.bool(), b.bool())
    gen = mf.generate.build_generator("nsf", input_features=d, output_features=d, hidden_layers=3, hidden_units=64,
                                      transforms=4, bins=20, passes=passes)
    assert gen.passes == passes and not ops.orders_autoregressive(gen._orders)
    assert not ops.nsf_tc_supported(d, 64, 3, 20, gen._orders)        # coupling layers run on the CUDA-core kernels
    sd = gen.state_dict()
    sd2 = {k.replace("_flow.transform.transforms.", "_flow.transform.transform.transforms."): v for k, v in sd.items()}
    other = mf.generate.NSFGenerator(d, transforms=4, passes=passes)
    other.load_state_dict(sd2)                                          # both zuko key spellings load
    assert torch.equal(other.w_out, gen.w_out)


def test_generator_matches_oracle_initialisation_and_names():
    torch.manual_seed(7)
    gen = mf.generate.build_generator("nsf", input_features=6, output_features=6, hidden_layers=3,
                                      hidden_units=64, transforms=5, bins=20)
    from oracle.zuko_nsf import NSFOracle
    torch.manual_seed(7)
    ref = NSFOracle(6)
    cp = oracle_from_generator(gen, torch.float32)
    for (ka, a), (kb, b) in zip(ref.state_dict().items(), cp.state_dict().items()):
        assert ka == kb and torch.equal(a, b), ka
    assert sum(p.numel() for p in gen.parameters()) == 158890
    sd = gen.state_dict()
    gen2 = mf.generate.NSFGenerator(6)
    gen2.load_state_dict(sd)
    assert torch.equal(gen2.w_out, gen.w_out) and torch.equal(gen2.b_hid, gen.b_hid)


def _emulate_packed_layer(packed, v, d, hidden_layers, bins):
    """What the CUDA kernel computes from one layer's packed block, in torch (float64)."""
    H, PP = 64, 64
    o = 0
    w1 = packed[o:o + d * H].reshape(d, H); o += d * H
    b1 = packed[o:o + H]; o += H
    h = torch.relu(v @ w1 + b1)
    for _ in range(hidden_layers - 1):
        w = packed[o:o + H * H].reshape(H, H); o += H * H
        b = packed[o:o + H]; o += H
        h = torch.relu(h @ w + b)
    wo = packed[o:o + d * H * PP].reshape(d, H, PP); o += d * H * PP
    bo = packed[o:o + d * PP].reshape(d, PP); o += d * PP
    assert o == packed.numel()
    phi = torch.einsum("nh,dhp->ndp", h, wo) + bo
    return phi[:, :, :3 * bins - 1]


def test_packed_layout_reproduces_conditioner(golden):
    g = golden("nsf_6d")
    gen = generator_from_golden(g)
    ref = oracle_from_generator(gen)
    packed = gen.packed_parameters().double()
    assert packed.shape[1] == ops.nsf_layer_param_floats(6, 64, 3, 20)
    v = torch.from_numpy(g["z"])
    for t, layer in enumerate(ref.layers):
        phi = _emulate_packed_layer(packed[t], v, 6, 3, 20)
        want = layer.hyper(v).unflatten(-1, (6, 59))
        assert torch.allclose(phi, want, atol=1e-12)


def test_packing_is_differentiable_and_masked():
    gen = mf.generate.NSFGenerator(4, transforms=2)
    packed = gen.packed_parameters()
    packed.sum().backward()
    assert gen.w_in.grad is not None
    # masked-out weights get zero gradient
    assert torch.equal(gen.w_in.grad != 0, gen.m_in.bool())
    assert torch.equal(gen.w_out.grad != 0, gen.m_out.bool())


def test_diagnostic_interface_and_no_cpu_fallback():
    e = torch.linspace(-3.5, 3.5, 65)
    d = mf.diagnostics.Histogram1D(axis=0, edges=e, bandwidth=0.5, noise=True, noise_scale=0.0, seed=1)
    assert d.ndim == 1 and d.kde and d.edges.shape == (65,) and d.coords.shape == (64,)
    assert abs(float(d.bandwidth) - 0.5 * float(e[1] - e[0])) < 1e-9
    c0, spacing, sigma, delta = d.geometry()
    assert abs(c0 - float(d.coords[0])) < 1e-7 and delta == float(d.coords[1] - d.coords[0])
    assert abs(spacing - 7.0 / 64) < 1e-9 and abs(spacing - delta) < 1e-5 * delta
    x = torch.randn(10, 6)
    assert torch.equal(d.project(x), x[:, 0])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        d(x)
    d2 = mf.diagnostics.Histogram2D(axis=(0, 2), edges=[e, e], bandwidth=(0.5, 0.5))
    assert d2.ndim == 2 and d2.shape == (64, 64) and len(d2.edges) == 2
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        d2(x)
    with pytest.raises(NotImplementedError):
        mf.diagnostics.Histogram1D(edges=torch.tensor([0.0, 1.0, 3.0, 7.0])).geometry()
    gen = mf.generate.NSFGenerator(2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gen.forward(torch.randn(4, 2))


def test_kde_window_radius_and_bandwidth_limits():
    """The window radius the kernels pick from sigma / bin spacing (kde1d.cu window_radius), the boundaries of the
    compiled templates, and the refusal of wider kernels before anything needs the GPU."""
    from mentflow_b200 import ops
    assert ops.kde_window_radius(0.5) == 4 and ops.kde_window_radius(0.0) == 4      # <= 0: the default 0.5
    assert ops.kde_window_radius(0.05) == 1
    assert ops.kde_window_radius(0.505) == 4 and ops.kde_window_radius(0.515) == 5
    assert ops.kde_window_radius(1.07) == 9 and ops.kde_window_radius(1.08) == 10
    assert ops.kde_window_radius(1.52) == 13 and ops.kde_window_radius(1.53) == 14
    for radius in (4, 9, 13):
        top = ops.kde_max_ratio(radius)
        assert ops.kde_window_radius(top * (1 - 1e-6)) == radius and ops.kde_window_radius(top * (1 + 1e-6)) == radius + 1
    assert abs(ops.kde_max_ratio(ops.KDE1D_MAX_RADIUS) - 1.5254) < 1e-4
    assert abs(ops.kde_max_ratio(ops.KDE2D_MAX_RADIUS) - 1.0734) < 1e-4
    ops.check_kde_ratio(1.52, ops.KDE1D_MAX_RADIUS, "1-D")
    with pytest.raises(ValueError, match="1.5254"):
        ops.check_kde_ratio(1.53, ops.KDE1D_MAX_RADIUS, "1-D")
    with pytest.raises(ValueError, match="1.0734"):
        ops.check_kde_ratio(1.08, ops.KDE2D_MAX_RADIUS, "2-D")
    # the reference's default absolute bandwidth (1.0) on typical bins is refused with the limit, not a library error
    from mentflow_b200.diagnostics.histogram import kde_histogram_1d
    with pytest.raises(ValueError, match="bandwidth too wide"):
        kde_histogram_1d(torch.randn(100), torch.linspace(-3.5, 3.5, 65))


def test_projection_vectors_follow_transform_and_direction():
    m = torch.randn(4, 4)
    e = torch.linspace(-1, 1, 9)
    d_axis = mf.diagnostics.Histogram1D(axis=2, edges=e)
    d_dir = mf.diagnostics.Histogram1D(edges=e, direction=torch.tensor([1.0, 2.0, 0.0, -1.0]))
    x = torch.randn(50, 4)
    u = x @ m.T
    assert torch.allclose(x @ d_axis.projection_vector(m, 4, "cpu"), d_axis.project(u), atol=1e-5)
    assert torch.allclose(x @ d_dir.projection_vector(m, 4, "cpu"), d_dir.project(u), atol=1e-5)
    d2 = mf.diagnostics.Histogram2D(axis=(0, 2), edges=[e, e])
    assert torch.allclose(x @ d2.projection_vectors(m, 4, "cpu").T, d2.project(u), atol=1e-5)


def test_kl_matches_torch_kl_div():
    torch.manual_seed(0)
    p, t = torch.rand(64) + 0.01, torch.rand(64)
    t[:5] = 0.0
    want = torch.nn.functional.kl_div(torch.log(p + 1e-12), t, reduction="batchmean")
    assert torch.allclose(mf.loss.kl_divergence(p, t), want, rtol=1e-6)
    P, T = torch.rand(3, 8, 9) + 0.01, torch.rand(3, 8, 9)
    want = torch.stack([torch.nn.functional.kl_div(torch.log(a + 1e-12), b, reduction="batchmean")
                        for a, b in zip(P, T)])
    assert torch.allclose(mf.loss.kl_divergence_batched(P, T), want, rtol=1e-6)


def test_tensor_core_flow_host_side_contract():
    """Host-only parts of the flow entry points (dummy device pointers: every call fails before any CUDA call): which
    shapes the tcgen05 kernels are compiled for, the operand-image size, and the argument checks of the forward,
    inverse and backward when they are given an operand image."""
    import ctypes
    from mentflow_b200 import _lib
    lib = _lib.load()
    assert lib.mfb_nsf_tc_supported(6, 64, 3, 20) == 1 and lib.mfb_nsf_tc_supported(2, 64, 3, 20) == 1
    assert lib.mfb_nsf_tc_supported(6, 64, 2, 20) == 0 and lib.mfb_nsf_tc_supported(6, 64, 3, 16) == 0
    assert lib.mfb_nsf_tc_supported(7, 64, 3, 20) == 0 and lib.mfb_nsf_tc_supported(6, 32, 3, 20) == 0
    sizes = [lib.mfb_nsf_tc_image_bytes(d, 3) for d in range(2, 7)]
    assert all(s % 1024 == 0 for s in sizes) and sizes == sorted(sizes)
    # image + three 32 KB activation buffers + particle staging + barriers must fit one SM (227 KB)
    assert sizes[-1] + 3 * 32768 + 3 * 2 * 128 * 6 * 4 + 256 + 1024 <= 227 * 1024
    assert lib.mfb_nsf_tc_image_bytes(7, 3) == 0
    good_order = ctypes.cast((ctypes.c_int32 * 6)(5, 4, 3, 2, 1, 0), ctypes.c_void_p)
    bad_order = ctypes.cast((ctypes.c_int32 * 6)(0, 1, 2, 3, 4, 4), ctypes.c_void_p)      # not a permutation
    dummy = ctypes.c_void_p(16)
    assert lib.mfb_nsf_tc_prepare(dummy, 1, 1, 6, 64, 3, 20, bad_order, dummy, None) == -1
    assert b"bad argument" in lib.mfb_error_string(-1)

    def fwd(hidden_layers, image, order):
        return lib.mfb_nsf_layer_fwd(dummy, 10, 6, 64, hidden_layers, 20, dummy, image, order, None, 1, dummy, None,
                                     None)

    def inv(hidden_layers, image, order):
        return lib.mfb_nsf_layer_inv(dummy, 10, 6, 64, hidden_layers, 20, dummy, image, order, None, 1, dummy, None,
                                     None)

    def bwd(hidden_layers, image, order):
        return lib.mfb_nsf_layer_bwd(dummy, dummy, None, 10, 6, 64, hidden_layers, 20, dummy, dummy, image, order, 1,
                                     dummy, dummy, 0, dummy, 0, None)

    for call in (fwd, inv, bwd):
        assert call(2, dummy, good_order) == -2              # hidden_layers = 2 is not compiled for tcgen05
        assert call(3, dummy, bad_order) == -1               # the tcgen05 kernels need a permutation
        assert call(3, ctypes.c_void_p(24), good_order) == -1    # the image is loaded with a bulk copy: 16-byte aligned
        assert call(3, None, None) == -1                     # the order is required, with or without an image
        assert call(3, dummy, None) == -1
    # the tcgen05 forward and backward bulk-copy tiles of the layer input v: rows that start 4 bytes past a 16-byte
    # boundary are refused before anything else about the batch is looked at (an empty forward, a backward without
    # a workspace); the CUDA-core forward reads rows one by one and has nothing to do for n = 0
    v = ctypes.c_void_p(20)
    assert lib.mfb_nsf_layer_fwd(v, 0, 6, 64, 3, 20, dummy, dummy, good_order, None, 1, dummy, None, None) == -1
    assert lib.mfb_nsf_layer_fwd(v, 0, 6, 64, 3, 20, dummy, None, good_order, None, 1, dummy, None, None) == 0
    assert lib.mfb_nsf_layer_bwd(v, dummy, None, 10, 6, 64, 3, 20, dummy, dummy, dummy, good_order, 1, dummy, dummy, 0,
                                 dummy, 0, None) == -1


def test_flow_backward_chunks_start_on_aligned_rows(monkeypatch):
    """nsf_backward runs a batch in chunks of NSF_BWD_CHUNK particles rounded down to a multiple of 128 (at least 128):
    every chunk then starts on a 16-byte aligned row for every D, which the tcgen05 kernels' bulk copies need."""
    for chunk, n, want in [(1 << 20, 5, 5), (1 << 20, 2_000_000, 1 << 20), (1000, 5000, 896), (1, 5000, 128),
                           (0, 300, 128), (128, 100, 100), (1029, 100_000, 1024)]:
        monkeypatch.setattr(ops, "NSF_BWD_CHUNK", chunk)
        got = ops.nsf_bwd_chunk(n)
        assert got == want, (chunk, n)
        assert all(start * d * 4 % 16 == 0 for d in range(2, 7) for start in range(0, n, got))


def test_ment_entry_points_refuse_bad_arguments(monkeypatch):
    """Argument checks of the classical MENT entry points (dummy device pointers: every call fails before any CUDA
    call), and the refusal of a library built for another ABI version."""
    import ctypes
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)
    shape = (ctypes.c_int32 * 4)(8, 8, 8, 8)
    first = (ctypes.c_float * 4)(0.0, 0.0, 0.0, 0.0)
    step = (ctypes.c_float * 4)(0.1, 0.1, 0.1, 0.1)
    hp = [ctypes.cast(a, ctypes.c_void_p) for a in (shape, first, step)]

    def tables(mp=None, mp2=None):
        # 1-D family: k = 3 tables of 8 bins; 2-D family: k2 = 2 tables of 8 x 8 bins
        return [dummy, dummy, dummy, 3, 8, mp, dummy, dummy, dummy, dummy, 2, 8, 8, mp2]

    def prob(*t):
        return lib.mfb_ment_prob(dummy, 100, 4, *t, 0.0, 0.0, dummy, None)

    def prob_grid(*t):
        return lib.mfb_ment_prob_grid(4, *hp, *t, 0.0, 0.0, dummy, None)

    def integrate(*t, ax2=1, inv_mp=dummy):
        return lib.mfb_ment_integrate(4, dummy, 8, 0, dummy, 8, ax2, 2, *hp, dummy, inv_mp, *t, 0.0, 0.0, dummy, None)

    # a 2-D screen measured twice on one axis
    assert integrate(*tables(), ax2=0, inv_mp=None) == -1
    # with kicks, a non-empty family needs its multipole rows
    for call in (prob, prob_grid, integrate):
        assert call(*tables(mp=None, mp2=dummy)) == -1
        assert call(*tables(mp=dummy, mp2=None)) == -1
    # with kicks, integrate mode needs the inverse kick
    assert integrate(*tables(mp=dummy, mp2=dummy), inv_mp=None) == -1
    # names of this ABI exist in older libraries with other argument lists: another version is refused
    monkeypatch.setattr(_lib, "ABI_VERSION", _lib.ABI_VERSION - 1)
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(_lib.LibraryMissing, match="ABI version"):
        _lib.load()


def test_kde1d_forward_refuses_inconsistent_outputs():
    """Argument checks of mfb_project_kde1d_fwd's two modes (sums only / sums + profiles (+ KL)); dummy device
    pointers: every call fails before any CUDA call."""
    import ctypes
    lib = _lib.load()
    dummy = ctypes.c_void_p(16)

    def fwd(n=1000, n_total=1000.0, meas=None, profiles=None, kl=None):
        return lib.mfb_project_kde1d_fwd(dummy, n, 4, dummy, None, dummy, 3, 64, 0.5, n_total, meas, 1e-12, dummy,
                                         profiles, kl, dummy, 1 << 20, None)

    assert fwd(meas=dummy, profiles=dummy) == -1                 # meas without kl
    assert fwd(profiles=dummy, kl=dummy) == -1                   # kl without meas
    assert fwd(meas=dummy, kl=dummy) == -1                       # meas / kl without profiles
    assert fwd(n=0, profiles=dummy) == -1                        # profiles of no particles
    assert fwd(n_total=0.0, profiles=dummy) == -1
    assert fwd(n_total=-1.0, profiles=dummy, meas=dummy, kl=dummy) == -1


def test_graphed_loss_chunk_plan():
    """Pieces of the pinned-host input: tile aligned, growing, covering the batch exactly."""
    from mentflow_b200.graphs import GraphedLoss
    g = GraphedLoss.__new__(GraphedLoss)
    for n, c in [(1_000_000, 1), (1_000_000, 2), (1_000_000, 4), (20_000, 3), (1000, 3), (129, 2)]:
        g.batch_size, g.host_chunks = n, c
        b = g._chunk_bounds()
        assert b[0][0] == 0 and b[-1][1] == n and all(x[1] == y[0] for x, y in zip(b, b[1:]))
        assert all(a % 128 == 0 for a, _ in b) and len(b) <= c
        if len(b) > 1:
            assert b[0][1] - b[0][0] <= b[1][1] - b[1][0]


def test_plan_groups_multipole_chains_and_tracks_their_parameters():
    """simulate.forward's plan (host logic only, no kernel runs): linear maps and linear -> kick -> linear
    chains in front of 1-D screens go to fused groups, everything else to the object-by-object path; the
    plan key follows the kick's mutable attributes."""
    import mentflow_b200 as mf
    from mentflow_b200.simulate import simulate as sim
    x = torch.zeros(4, 4)
    edges = torch.linspace(-1.0, 1.0, 9)
    h1 = mf.diagnostics.Histogram1D(axis=0, edges=edges, bandwidth=0.5)
    h2 = mf.diagnostics.Histogram2D(axis=(0, 2), edges=(edges, edges), bandwidth=(0.5, 0.5))
    lin = mf.simulate.LinearTransform(torch.eye(4))
    kick = mf.simulate.MultipoleTransform(order=3, strength=0.5)
    chain = mf.simulate.CompositeTransform(lin, kick, mf.simulate.LinearTransform(2.0 * torch.eye(4)))
    two_kicks = mf.simulate.CompositeTransform(kick, mf.simulate.MultipoleTransform(order=4, strength=0.1))

    class Custom(mf.simulate.Transform):
        def forward(self, x):
            return x

    transforms = [lin, chain, kick, two_kicks, Custom(), mf.simulate.CompositeTransform(lin, lin)]
    diagnostics = [[h1, h2], [h1, h2], [h1], [h1], [h1], [h1]]
    plan = sim._build_plan(x, transforms, diagnostics)
    kinds = {key[0]: grp for key, grp in plan.groups.items()}
    assert set(kinds) == {"1d", "2d", "1d-mp"}
    assert kinds["1d"].slots == [(0, 0), (5, 0)] and kinds["2d"].slots == [(0, 1)]
    assert kinds["1d-mp"].slots == [(1, 0), (2, 0)]
    assert kinds["1d-mp"].proj.shape == (2, 4) and kinds["1d-mp"].mp.shape == (2, 12)
    # a 2-D screen behind a kick, a chain with two kicks and a user-defined map are not fused
    assert plan.fallback == [(1, 1), (3, 0), (4, 0)]
    # measured row of the chain: post = 2 I, pre = I, normal kick: w = 2 e0, a = b = 0 (row has no momentum part)
    w, mp = kinds["1d-mp"].proj[0], kinds["1d-mp"].mp[0]
    assert torch.allclose(w, torch.tensor([2.0, 0.0, 0.0, 0.0])) and float(mp[8]) == 0.0 and float(mp[9]) == 0.0
    assert int(mp[10]) == 3
    key = sim._plan_key(transforms, diagnostics)
    kick.strength = 0.7
    assert sim._plan_key(transforms, diagnostics) != key
    kick.strength = 0.5
    assert sim._plan_key(transforms, diagnostics) == key
    kick.order = 2                      # not an order the reference accepts: no folding
    assert sim._multipole_chain(chain) is None


def test_plan_cache_is_not_fooled_by_recycled_ids(monkeypatch):
    """A fresh LinearTransform per call (its id may be the id of a freed one) must never reuse the projection
    rows of an earlier transform; editing a screen's bandwidth in place rebuilds its geometry."""
    from mentflow_b200.simulate import simulate as sim
    seen = []

    def fake_project_kde1d(x, proj, geom, ratio, nbins, reducer=None, meas=None, mp=None):
        seen.append((proj.clone(), geom.clone()))
        return torch.zeros(proj.shape[0], nbins)

    monkeypatch.setattr(sim.ops, "project_kde1d", fake_project_kde1d)
    sim._plan_cache.clear()
    diag = mf.diagnostics.Histogram1D(axis=0, edges=torch.linspace(-3, 3, 33), bandwidth=0.5)
    x = torch.zeros(4, 2)
    torch.manual_seed(0)
    for it in range(300):
        m = torch.randn(2, 2)
        sim.forward(x, [mf.simulate.LinearTransform(m)], [[diag]])
        proj, _ = seen[-1]
        assert torch.equal(proj[0], m[0]), f"stale projection row at call {it}"
    sigma0 = float(seen[-1][1][0, 2])
    t = mf.simulate.LinearTransform(torch.eye(2))
    sim.forward(x, [t], [[diag]])
    diag.bandwidth.mul_(2.0)
    sim.forward(x, [t], [[diag]])
    assert abs(float(seen[-1][1][0, 2]) - 2.0 * sigma0) < 1e-7


def test_philox_stream_contract_without_gpu():
    """base noise never falls back to the host: a CPU tensor is refused"""
    with pytest.raises(RuntimeError):
        ops.PhiloxStream("cpu").normal_(torch.empty(4, 2))
    lib = _lib.load()
    assert lib.mfb_randn_offset_increment(0) == 0


def test_mentflow_checkpoint_round_trip(tmp_path):
    """MENTFlow.save / load (core.py:122-143): generator weights under zuko-style names plus the pickled
    measurement setup; loading into a freshly initialised model reproduces weights and setup."""
    import mentflow_b200 as mf
    torch.manual_seed(0)
    edges = torch.linspace(-2.0, 2.0, 17)

    def make(seed):
        torch.manual_seed(seed)
        gen = mf.generate.build_generator("nsf", input_features=2, output_features=2, hidden_layers=3,
                                          hidden_units=64, transforms=2, bins=20)
        tfs = [mf.simulate.LinearTransform(mf.simulate.rotation_matrix(a).float()) for a in (0.0, 0.7)]
        diags = [[mf.diagnostics.Histogram1D(axis=0, edges=edges, bandwidth=0.5)] for _ in tfs]
        meas = [[torch.rand(16)] for _ in tfs]
        prior = mf.prior.Gaussian(ndim=2, scale=2.0)
        return mf.MENTFlow(transforms=tfs, diagnostics=diags, measurements=meas, generator=gen, prior=prior,
                           entropy_estimator=mf.entropy.MonteCarloEntropyEstimator(prior=prior),
                           discrepancy_function="kld", penalty_parameter=5.0)

    a, b = make(1), make(2)
    assert a.discrepancy_function is mf.loss.kl_divergence          # the reference's string default is resolved
    assert not torch.equal(next(a.parameters()), next(b.parameters()))
    path = tmp_path / "model.pt"
    a.save(path)
    b.load(path, device="cpu")
    for pa, pb in zip(a.parameters(), b.parameters()):
        assert torch.equal(pa, pb)
    assert torch.equal(b.measurements[1][0], a.measurements[1][0])
    assert torch.equal(b.transforms[1].matrix, a.transforms[1].matrix)
    assert isinstance(b.entropy_estimator, mf.entropy.MonteCarloEntropyEstimator)
    state = torch.load(path, weights_only=False)
    assert set(state) == {"generator", "entropy_estimator", "transforms", "diagnostics", "measurements"}
    assert any(k.startswith("_flow.transform.transforms.0.hyper.0.") for k in state["generator"])
