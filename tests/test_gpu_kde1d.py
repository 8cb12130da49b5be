"""GPU parity: fused projection + 1-D KDE / exact histogram vs the reference goldens and the
CPU oracle.  Tolerances follow SURVEY.md 8c: KDE profiles |a-b| <= 1e-4 * max|ref| per
profile; histogram counts bit-exact; loss / gradients rel 1e-4."""
import numpy as np
import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200 import ops
from mfb_testutil import cuda, geom_rows, profile_err, t32
from oracle import hotpath as hp

pytestmark = pytest.mark.gpu
TOL = 1.0e-4


def _setup(g, bandwidth=0.5, direction=None, kde=True):
    mats, edges = t32(g["matrices"]), t32(g["edges"])
    tfs = [mf.simulate.LinearTransform(m.cuda()) for m in mats]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=edges, bandwidth=bandwidth, direction=direction, kde=kde).to("cuda")
    return tfs, [[diag] for _ in tfs], diag


def test_kde1d_6d_matches_reference_golden(golden):
    g = golden("kde1d_6d")
    tfs, diags, _ = _setup(g)
    x = cuda(g["x"])
    out = mf.simulate.forward(x, tfs, diags)
    got = torch.stack([o[0] for o in out])
    assert profile_err(got, t32(g["kde"])) < TOL
    # each diagnostic called on its own (reference usage: diagnostic(transform(x)))
    single = diags[3][0](tfs[3](x))
    assert profile_err(single[None], t32(g["kde"])[3:4]) < TOL


def test_kde1d_2d_rotations_direction_and_wide_kernel(golden):
    g = golden("kde1d_2d")
    x = cuda(g["x"])
    tfs, diags, _ = _setup(g)
    got = torch.stack([o[0] for o in mf.simulate.forward(x, tfs, diags)])
    assert profile_err(got, t32(g["kde"])) < TOL
    tfs, diags, _ = _setup(g, bandwidth=float(g["bandwidth_dir"]), direction=t32(g["direction"]))
    got = torch.stack([o[0] for o in mf.simulate.forward(x, tfs, diags)])
    assert profile_err(got, t32(g["kde_dir"])) < TOL


def test_hard_histogram_bit_exact(golden):
    g = golden("kde1d_6d")
    edges = t32(g["edges"])
    # identical x_proj -> identical integer counts and bit-identical density
    for k in range(g["uproj"].shape[0]):
        u = t32(g["uproj"][k])
        counts = ops.project_hist1d(u.cuda().reshape(-1, 1), torch.ones(1, 1, device="cuda"), edges.cuda()[None])
        assert torch.equal(counts[0].cpu(), hp.hist_counts_1d(u, edges))
        diag = mf.diagnostics.Histogram1D(axis=0, edges=edges, kde=False).to("cuda")
        assert torch.equal(diag.bin(u.cuda()).cpu(), t32(g["hard"][k]))
    # edge cases: values exactly on edges, outside, NaN, +-inf
    e = edges
    u = torch.cat([e, e[:-1] + 0.5 * (e[1] - e[0]), torch.tensor([-10.0, 10.0, float("nan"), float("inf"),
                                                                 -float("inf")]),
                   torch.nextafter(e, torch.tensor(10.0)), torch.nextafter(e, torch.tensor(-10.0))])
    counts = ops.project_hist1d(u.cuda().reshape(-1, 1), torch.ones(1, 1, device="cuda"), e.cuda()[None])
    assert torch.equal(counts[0].cpu(), hp.hist_counts_1d(u, e))
    assert torch.equal(counts[0].cpu().float(), torch.histogram(u[~torch.isnan(u)], e).hist)


def test_fused_hard_histogram_through_simulate(golden):
    g = golden("kde1d_6d")
    tfs, diags, diag = _setup(g, kde=False)
    x = cuda(g["x"])
    got = torch.stack([o[0] for o in mf.simulate.forward(x, tfs, diags)]).cpu()
    ref = t32(g["hard"])
    # The fused projection is an ascending fused-multiply-add chain from zero, which reproduces the reference's
    # `x @ M.T` (MKL sgemm, K = 6) BIT FOR BIT: checked on the CPU against the golden `uproj`
    # (tests/test_oracle_golden.py::test_projection_order_reproduces_reference_bits), so every particle lands in
    # the reference's bin and the counts are identical
    width = torch.diff(t32(g["edges"]))
    n = g["x"].shape[0]
    cg = torch.round(got * width * n)
    cr = torch.round(ref * width * n)
    assert torch.equal(cg, cr)
    assert torch.allclose(got, ref, rtol=1e-6, atol=0)


def test_kl_gradient_matches_reference_autograd(golden):
    g = golden("kde1d_6d")
    tfs, diags, _ = _setup(g)
    meas = cuda(g["meas"])
    x = cuda(g["x"]).requires_grad_(True)
    out = mf.simulate.forward(x, tfs, diags)
    kl = torch.stack([mf.loss.kl_divergence(o[0], m) for o, m in zip(out, meas)])
    assert torch.allclose(kl.detach().cpu(), t32(g["kl"]), rtol=TOL, atol=1e-7)
    loss = kl.sum() / len(tfs)
    loss.backward()
    assert abs(float(loss) - float(g["mean_kl"])) <= TOL * abs(float(g["mean_kl"]))
    ref = t32(g["grad_x"])
    assert (x.grad.cpu() - ref).abs().max() <= TOL * ref.abs().max()
    mae = torch.stack([mf.loss.mean_absolute_error(o[0], m) for o, m in zip(out, meas)])
    assert torch.allclose(mae.detach().cpu(), t32(g["mae"]), rtol=TOL)


@pytest.mark.parametrize("n,d,k,nb", [(1, 6, 3, 64), (5, 2, 1, 8), (1023, 3, 7, 33), (70001, 6, 100, 64),
                                      (4097, 5, 300, 16), (300000, 2, 7, 85), (2000, 8, 4, 200)])
def test_kde1d_vs_oracle_ragged_shapes(n, d, k, nb):
    gen = torch.Generator().manual_seed(n + d + k)
    x = torch.randn(n, d, generator=gen)
    w = torch.randn(k, d, generator=gen)
    w = w / w.norm(dim=1, keepdim=True)
    edges = torch.linspace(-3.5, 3.5, nb + 1)
    geom, sigma = geom_rows(edges, 0.5, k)
    sums = ops.kde1d_sums(x.cuda(), w.cuda(), geom.cuda(), 0.5, nb).cpu().double()
    ref = torch.stack([hp.kde_sums_1d(x @ w[i], edges, sigma) for i in range(k)])
    assert float((sums - ref).abs().max() / ref.abs().max()) < 2e-5
    # deterministic: same launch twice gives the same bits
    again = ops.kde1d_sums(x.cuda(), w.cuda(), geom.cuda(), 0.5, nb).cpu().double()
    assert torch.equal(sums, again)
    counts = ops.project_hist1d(x.cuda(), w.cuda(), edges.cuda()[None].repeat(k, 1)).cpu()
    tot = 0
    for i in range(k):
        refc = hp.hist_counts_1d(x @ w[i], edges)
        tot += int((counts[i] - refc).abs().sum())
    assert tot <= max(4, n * k // 20000)      # 1-ulp projection differences at bin edges only
    assert int(counts.sum()) <= n * k


def test_full_size_properties():
    """BASELINE size (D=6, K=100, B=64, N=1e6): linearity in the particle set and mass
    conservation -- properties that do not need the dense oracle."""
    n, d, k, nb = 1_000_000, 6, 100, 64
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, d, generator=gen, device="cuda")
    w = torch.randn(k, d, generator=gen, device="cuda")
    w = w / w.norm(dim=1, keepdim=True)
    edges = torch.linspace(-3.5, 3.5, nb + 1)
    delta = float(edges[1] - edges[0])
    geom = geom_rows(edges, 0.5, k)[0].cuda()
    full = ops.kde1d_sums(x, w, geom, 0.5, nb).double()
    half = ops.kde1d_sums(x[: n // 2], w, geom, 0.5, nb).double() + ops.kde1d_sums(x[n // 2:], w, geom, 0.5, nb).double()
    assert float((full - half).abs().max() / full.max()) < 1e-5
    # total kernel mass per particle = sigma*sqrt(2 pi)/delta for particles well inside the screen
    inside = (x @ w.T).abs().max(dim=1).values < 2.5
    s_in = ops.kde1d_sums(x[inside].contiguous(), w, geom, 0.5, nb).double().sum(dim=1) / int(inside.sum())
    assert torch.allclose(s_in, torch.full_like(s_in, 0.5 * np.sqrt(2 * np.pi)), rtol=1e-3)
    counts = ops.project_hist1d(x, w, edges.cuda()[None].repeat(k, 1))
    n_in = ((x @ w.T >= edges[0]) & (x @ w.T <= edges[-1])).sum(dim=0)
    assert (counts.sum(dim=1) - n_in).abs().max() <= 2
    prof = ops.kde1d_finish(full.float(), n, geom, None)[0]
    assert torch.allclose(prof.sum(dim=1) * delta, torch.ones(k, device="cuda"), atol=1e-5)


@pytest.mark.parametrize("n,d,k,nb,kick", [pytest.param(*c, False, id="-".join(map(str, c))) for c in
                                           [(1, 6, 3, 64), (4097, 4, 11, 37), (70001, 6, 100, 64), (3000, 2, 5, 300),
                                            (2000, 3, 2, 1000)]] + [pytest.param(30001, 4, 7, 64, True, id="30001-4-7-64-kick")])
def test_fused_loss_tail_matches_separate_kernels_and_torch_kl(n, d, k, nb, kick):
    """deposit + merge + normalise + KL in two launches (mfb_project_kde1d_fwd with profiles / _finish / _finish_bwd)
    vs the torch expression of loss.py:15-17, values and gradients; ``kick``: screens behind a multipole kick."""
    gen = torch.Generator().manual_seed(7 * n + k)
    x = torch.randn(n, d, generator=gen).cuda()
    w = torch.randn(k, d, generator=gen)
    w = (w / w.norm(dim=1, keepdim=True)).cuda()
    mp = None
    if kick:                                      # kick -> screen row, orders 3, 4, 5, normal and skew
        from mentflow_b200.simulate.simulate import multipole_terms
        terms = [multipole_terms(w[i], None, mf.simulate.MultipoleTransform(3 + i % 3, 0.5 - 0.15 * i, i % 2 == 1), d)
                 for i in range(k)]
        w = torch.stack([t[0] for t in terms]).cuda()
        mp = torch.stack([t[1] for t in terms]).cuda()
    edges = torch.linspace(-3.5, 3.5, nb + 1)
    geom = geom_rows(edges, 0.5, k)[0].cuda()
    meas = torch.rand(k, nb, generator=gen)
    meas[:, : nb // 4] = 0.0                      # empty bins: 0 log 0 = 0
    meas = (meas / meas.sum(dim=1, keepdim=True) * nb / 7.0).cuda()

    xa = x.clone().requires_grad_(True)
    prof_a, kl_a = ops.project_kde1d(xa, w, geom, 0.5, nb, None, meas, mp)
    xb = x.clone().requires_grad_(True)
    prof_b = ops.project_kde1d(xb, w, geom, 0.5, nb, mp=mp)
    kl_b = mf.loss.kl_divergence_batched(prof_b, meas)
    assert float((prof_a - prof_b).abs().max()) <= 2e-6 * float(prof_b.abs().max())
    assert torch.allclose(kl_a, kl_b, rtol=2e-5, atol=1e-6)
    # the merged sums agree with the stand-alone merge bit for bit (same kernel, same order)
    sums = ops.kde1d_sums(x, w, geom, 0.5, nb, mp)
    prof_c, kl_c = ops.kde1d_finish(sums, float(n), geom, meas)
    assert torch.equal(prof_c, prof_a) and torch.equal(kl_c, kl_a)

    coef = torch.linspace(0.5, 1.5, k).cuda()
    side = torch.randn(k, nb, generator=gen).cuda()
    ((kl_a * coef).sum() + (prof_a * side).sum()).backward()
    ((kl_b * coef).sum() + (prof_b * side).sum()).backward()
    scale = float(xb.grad.abs().max())
    assert float((xa.grad - xb.grad).abs().max()) <= 1e-4 * scale
    # KL only (no gradient through the profiles): the materialised-zero path is skipped
    xc = x.clone().requires_grad_(True)
    _, kl_only = ops.project_kde1d(xc, w, geom, 0.5, nb, None, meas, mp)
    kl_only.sum().backward()
    xd = x.clone().requires_grad_(True)
    mf.loss.kl_divergence_batched(ops.project_kde1d(xd, w, geom, 0.5, nb, mp=mp), meas).sum().backward()
    assert float((xc.grad - xd.grad).abs().max()) <= 1e-4 * float(xd.grad.abs().max())


def test_fused_loss_tail_with_reducer_path():
    """With a reducer (sharded particles) the tail runs from the all-reduced sums: two half batches whose
    sums are added by the 'reducer' give the profiles and KL of the whole batch."""
    gen = torch.Generator().manual_seed(5)
    n, d, k, nb = 20000, 6, 9, 64
    x = torch.randn(n, d, generator=gen).cuda()
    w = torch.randn(k, d, generator=gen)
    w = (w / w.norm(dim=1, keepdim=True)).cuda()
    geom = geom_rows(torch.linspace(-3.5, 3.5, nb + 1), 0.5, k)[0].cuda()
    meas = torch.rand(k, nb, generator=gen).cuda()
    other = ops.kde1d_sums(x[n // 2:].contiguous(), w, geom, 0.5, nb)

    def reducer(sums, n_local):
        if sums.dtype == torch.float32 and sums.shape == other.shape:
            sums += other
        return float(n)

    prof_r, kl_r = ops.project_kde1d(x[: n // 2].contiguous(), w, geom, 0.5, nb, reducer, meas)
    prof_f, kl_f = ops.project_kde1d(x, w, geom, 0.5, nb, None, meas)
    assert float((prof_r - prof_f).abs().max()) <= 1e-5 * float(prof_f.abs().max())
    assert torch.allclose(kl_r, kl_f, rtol=1e-4, atol=1e-6)


def _nonlinear_setup(g):
    matrix = t32(g["nl_matrix"]).cuda()
    tfs = [mf.simulate.CompositeTransform(mf.simulate.MultipoleTransform(order=int(g["nl_order"]), strength=float(st)),
                                          mf.simulate.LinearTransform(matrix)) for st in g["nl_strengths"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=t32(g["nl_edges"]), bandwidth=0.5).to("cuda")
    return tfs, [[diag] for _ in tfs], diag


def test_multipole_chain_runs_in_the_fused_kernel_and_matches_reference(golden):
    """rec_2d/nonlinear (experiments/rec_2d/nonlinear/setup.py:24-44): multipole kick -> rotation -> screen.
    KDE profiles, exact histograms and the gradient of the mean KL against the reference's own outputs."""
    from mentflow_b200.simulate import simulate as sim
    g = golden("multipole")
    tfs, diags, diag = _nonlinear_setup(g)
    x = cuda(g["nl_x"]).requires_grad_(True)
    sim._plan_cache.clear()
    out = mf.simulate.forward(x, tfs, diags)
    plan = next(iter(sim._plan_cache.values()))
    assert not plan.fallback and [k[0] for k in plan.groups] == ["1d-mp"]     # no object-by-object path
    kde = torch.stack([o[0] for o in out])
    ref = t32(g["nl_kde"])
    assert profile_err(kde.detach().cpu(), ref) < TOL
    meas = cuda(g["nl_meas"])
    loss = torch.stack([mf.loss.kl_divergence(o[0], m) for o, m in zip(out, meas)]).sum() / len(tfs)
    loss.backward()
    assert abs(float(loss) - float(g["nl_mean_kl"])) <= TOL * abs(float(g["nl_mean_kl"]))
    gref = t32(g["nl_grad_x"])
    assert (x.grad.cpu() - gref).abs().max() <= TOL * gref.abs().max()
    # exact histograms: identical up to particles whose fp32 coordinate rounds across an edge
    diag.kde = False
    hard = torch.stack([o[0] for o in mf.simulate.forward(x.detach(), tfs, diags)]).cpu()
    diag.kde = True
    n, width = x.shape[0], float(g["nl_edges"][1] - g["nl_edges"][0])
    moved = ((hard - t32(g["nl_hard"])).abs() * n * width).sum(dim=1)          # in particles, per screen
    assert float(moved.max()) <= 4.5


@pytest.mark.parametrize("d,order,skew", [(2, 4, False), (4, 3, False), (4, 5, True), (6, 3, True), (6, 4, False)])
def test_multipole_chain_general_matrices_vs_oracle(d, order, skew):
    """linear -> kick -> linear with random matrices in 2, 4 and 6 dimensions: fused kernel vs the dense CPU
    oracle applied to the coordinates the transform classes produce (reference semantics), and the
    particle gradient vs torch autograd through the same classes."""
    gen = torch.Generator().manual_seed(100 * d + order)
    n, k, nb = 5000, 5, 64
    x = (torch.randn(n, d, generator=gen) * 0.7).float()
    edges = torch.linspace(-3.5, 3.5, nb + 1)
    chains, cpu_chains = [], []
    for i in range(k):
        pre = torch.eye(d) + 0.3 * torch.randn(d, d, generator=gen)
        post = torch.eye(d) + 0.3 * torch.randn(d, d, generator=gen)
        st = 0.5 - 0.2 * i
        cpu_chains.append(mf.simulate.CompositeTransform(mf.simulate.LinearTransform(pre.double()),
                                                         mf.simulate.MultipoleTransform(order, st, skew),
                                                         mf.simulate.LinearTransform(post.double())))
        chains.append(mf.simulate.CompositeTransform(mf.simulate.LinearTransform(pre.cuda()),
                                                     mf.simulate.MultipoleTransform(order, st, skew),
                                                     mf.simulate.LinearTransform(post.cuda())))
    diag = mf.diagnostics.Histogram1D(axis=0, edges=edges, bandwidth=0.5).to("cuda")
    xg = x.cuda().requires_grad_(True)
    out = mf.simulate.forward(xg, chains, [[diag] for _ in chains])
    side = torch.randn(k, nb, generator=gen).cuda()
    (torch.stack([o[0] for o in out]) * side).sum().backward()
    sigma = 0.5 * float(edges[1] - edges[0])
    xr = x.double().requires_grad_(True)
    ref = []
    for c in cpu_chains:
        u = c(xr)[:, 0]
        ref.append(hp.kde_profile_1d(u, edges.double(), sigma))
    ref = torch.stack(ref)
    (ref * side.cpu().double()).sum().backward()
    got = torch.stack([o[0] for o in out]).detach().cpu().double()
    assert float((got - ref.detach()).abs().max()) <= TOL * float(ref.abs().max())
    assert float((xg.grad.cpu().double() - xr.grad).abs().max()) <= TOL * float(xr.grad.abs().max())


def test_p2p_finish_kernel_with_one_rank_matches_fused_tail():
    """The sharded tail (cross-rank sum over peer memory inside the finish kernel) with world = 1: the "peer" block
    is this rank's own buffer, so the result must equal the single-GPU fused tail bit for bit, across several
    steps (epoch counter, double buffering) and with a double tail riding along.  Two or more ranks are checked by
    bench.py's shard_parity at N > 1."""
    from mentflow_b200 import _lib
    lib = _lib.load()
    torch.manual_seed(3)
    n, d, k, nb = 50_001, 6, 10, 64
    w = torch.randn(k, d)
    w = (w / w.norm(dim=1, keepdim=True)).cuda()
    edges = torch.linspace(-3.5, 3.5, nb + 1)
    geom = geom_rows(edges, 0.5, k)[0].cuda()
    meas = torch.rand(k, nb).cuda()
    meas = meas / meas.sum(dim=1, keepdim=True) / float(edges[1] - edges[0])

    class OneRank:
        rank, world = 0, 1

        def __init__(self):
            self.block = torch.zeros(int(lib.mfb_kde1d_p2p_block_floats(k, nb, 2)), dtype=torch.float32, device="cuda")
            self.state = torch.zeros(4, dtype=torch.int32, device="cuda")

        def block_for(self, k_, b_, tail_, device):
            return self.block, None, [self.block.data_ptr()], self.state

    peer = OneRank()
    for step in range(1, 5):
        x = torch.randn(n, d, device="cuda") * (0.5 + 0.2 * step)
        tail = torch.tensor([1.5 * step, -2.25], dtype=torch.float64, device="cuda")
        sums, prof, kl, tail_sum = ops.kde1d_loss_forward_p2p(peer, x, w, geom, 0.5, nb, tail, float(n), meas)
        s0, p0, k0 = ops.kde1d_loss_forward(x, w, geom, 0.5, nb, float(n), meas)
        assert torch.equal(sums, s0) and torch.equal(prof, p0) and torch.equal(kl, k0)
        assert torch.equal(tail_sum, tail)
        assert peer.state[:3].tolist() == [2 * step - 1, 0, 0]
        # the already merged variant of the same kernel (a second epoch on the same block)
        s1, p1, k1, t1 = ops.kde1d_finish_p2p(peer, s0, tail, float(n), geom, meas)
        assert torch.equal(p1, p0) and torch.equal(k1, k0) and torch.equal(t1, tail)
        assert peer.state[:3].tolist() == [2 * step, 0, 0]
