"""GPU parity: fused projection + 2-D KDE / exact 2-D histogram vs reference goldens."""
import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200 import ops
from mfb_testutil import cuda, geom_rows, profile_err, t32
from oracle import hotpath as hp

pytestmark = pytest.mark.gpu
TOL = 1.0e-4


def _setup(g, kde=True):
    mats = t32(g["matrices"])
    ex, ey = t32(g["edges_x"]), t32(g["edges_y"])
    bw = tuple(float(b) for b in g["bandwidth"])
    tfs = [mf.simulate.LinearTransform(m.cuda()) for m in mats]
    diag = mf.diagnostics.Histogram2D(axis=(0, 2), edges=[ex, ey], bandwidth=bw, kde=kde).to("cuda")
    return tfs, [[diag] for _ in tfs]


def test_kde2d_matches_reference_golden(golden):
    g = golden("kde2d_4d")
    tfs, diags = _setup(g)
    x = cuda(g["x"])
    got = torch.stack([o[0] for o in mf.simulate.forward(x, tfs, diags)])
    assert profile_err(got, t32(g["kde"])) < TOL
    again = torch.stack([o[0] for o in mf.simulate.forward(x, tfs, diags)])
    assert torch.equal(got, again)           # fixed-point accumulation: bit-reproducible
    meas = cuda(g["meas"])
    kl = torch.stack([mf.loss.kl_divergence(p, m) for p, m in zip(got, meas)])
    assert torch.allclose(kl.cpu(), t32(g["kl"]), rtol=TOL, atol=1e-7)


def test_hist2d_exact_on_permutation_screens(golden):
    g = golden("kde2d_4d")
    tfs, diags = _setup(g, kde=False)
    x = cuda(g["x"])
    got = torch.stack([o[0] for o in mf.simulate.forward(x, tfs, diags)]).cpu()
    # corner matrices are permutations: projections are exact, so counts are bit-exact
    ref = t32(g["hard"])
    assert torch.allclose(got, ref, rtol=2e-6, atol=0)
    ex, ey = t32(g["edges_x"]), t32(g["edges_y"])
    mats = t32(g["matrices"])
    for k in range(len(mats)):
        uv = hp.linear_map(t32(g["x"]), mats[k])[:, [0, 2]]
        proj = mats[k][[0, 2]].cuda()[None]
        counts = ops.project_hist2d(x, proj, ex.cuda()[None], ey.cuda()[None])[0].cpu()
        assert torch.equal(counts, hp.hist_counts_2d(uv, ex, ey))


def test_kde2d_gradient_matches_reference_autograd(golden):
    g = golden("kde2d_4d")
    tfs, diags = _setup(g)
    meas = cuda(g["meas"])
    x = cuda(g["x"]).requires_grad_(True)
    out = mf.simulate.forward(x, tfs, diags)
    loss = sum(mf.loss.kl_divergence(o[0], m) for o, m in zip(out, meas)) / len(tfs)
    loss.backward()
    assert abs(float(loss) - float(g["mean_kl"])) <= TOL * abs(float(g["mean_kl"]))
    ref = t32(g["grad_x"])
    assert (x.grad.cpu() - ref).abs().max() <= TOL * ref.abs().max()


@pytest.mark.parametrize("n,d,k,bx,by", [(1, 4, 1, 8, 8), (999, 6, 15, 85, 85), (200000, 4, 6, 85, 85), (5000, 3, 2, 20, 31),
                                         # limits of the tensor-core path: the largest screen it takes and one bin more
                                         (5000, 4, 3, 128, 96), (5000, 4, 2, 129, 96), (5000, 4, 2, 128, 97),
                                         # either side of the batch size that selects it, and a ragged 64-particle tile
                                         (4095, 6, 3, 32, 32), (4096, 6, 3, 32, 32), (4097, 6, 3, 32, 32),
                                         # five screens' accumulators are resident in TMEM at a time
                                         (8192, 4, 5, 40, 40), (8192, 4, 6, 40, 40), (8192, 4, 10, 40, 40),
                                         (8192, 4, 11, 40, 40)])
def test_kde2d_vs_oracle_shapes(n, d, k, bx, by):
    gen = torch.Generator().manual_seed(n + k)
    x = torch.randn(n, d, generator=gen)
    w = torch.randn(k, 2, d, generator=gen)
    w = w / w.norm(dim=2, keepdim=True)
    ex, ey = torch.linspace(-3.5, 3.5, bx + 1), torch.linspace(-3.0, 3.0, by + 1)
    (gx, sx), (gy, sy) = geom_rows(ex, 0.5, k), geom_rows(ey, 0.5, k)
    geom = torch.stack([gx, gy], dim=1)
    prof = ops.project_kde2d(x.cuda(), w.cuda(), geom.cuda(), 0.5, bx, by).cpu()
    ref = torch.stack([hp.kde_profile_2d(x @ w[i, 0], x @ w[i, 1], ex, ey, sx, sy, chunk=20000)
                       for i in range(k)])
    assert profile_err(prof, ref) < TOL
    # screens up to 128 x 96 bins and batches of at least 4096 particles run on the tensor cores
    from mentflow_b200 import _lib
    tc = bool(_lib.load().mfb_kde2d_uses_tensor_cores(n, d, bx, by, 0 if ops.KDE2D_USE_TENSOR_CORES else 1))
    assert tc == (ops.KDE2D_USE_TENSOR_CORES and n >= 4096 and bx <= 128 and by <= 96)


def test_kde2d_tensor_core_and_fixed_point_paths_agree():
    """The tcgen05 GEMM over the particle axis (dense kernel rows in split bf16, kde2d_tc.cu) and the windowed
    44-bit fixed-point deposits against a float64 evaluation of the reference's dense form
    (diagnostics/histogram.py:47-74), bin by bin and by magnitude decade, far tails included; the
    tensor-core path is run-to-run bit-reproducible and its fixed-point planes reproduce its sums."""
    from mentflow_b200 import _lib
    lib = _lib.load()
    gen = torch.Generator().manual_seed(9)
    n, d, k, bx, by = 60_000, 6, 7, 85, 85          # 7 screens: two groups of TMEM-resident accumulators
    x = (torch.randn(n, d, generator=gen) * 0.8).cuda()
    w = torch.randn(k, 2, d, generator=gen)
    w = (w / w.norm(dim=2, keepdim=True)).cuda()
    ex, ey = torch.linspace(-3.5, 3.5, bx + 1), torch.linspace(-3.5, 3.5, by + 1)
    (gx, sx), (gy, sy) = geom_rows(ex, 0.5, k), geom_rows(ey, 0.5, k)
    geom = torch.stack([gx, gy], dim=1).cuda()
    prev = ops.KDE2D_USE_TENSOR_CORES
    try:
        ops.KDE2D_USE_TENSOR_CORES = True
        tc, acc = ops.kde2d_sums(x, w, geom, 0.5, bx, by)
        tc2, _ = ops.kde2d_sums(x, w, geom, 0.5, bx, by)
        ops.KDE2D_USE_TENSOR_CORES = False           # MFB_FLAG_NO_TENSOR_CORES on the call
        fx, _ = ops.kde2d_sums(x, w, geom, 0.5, bx, by)
    finally:
        ops.KDE2D_USE_TENSOR_CORES = prev
    assert torch.equal(tc, tc2)
    assert not torch.equal(tc, fx)                   # the two paths really are different kernels
    cx, cy = (0.5 * (ex[1:] + ex[:-1])).double().cuda(), (0.5 * (ey[1:] + ey[:-1])).double().cuda()
    xd = x.double()
    ref = torch.stack([
        torch.exp(-0.5 * (((xd @ w[i, 0].double())[:, None] - cx[None]) / float(sx)) ** 2).T
        @ torch.exp(-0.5 * (((xd @ w[i, 1].double())[:, None] - cy[None]) / float(sy)) ** 2) for i in range(k)])
    peak = float(ref.max())
    tc, fx = tc.double(), fx.double()
    for lo, bound in [(1e-3, 1e-4), (1e-9, 3e-4), (1e-12, 1e-3)]:
        m = ref > lo * peak
        err_tc = float(((tc - ref).abs() / ref)[m].max())
        err_fx = float(((fx - ref).abs() / ref)[m].max())
        assert err_tc < bound and err_fx < bound, (lo, err_tc, err_fx)
    planes = acc.double()
    rebuilt = (planes[0] + planes[1] / 2 ** 22) / 2 ** 22
    assert float((rebuilt - tc).abs().max()) <= 1e-6 * float(tc.max())
