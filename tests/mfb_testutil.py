"""Shared helpers for the test-suite (imported as a top-level module; tests/ has no __init__)."""
import numpy as np
import torch


def t32(a):
    return torch.from_numpy(np.asarray(a)).to(torch.float32)


def cuda(a):
    return t32(a).cuda()


def oracle_from_generator(gen, dtype=torch.float64):
    """NSFOracle carrying the weights of a mentflow_b200 NSFGenerator (via zuko-style names)."""
    from oracle.zuko_nsf import NSFOracle
    flow = NSFOracle(gen.features, gen.hidden_units, gen.hidden_layers, gen.transforms, gen.bins,
                     passes=getattr(gen, "passes", None))
    sd = gen.state_dict()
    new = {}
    for k, v in flow.state_dict().items():
        # layers.{t}.hyper.{i}.{weight,bias,mask} / layers.{t}.order
        parts = k.split(".")
        src = "_flow.transform.transforms." + ".".join(parts[1:])
        new[k] = sd[src].detach().cpu().to(v.dtype)
    flow.load_state_dict(new)
    return flow.to(dtype)


def generator_from_golden(g, device="cpu"):
    """NSFGenerator loaded with the weights stored in tests/golden/nsf_*.npz."""
    import mentflow_b200 as mf
    d = g["z"].shape[1]
    gen = mf.generate.NSFGenerator(d)
    sd = {}
    for k, v in g.items():
        if k.startswith("sd:") and (k.endswith("weight") or k.endswith("bias")):
            sd["_flow.transform.transforms." + k[len("sd:layers."):]] = torch.from_numpy(v).float()
    gen.load_state_dict(sd)
    return gen.to(device)


def rel_err(a, b):
    """max |a-b| / max(1, |b|) elementwise (SURVEY 8c metric for x and log q)."""
    a, b = a.double().cpu(), b.double().cpu()
    return float(((a - b).abs() / b.abs().clamp_min(1.0)).max())


def profile_err(a, b):
    """max over profiles of max|a-b| / max|b| (SURVEY 8c metric for KDE profiles)."""
    a, b = a.double().cpu(), b.double().cpu()
    a, b = a.reshape(a.shape[0], -1), b.reshape(b.shape[0], -1)
    return float(((a - b).abs().max(dim=1).values / b.abs().max(dim=1).values).max())


def geom_rows(edges, bandwidth, k):
    """k identical C-ABI geometry records [c0, spacing, sigma, delta, 0...] for fp32 edges."""
    e = edges.float()
    c = 0.5 * (e[:-1] + e[1:])
    delta = float(c[1] - c[0])
    spacing = float((c[-1].double() - c[0].double()) / (c.numel() - 1))
    sigma = float(bandwidth * (e[1] - e[0]))
    return torch.tensor([[float(c[0]), spacing, sigma, delta, 0, 0, 0, 0]] * k, dtype=torch.float32), sigma


def err_stats(a, b):
    """elementwise |a-b| / max(1,|b|): (max, 99.9th percentile)."""
    e = ((a.double().cpu() - b.double().cpu()).abs() / b.double().cpu().abs().clamp_min(1.0)).flatten()
    k = max(1, int(e.numel() * 0.999))
    return float(e.max()), float(e.kthvalue(k).values)


# ------------------------------------------------------------------------------------ float64 classical-MENT oracle
def _cpu64(t):
    """float64 CPU copy of a transfer map."""
    from mentflow_b200.simulate.transform import CompositeTransform, LinearTransform, MultipoleTransform
    if isinstance(t, LinearTransform):
        return LinearTransform(t.matrix.detach().to("cpu", torch.float64))
    if isinstance(t, CompositeTransform):
        return CompositeTransform(*[_cpu64(s) for s in t.transforms])
    return MultipoleTransform(order=t.order, strength=t.strength, skew=t.skew)


def _h(diag, table, u):
    """Lagrange function of ``diag`` at the transformed points u (float64), as the reference's interpolator."""
    import mentflow_b200 as mf
    from oracle import hotpath as hp
    if isinstance(diag, mf.diagnostics.Histogram2D):
        cx, cy = (hp.centres(e.cpu()) for e in (diag.edges_x, diag.edges_y))
        return hp.lagrange_interp_2d(table.cpu(), cx, cy, u[:, list(diag.axis)])
    return hp.lagrange_interp(table.cpu(), hp.centres(diag.edges.cpu()), u[:, diag.axis])


def oracle_prob(model, x):
    """hp.ment_prob with transform.forward in float64 in place of the matrix; Gaussian or Uniform prior."""
    import math

    import mentflow_b200 as mf
    from oracle import hotpath as hp
    x = x.detach().cpu().double()
    prob = torch.ones(x.shape[0], dtype=torch.float32)
    for i, t in enumerate(model.transforms):
        u = _cpu64(t)(x)
        for j, diag in enumerate(model.diagnostics[i]):
            h = _h(diag, model.lagrange_functions[i][j].values, u)
            prob = prob * torch.clamp(h.type(torch.float32), 0.0, 1.0e10)
    if isinstance(model.prior, mf.prior.Uniform):
        return prob * torch.exp(torch.full_like(prob, -math.log(model.prior.volume)))
    return prob * torch.exp(hp.gaussian_log_prob(x, float(model.prior.scale)).float())


def oracle_integrate(model, i, j):
    """Normalised integrate-mode prediction: sum over the integration grid of rho(transform.inverse(points))."""
    import mentflow_b200 as mf
    from oracle import hotpath as hp
    diag = model.diagnostics[i][j]
    limits, shape = model.integration_limits[i][j], model.integration_shape[i][j]
    grid = [torch.linspace(float(lo), float(hi), int(n), dtype=torch.float64) for (lo, hi), n in zip(limits, shape)]
    if isinstance(diag, mf.diagnostics.Histogram2D):
        meas = [hp.centres(diag.edges_x.cpu()).double(), hp.centres(diag.edges_y.cpu()).double()]
        axes = list(diag.axis)
    else:
        meas = [hp.centres(diag.edges.cpu()).double()]
        axes = [diag.axis]
    d = model.ndim
    others = [a for a in range(d) if a not in axes]
    mesh = torch.meshgrid(*meas, *grid, indexing="ij")
    u = torch.zeros(mesh[0].numel(), d, dtype=torch.float64)
    for a, m in zip(axes + others, mesh):
        u[:, a] = m.reshape(-1)
    x = _cpu64(model.transforms[i]).inverse(u)
    rho = oracle_prob(model, x).double().reshape(*[m.numel() for m in meas], -1).sum(dim=-1)
    if isinstance(diag, mf.diagnostics.Histogram2D):
        vol = float(diag.edges_x[1] - diag.edges_x[0]) * float(diag.edges_y[1] - diag.edges_y[0])
    else:
        vol = float(diag.edges[1] - diag.edges[0])
    return (rho / rho.sum() / vol).float()


def oracle_sweeps(model, n, lr=1.0, thresh=1.0e-10):
    """``n`` Gauss-Seidel sweeps of integrate mode on the oracle (model's tables are read, not changed)."""
    from oracle import hotpath as hp
    saved = [[lf.values.clone() for lf in row] for row in model.lagrange_functions]
    out = None
    try:
        for _ in range(n):
            for i in range(len(model.transforms)):
                for j in range(len(model.diagnostics[i])):
                    pred = oracle_integrate(model, i, j)
                    lf = model.lagrange_functions[i][j]
                    meas = model.measurements[i][j].cpu()
                    new = hp.gauss_seidel_table(lf.values.cpu(), meas, pred, lr, thresh)
                    lf.set_values(new.to(lf.values.device))
        out = [[lf.values.cpu().clone() for lf in row] for row in model.lagrange_functions]
    finally:
        for row, vals in zip(model.lagrange_functions, saved):
            for lf, v in zip(row, vals):
                lf.set_values(v)
    return out


def positive_tables(model, seed):
    """Positive random tables, zero on the outermost centres so that h is continuous (a point whose fp32 and float64
    projections straddle the last centre would otherwise see a jump)."""
    gen = torch.Generator().manual_seed(seed)
    for row in model.lagrange_functions:
        for lf in row:
            v = torch.rand(lf.values.shape, generator=gen) + 0.2
            if v.ndim == 1:
                v[0] = v[-1] = 0.0
            else:
                v[0], v[-1], v[:, 0], v[:, -1] = 0.0, 0.0, 0.0, 0.0
            lf.set_values(v.cuda())


def check_density(model, x, want_x):
    """prob at explicit points, prob_on_grid and prob at the materialised grid points against the float64 oracle.
    The kernels project in fp32: where a factor sits near the zero end of its table its relative error is that of
    the projection over the distance to the end (a fp32 emulation of the kernels' arithmetic reaches 7e-7 of the
    maximum there), hence an absolute tolerance of 2e-6 of the maximum at the explicit points as on the grid."""
    prob = model.prob(x.cuda()).cpu()
    assert int((want_x > 0).sum()) > 0.2 * want_x.numel()               # not vacuous
    assert torch.allclose(prob, want_x, rtol=1e-4, atol=2e-6 * float(want_x.max()))
    grid = model.prob_on_grid(model.sampler).cpu()
    pts = model.sampler.get_grid_points()
    refg = oracle_prob(model, pts)
    assert int((refg > 0).sum()) > 0.05 * refg.numel()
    # grid points come from the index (lo + i*step) instead of fp32 linspace centres: 1-ulp shifts
    assert torch.allclose(grid, refg, rtol=1e-4, atol=2e-6 * float(refg.max()))
    assert torch.allclose(model.prob(pts).cpu(), refg, rtol=1e-4, atol=2e-6 * float(refg.max()))


def integrate_check(model, slots):
    """simulate(i, j) against the oracle, then two Gauss-Seidel sweeps against the oracle's sweeps.  A screen's own
    pixels sit exactly on its bin centres: where the table is 0 next to a nonzero value, fp32 rounding of the pixel's
    own projection (a few 1e-7) turns h = 0 into slope x rounding, up to ~1e-5 of the maximum prediction.  Such entries
    stay 0 through the update (0 x anything), so the tables keep the tight tolerances."""
    for i, j in slots:
        pred = model.simulate(i, j).cpu()
        want = oracle_integrate(model, i, j)
        assert pred.shape == want.shape and int((want > 0).sum()) > 5
        assert torch.allclose(pred, want, rtol=1e-4, atol=1e-5 * float(want.max())), (i, j)
    want = oracle_sweeps(model, 2)
    model.gauss_seidel_update(lr=1.0, thresh=1.0e-10)
    model.gauss_seidel_step(lr=1.0, thresh=1.0e-10)
    for row_g, row_w in zip(model.lagrange_functions, want):
        for lf, w in zip(row_g, row_w):
            got = lf.values.cpu()
            assert torch.allclose(got, w, rtol=2e-4, atol=1e-6)
            assert torch.equal(got == 0, w == 0)


# ------------------------------------------------------------------------------------ the grid sampler's arithmetic
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Random123) in numpy uint64 arithmetic, as ment.cu's philox4x32.  ctr (..., 4), key (..., 2): uint32
    words, broadcast against each other; returns (..., 4) uint32."""
    ctr, key = np.asarray(ctr, dtype=np.uint64), np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (ctr[..., i] for i in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2      # < 2^64: exact
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def philox_ment(counter, stream, seed):
    """ment.cu philox4x32(counter, stream, seed): ctr = (counter lo, counter hi, stream, 0), key = (seed lo, seed hi)."""
    counter = np.asarray(counter, dtype=np.uint64)
    ctr = np.stack([counter & _M32, counter >> np.uint64(32), np.full_like(counter, stream), np.zeros_like(counter)], -1)
    seed = int(seed)
    return philox4x32_10(ctr, np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64))


def sampler_uniforms(seed, offset, size, d):
    """(uu, rnd) of cdf_sample_kernel for draws s < size: the 53-bit uniform of the cell choice and the 2 * d words
    rnd[2i] (position in the cell) / rnd[2i+1] (jitter) of axis i."""
    counter = np.uint64(offset) + np.arange(size, dtype=np.uint64)
    r0 = philox_ment(counter, 0, seed).astype(np.uint64)
    bits = (r0[:, 0] << np.uint64(21)) ^ (r0[:, 1] >> np.uint64(11))
    uu = (bits.astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)
    words = [r0[:, 2], r0[:, 3]]
    for b in range((2 * d + 1) // 4 + 1):
        words += list(philox_ment(counter, 1 + b, seed).astype(np.uint64).T)
    return uu, np.stack(words[:2 * d], axis=1).astype(np.uint32)


def u01(r):
    """ment.cu u01: the top 24 bits of r as a float32 in [0, 1)."""
    return ((np.asarray(r, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0))


def fmaf(a, b, c):
    """fp32 fma, correctly rounded: the product of two fp32 is exact in float64, TwoSum gives the float64 sum s and its
    exact error e, and s rounds to fp32 like s + e except on a tie of s, which the sign of e breaks."""
    p = np.asarray(a, np.float32).astype(np.float64) * np.asarray(b, np.float32).astype(np.float64)
    c = np.asarray(c, np.float32).astype(np.float64)
    p, c = np.broadcast_arrays(p, c)
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)
    f = s.astype(np.float32)
    d = s - f.astype(np.float64)                              # s - round(s)
    other = np.nextafter(f, np.where(d > 0, np.float32(np.inf), np.float32(-np.inf)))
    tie = (d != 0) & (np.abs(d) == np.abs(other.astype(np.float64) - f.astype(np.float64)) / 2)
    return np.where(tie & (e != 0) & (np.sign(e) == np.sign(d)), other, f)
