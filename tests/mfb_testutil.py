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


# ------------------------------------------------------------------------------------ flow gradients
def nsf_case(d, n, scale, hidden_layers=3, transforms=5, bins=20, seed=0, wide=False):
    """A seeded flow and its inputs: (NSFGenerator on the CPU with every parameter x ``scale``, its float64 oracle,
    z (n, d), and the upstream gradients a = dL/dx (n, d), b = dL/dlog q (n,) of L = sum(x a) + sum(log q b))."""
    import mentflow_b200 as mf
    torch.manual_seed(seed)
    gen = mf.generate.NSFGenerator(d, hidden_layers=hidden_layers, transforms=transforms, bins=bins)
    with torch.no_grad():
        for p in gen.parameters():
            p.mul_(scale)
    ref = oracle_from_generator(gen)      # before the draws below: building it advances the generator
    z = torch.randn(n, d)
    if wide:      # the whole spline box and beyond: first / last bins, identity outside [-5, 5]
        z = (torch.rand(n, d) - 0.5) * 13.0
    a, b = torch.randn(n, d), torch.randn(n)
    return gen, ref, z, a, b


def nsf_loss(x, lq, a, b, loss):
    """"both": sum(x a) + sum(log q b); "x": sum(x a) (log q not computed); "logq": sum(log q b) (dL/dx = 0)."""
    if loss == "x":
        return (x * a).sum()
    if loss == "logq":
        return (lq * b).sum()
    return (x * a).sum() + (lq * b).sum()


def nsf_kernel_grads(gen, z, a, b, loss="both"):
    """dL/dz and dL/dtheta of ``nsf_loss`` through the CUDA flow ``gen``: {"z", "w_in", "b_in", "w_hid", "b_hid",
    "w_out", "b_out"}, each as the kernels left it (the x-only loss runs gen.forward, which computes no log q)."""
    for p in gen.parameters():
        p.grad = None
    zc = z.cuda().requires_grad_(True)
    if loss == "x":
        x, lq = gen.forward(zc), None
    else:
        x, lq = gen.forward_and_log_prob(zc)
    nsf_loss(x, lq, a.cuda(), b.cuda(), loss).backward()
    out = {"z": zc.grad}
    for name in ("w_in", "b_in", "w_hid", "b_hid", "w_out", "b_out"):
        out[name] = getattr(gen, name).grad
    return out


def nsf_named_grads(g, hidden_layers, transforms):
    """``nsf_kernel_grads`` split per layer under the names of ``nsf_oracle_grads``."""
    out = {"z": g["z"]}
    for t in range(transforms):
        out[f"w_in{t}"], out[f"b_in{t}"] = g["w_in"][t], g["b_in"][t]
        for l in range(hidden_layers - 1):
            out[f"w_hid{t}.{l}"], out[f"b_hid{t}.{l}"] = g["w_hid"][t, l], g["b_hid"][t, l]
        out[f"w_out{t}"], out[f"b_out{t}"] = g["w_out"][t], g["b_out"][t]
    return out


def nsf_oracle_grads(flow, z, a, b, loss="both"):
    """Autograd of ``nsf_loss`` through the oracle ``flow`` in its own dtype: {"z", "w_in{t}", "b_in{t}",
    "w_hid{t}.{l}", "b_hid{t}.{l}", "w_out{t}", "b_out{t}"} (float64), masked weights' entries zeroed; and
    {"w_in{t}", "w_hid{t}.{l}", "w_out{t}"}: the masks."""
    dtype = next(flow.parameters()).dtype
    for q in flow.parameters():
        q.grad = None
    zz = z.to(dtype).clone().requires_grad_(True)
    x, lq = flow.forward_and_log_prob(zz)
    nsf_loss(x, lq, a.to(dtype), b.to(dtype), loss).backward()
    out, masks = {"z": zz.grad.double()}, {}
    for t in range(len(flow.layers)):
        lin = [m for m in flow.layers[t].hyper if hasattr(m, "weight")]
        names = [f"in{t}"] + [f"hid{t}.{l}" for l in range(len(lin) - 2)] + [f"out{t}"]
        for name, m in zip(names, lin):
            gw = torch.zeros_like(m.weight) if m.weight.grad is None else m.weight.grad
            gb = torch.zeros_like(m.bias) if m.bias.grad is None else m.bias.grad
            out["w_" + name], out["b_" + name] = (gw * m.mask).double(), gb.double()
            masks["w_" + name] = m.mask.detach().bool()
    return out, masks


def nsf_relu_kink_particles(flow, z, margin=1e-6):
    """Boolean mask of the particles whose forward pass through the oracle ``flow`` puts some hidden pre-activation
    within ``margin`` of the ReLU kink, relative to the sum of the magnitudes of its terms (|b| + sum |w h|).  An fp32
    evaluation may take the other branch there: the particle's whole upstream gradient then moves between the unit's
    parameter gradients, while its dL/dz barely changes."""
    near, hooks = torch.zeros(z.shape[0], dtype=torch.bool), []

    def check(m, inputs, out):
        nonlocal near
        h = inputs[0]
        size = h.abs() @ (m.weight * m.mask).abs().T + m.bias.abs()
        near = near | (out.abs() <= margin * size).any(dim=1)

    for layer in flow.layers:
        lin = [m for m in layer.hyper if hasattr(m, "weight")]
        hooks += [m.register_forward_hook(check) for m in lin[:-1]]      # the output layer feeds no ReLU
    try:
        with torch.no_grad():
            flow.forward_and_log_prob(z.to(next(flow.parameters()).dtype))
    finally:
        for hk in hooks:
            hk.remove()
    return near


def grads_case(d, n, scale, hidden_layers=3, transforms=5, bins=20, seed=0, keep=None, wide=False, loss="both",
               upstream=None):
    """{name: (CUDA flow's gradient, float64 oracle autograd's)} for the seeded ``nsf_case``.  ``upstream(a, b)``
    returns the upstream gradients to use instead of a, b; ``keep``: boolean mask of the particles to keep."""
    gen, ref, z, a, b = nsf_case(d, n, scale, hidden_layers, transforms, bins, seed, wide)
    if upstream is not None:
        a, b = upstream(a, b)
    if keep is not None:
        z, a, b = z[keep], a[keep], b[keep]
    got = nsf_named_grads(nsf_kernel_grads(gen.to("cuda"), z, a, b, loss), hidden_layers, transforms)
    want, _ = nsf_oracle_grads(ref, z, a, b, loss)
    return {k: (got[k], want[k]) for k in want}


def grad_rel(got, want):
    """|got - want| relative to the largest entry of ``want`` (the metric of every flow-gradient test)."""
    want = want.double().cpu()
    return (got.double().cpu() - want).abs() / want.abs().max().clamp_min(1e-30)


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
