"""NNGenerator on the GPU (ops.nn_forward, csrc/nn.cu) against a float64 nn.Sequential on the same fp32 weights and
noise: forward over every compiled shape, tanh alone, gradients, reproducibility, the base draw and MENTFlow."""
import math

import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200 import ops, workloads
from mentflow_b200.generate import NNGenerator

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda")
SHAPES = sorted({(d, 6) for d in range(1, 9)} | {(6, d) for d in range(1, 9)} | {(1, 1), (8, 8)})
LAYERS = (1, 2, 3, 5, 8)
SIZES = (1, 127, 128, 129, 5_000, 100_003)


def params64(gen):
    return [p.detach().double() for p in (gen.w_in, gen.b_in, gen.w_hid, gen.b_hid, gen.w_out, gen.b_out)]


def oracle(z, w_in, b_in, w_hid, b_hid, w_out, b_out):
    """float64 nn.Sequential(Linear, Tanh, ..., Linear) on the given (float64) parameters."""
    h = torch.tanh(z @ w_in.T + b_in)
    for l in range(w_hid.shape[0]):
        h = torch.tanh(h @ w_hid[l].T + b_hid[l])
    return h @ w_out.T + b_out


def make(din, dout, layers, seed=0, scale=1.0):
    torch.manual_seed(seed)
    gen = NNGenerator(din, dout, layers, 64, device=DEV)
    if scale != 1.0:
        with torch.no_grad():
            for p in gen.parameters():
                p.mul_(scale)
    return gen


@pytest.mark.parametrize("layers", LAYERS)
@pytest.mark.parametrize("din,dout", SHAPES)
def test_forward_matches_float64(din, dout, layers):
    for scale in (1.0, 3.0):                  # default init, and saturating tanh
        gen = make(din, dout, layers, seed=din * 100 + dout * 10 + layers, scale=scale)
        z = torch.randn(max(SIZES), din, device=DEV)
        for n in SIZES:
            with torch.no_grad():
                x = gen(z[:n])
            x64 = oracle(z[:n].double(), *params64(gen))
            err = (x.double() - x64).abs() / x64.abs().clamp_min(1.0)
            assert x.shape == (n, dout)
            assert float(err.max()) <= 1e-4, (din, dout, layers, scale, n, float(err.max()))


def test_tanh_alone_is_accurate():
    """x = tanh(z) through the whole kernel: one input, one output, one layer, W_in[:, 0] = 1, W_out = e_0."""
    gen = make(1, 1, 1)
    with torch.no_grad():
        gen.w_in.fill_(1.0)
        gen.b_in.zero_()
        gen.w_out.zero_()
        gen.w_out[0, 0] = 1.0
        gen.b_out.zero_()
    dense = torch.linspace(-10.0, 10.0, 2_000_001, dtype=torch.float32)
    tiny = torch.tensor([0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.1754942e-38, 1.17549435e-38, 1e-30, -1e-20,
                         1e-10, 1e-6, -1e-4, 1e-3, 0.01], dtype=torch.float32)
    z = torch.cat([dense, tiny, -tiny]).to(DEV)[:, None]
    with torch.no_grad():
        x = gen(z)[:, 0]
    ref = torch.tanh(z[:, 0].double())
    rel = (x.double() - ref).abs() / ref.abs().clamp_min(1e-300)
    rel = torch.where(ref == 0, (x.double() - ref).abs(), rel)
    assert float(rel.max()) <= 1e-6, float(rel.max())


def linear_functional(gen, z, c):
    return (gen(z) * c).sum()


GRAD_CASES = [(6, 6, 1), (6, 6, 3), (6, 6, 4), (6, 6, 5), (6, 6, 8), (2, 2, 3), (1, 8, 2), (8, 1, 8), (3, 5, 6)]


@pytest.mark.parametrize("din,dout,layers", GRAD_CASES)
def test_gradients_match_float64_autograd(din, dout, layers):
    n = 100_003
    gen = make(din, dout, layers, seed=layers)
    torch.manual_seed(7)
    z = torch.randn(n, din, device=DEV, requires_grad=True)
    c = torch.randn(n, dout, device=DEV)
    linear_functional(gen, z, c).backward()
    got = [z.grad] + [p.grad for p in gen.parameters()]
    p64 = [p.requires_grad_(True) for p in params64(gen)]
    z64 = z.detach().double().requires_grad_(True)
    (oracle(z64, *p64) * c.double()).sum().backward()
    want = [z64.grad] + [p.grad for p in p64]
    for name, g, w in zip(("z", "w_in", "b_in", "w_hid", "b_hid", "w_out", "b_out"), got, want):
        if name in ("w_hid", "b_hid") and layers == 1:   # empty: nothing to compare
            continue
        assert g.shape == w.shape, name
        scale = float(w.abs().max())
        assert float((g.double() - w).abs().max()) <= 1e-4 * scale, (name, scale)


def kl_model(gen, ndim, estimator, n_truth=50_000):
    wl = workloads.rotations_2d(7, 64, 3.5)
    tfs = [mf.simulate.LinearTransform(m.to(DEV)) for m in wl["matrices"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to(DEV)
    diags = [[diag] for _ in tfs]
    truth = workloads.gaussian_mixture(n_truth, ndim=ndim, seed=1, device=DEV)
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    return mf.MENTFlow(transforms=tfs, diagnostics=diags, measurements=meas, generator=gen, prior=None,
                       entropy_estimator=estimator, discrepancy_function=mf.loss.kl_divergence, penalty_parameter=50.0)


def test_gradients_of_the_kl_loss_match_float64_autograd():
    n = 100_003
    gen = make(2, 2, 3, seed=11)
    model = kl_model(gen, 2, mf.entropy.CovarianceEntropyEstimator())
    torch.manual_seed(5)
    z = torch.randn(n, 2, device=DEV, requires_grad=True)
    L, _, _ = model.loss_from_particles(gen(z), None)
    L.backward()
    got = [z.grad] + [p.grad for p in gen.parameters()]
    # the same loss through the float64 network: the particles' gradient comes from the library's loss kernels,
    # the chain through the network from float64 autograd
    p64 = [p.requires_grad_(True) for p in params64(gen)]
    z64 = z.detach().double().requires_grad_(True)
    x64 = oracle(z64, *p64)
    xf = x64.detach().float().requires_grad_(True)
    model.loss_from_particles(xf, None)[0].backward()
    (x64 * xf.grad.double()).sum().backward()
    want = [z64.grad] + [p.grad for p in p64]
    for name, g, w in zip(("z", "w_in", "b_in", "w_hid", "b_hid", "w_out", "b_out"), got, want):
        scale = float(w.abs().max())
        assert float((g.double() - w).abs().max()) <= 1e-4 * scale, (name, scale)


@pytest.mark.parametrize("layers", (3, 8))
def test_forward_and_backward_are_bitwise_reproducible(layers):
    gen = make(6, 6, layers)
    z = torch.randn(100_003, 6, device=DEV, requires_grad=True)
    c = torch.randn(100_003, 6, device=DEV)
    runs = []
    for _ in range(3):
        gen.zero_grad(set_to_none=True)
        z.grad = None
        x = gen(z)
        (x * c).sum().backward()
        runs.append([x.detach().clone(), z.grad.clone()] + [p.grad.clone() for p in gen.parameters()])
    for other in runs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(runs[0], other))


def test_no_input_gradient_is_written_unless_asked():
    gen = make(6, 6, 3)
    z = torch.randn(1000, 6, device=DEV)
    (gen(z) ** 2).sum().backward()
    assert z.grad is None and gen.w_in.grad is not None


def test_base_draw_is_torch_randn_bitwise():
    gen = make(5, 3, 2)
    torch.manual_seed(123)
    z = gen.sample_base(10_001)
    after = torch.randn(7, device=DEV)
    torch.manual_seed(123)
    z_ref = torch.randn((10_001, 5), device=DEV)
    after_ref = torch.randn(7, device=DEV)
    assert z.shape == (10_001, 5) and torch.equal(z, z_ref) and torch.equal(after, after_ref)
    torch.manual_seed(9)
    x, logq = gen.sample_and_log_prob(4096)
    assert logq is None and x.shape == (4096, 3)
    torch.manual_seed(9)
    with torch.no_grad():
        assert torch.equal(x.detach(), gen(torch.randn((4096, 5), device=DEV)))


@pytest.mark.parametrize("estimator", ["covariance", "knn"])
def test_mentflow_loss_equals_the_loss_of_the_oracle_particles(estimator):
    n = 25_000
    gen = make(2, 2, 3, seed=4)
    est = mf.entropy.CovarianceEntropyEstimator() if estimator == "covariance" else mf.entropy.KNNEntropyEstimator()
    model = kl_model(gen, 2, est)
    torch.manual_seed(21)
    with torch.no_grad():
        L, H, D = model.loss(n)
    torch.manual_seed(21)
    z = torch.randn((n, 2), device=DEV)
    with torch.no_grad():
        x = oracle(z.double(), *params64(gen)).float()
        L64, _, _ = model.loss_from_particles(x, None)
    assert math.isfinite(float(L))
    assert abs(float(L) - float(L64)) <= 1e-5 * abs(float(L64)), (float(L), float(L64))


def test_monte_carlo_entropy_is_refused_with_a_pointer_to_the_particle_estimators():
    gen = make(2, 2, 3)
    prior = mf.prior.Gaussian(ndim=2, scale=3.0)
    model = kl_model(gen, 2, mf.entropy.MonteCarloEntropyEstimator(prior=prior))
    with pytest.raises(ValueError, match="CovarianceEntropyEstimator"):
        model.loss(1000)


def test_graphed_loss_replay_equals_eager():
    from mentflow_b200.graphs import GraphedLoss
    gen = make(2, 2, 3, seed=2)
    model = kl_model(gen, 2, mf.entropy.CovarianceEntropyEstimator())
    n = 25_000
    g = GraphedLoss(model, n)
    z = torch.randn(n, 2)

    def eager(zz):
        with torch.no_grad():
            x, lq = gen.forward_and_log_prob(zz.to(DEV))
            return model.loss_from_particles(x, lq)

    for source in (z, z.pin_memory()):
        L, H, D = g(source)
        Le, He, De = eager(z)
        assert torch.equal(L, Le) and torch.equal(H, He) and torch.equal(torch.stack(D), torch.stack(De))
    torch.manual_seed(3)
    L = g(None)[0].clone()
    torch.manual_seed(3)
    assert torch.equal(L, eager(torch.randn((n, 2), device=DEV))[0])


def test_graphed_train_step_reduces_the_kl():
    """C1-sized problem (2-D, 7 rotations, 25,000 particles) with fused capturable AdamW: the mean KL falls."""
    from mentflow_b200.graphs import GraphedTrainStep
    gen = make(2, 2, 3, seed=0)
    model = kl_model(gen, 2, mf.entropy.CovarianceEntropyEstimator())
    opt = torch.optim.AdamW(model.parameters(), lr=2e-3, weight_decay=0.0, capturable=True, fused=True)
    step = GraphedTrainStep(model, opt, 25_000)
    first = float(torch.stack(step()[2]).mean())
    for _ in range(50):
        L, H, D = step()
    last = float(torch.stack(D).mean())
    assert bool(step.finite) and last < first, (first, last)
    assert all(torch.isfinite(p).all() for p in model.parameters())
