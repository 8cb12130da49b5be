"""CPU checks of MetropolisHastingsSampler: the numpy replay of the chains' Philox layout that the GPU tests compare the
kernels against, the sampler's refusals (before anything is launched), and the C ABI's argument checks."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy import stats

import mentflow_b200 as mf
from mentflow_b200 import _lib, ops
from mfb_testutil import philox4x32_10

_M32 = np.uint64(0xFFFFFFFF)


def mh_blocks(d):
    """Philox blocks per step: ceil(d / 2) Box-Muller pairs and one acceptance word."""
    return (2 * ((d + 1) // 2) + 1 + 3) // 4


def mh_words(chains, t, seed, d):
    """(n, 4 * mh_blocks(d)) uint32 words of step t of the chains: block b is Philox4x32-10 of the counter
    (c mod 2^32, c div 2^32, t, b) under the key (seed mod 2^32, seed div 2^32)."""
    c = np.asarray(chains, dtype=np.uint64)
    key = np.array([int(seed) & 0xFFFFFFFF, (int(seed) >> 32) & 0xFFFFFFFF], dtype=np.uint64)
    out = []
    for b in range(mh_blocks(d)):
        ctr = np.stack([c & _M32, c >> np.uint64(32), np.full_like(c, t), np.full_like(c, b)], axis=-1)
        out.append(philox4x32_10(ctr, key))
    return np.concatenate(out, axis=-1)


def mh_draw64(chains, t, seed, d):
    """(xi (n, d), u (n,)) of step t in float64: Box-Muller on word pairs, u1 in (0, 1], u2 in [0, 1)."""
    w = mh_words(chains, t, seed, d).astype(np.float64)
    top = np.floor(w / 256.0)
    pairs = (d + 1) // 2
    xi = np.empty((w.shape[0], 2 * pairs))
    for j in range(pairs):
        u1, u2 = (top[:, 2 * j] + 1.0) * 2.0 ** -24, top[:, 2 * j + 1] * 2.0 ** -24
        r = np.sqrt(-2.0 * np.log(u1))
        xi[:, 2 * j], xi[:, 2 * j + 1] = r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)
    return xi[:, :d], (top[:, 2 * pairs] + 1.0) * 2.0 ** -24


def test_words_are_philox_of_chain_step_and_block_past_2_32_chains():
    seed, chains = 0x0123456789ABCDEF, np.array([0, 2**32 - 1, 2**32, 2**40 + 7, 2**64 - 1], dtype=np.uint64)
    for d in (1, 2, 3, 6, 8):
        w = mh_words(chains, 9, seed, d)
        assert w.shape == (5, 4 * mh_blocks(d))
        for n, c in enumerate(chains.tolist()):
            for b in range(mh_blocks(d)):
                want = philox4x32_10((c & 0xFFFFFFFF, c >> 32, 9, b), (seed & 0xFFFFFFFF, seed >> 32))
                assert np.array_equal(w[n, 4 * b:4 * b + 4], want)
    assert [mh_blocks(d) for d in range(1, 9)] == [1, 1, 2, 2, 2, 2, 3, 3]
    # every chain, step and block gets its own words
    a, b = mh_words(np.arange(4, dtype=np.uint64), 1, 5, 8), mh_words(np.arange(4, dtype=np.uint64), 2, 5, 8)
    assert len({int(v) for v in np.concatenate([a.ravel(), b.ravel()])}) == a.size + b.size


def test_box_muller_ends_are_finite_and_uniforms_in_the_half_open_interval():
    chains = np.arange(200_000, dtype=np.uint64)
    xi, u = mh_draw64(chains, 3, 11, 5)
    assert np.isfinite(xi).all() and (u > 0).all() and (u <= 1).all()
    assert float(np.abs(xi).max()) <= math.sqrt(2 * 24 * math.log(2)) + 1e-12   # u1 >= 2^-24
    # the documented layout is a standard normal generator: moments and KS per coordinate, u uniform
    n = xi.shape[0]
    assert np.abs(xi.mean(axis=0)).max() < 5 / math.sqrt(n)
    assert np.abs(np.cov(xi.T) - np.eye(5)).max() < 6 * math.sqrt(2 / n)
    for i in range(5):
        assert stats.kstest(xi[:, i], "norm").pvalue > 1e-4
    assert stats.kstest(u, "uniform").pvalue > 1e-4


@pytest.mark.parametrize("kw,match", [
    (dict(ndim=0, burnin=0), "ndim"), (dict(ndim=9, burnin=0), "ndim"),
    (dict(ndim=2, burnin=-1), "burnin"), (dict(ndim=2, burnin=0, steps=0), "steps"),
    (dict(ndim=2, burnin=0, thin=0), "thin"), (dict(ndim=2, burnin=2**31, steps=3, thin=2**31), "2\\^32"),
    (dict(ndim=2, burnin=0, proposal_cov=torch.eye(3)), "shape"),
    (dict(ndim=2, burnin=0, proposal_cov=torch.ones(2)), "shape"),
    (dict(ndim=2, burnin=0, proposal_cov=torch.tensor([[1.0, 2.0], [2.0, 1.0]])), "positive definite"),
    (dict(ndim=2, burnin=0, proposal_cov=torch.tensor([[1.0, 0.1], [0.0, 1.0]])), "symmetric"),
    (dict(ndim=2, burnin=0, proposal_cov=torch.tensor([[float("nan"), 0.0], [0.0, 1.0]])), "positive definite"),
    (dict(ndim=2, burnin=0, start=torch.zeros(3)), "start"),
    (dict(ndim=2, burnin=0, start_scale=float("inf")), "start_scale"),
])
def test_sampler_refuses_bad_arguments(kw, match):
    with pytest.raises(ValueError, match=match):
        mf.sample.MetropolisHastingsSampler(**kw)


def test_default_proposal_and_a_given_one():
    s = mf.sample.MetropolisHastingsSampler(4, burnin=3, steps=5, thin=2)
    assert torch.allclose(s.chol.double() @ s.chol.double().T, torch.eye(4, dtype=torch.float64) * 2.38 ** 2 / 4)
    assert s.proposals() == 3 + 4 * 2 and s.supports_offset and s.acceptance_rate is None
    cov = torch.tensor([[2.0, 0.5], [0.5, 1.0]], dtype=torch.float64)
    s = mf.sample.MetropolisHastingsSampler(2, burnin=0, proposal_cov=cov)
    assert s.chol.dtype == torch.float32 and float(s.chol[0, 1]) == 0.0
    assert torch.allclose(s.chol.double() @ s.chol.double().T, cov, rtol=1e-6)
    assert s.to("cuda:1") is s and s.device == "cuda:1"


def test_size_zero_returns_no_rows_without_calling_the_density_and_still_draws_a_seed():
    calls = []
    s = mf.sample.MetropolisHastingsSampler(3, burnin=1, device="cpu")
    torch.manual_seed(5)
    x = s(lambda p: calls.append(p), 0)
    after = torch.randint(0, 2 ** 62, (1,))
    torch.manual_seed(5)
    torch.randint(0, 2 ** 62, (1,))
    assert x.shape == (0, 3) and not calls and torch.equal(after, torch.randint(0, 2 ** 62, (1,)))


def test_cpu_tensors_are_refused():
    s = mf.sample.MetropolisHastingsSampler(2, burnin=1, device="cpu")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        s(lambda p: torch.ones(p.shape[0]), 10, seed=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.ment_mh(None, None, 0.0, 0.0, 2, 0, 4, torch.eye(2), 0, 1, 1, 1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.mh_propose(None, 4, 2, 0, None, 0, 1, "cpu")


def test_c_abi_checks_arguments_before_any_launch():
    """Every refusal below returns MFB_E_BADARG from the host-side checks (the pointers are never dereferenced)."""
    lib = _lib.load()
    p = ctypes.c_void_p(256)

    def mh(d=2, k=1, b=4, chain0=0, n=4, start=None, scale=1.0, chol=p, burnin=0, steps=1, thin=1, out=p, acc=p):
        return lib.mfb_ment_mh(d, p, p, p, k, b, None, None, None, None, None, 0, 0, 0, None, 0.0, 0.0, chain0, n,
                               start, scale, chol, burnin, steps, thin, 1, out, acc, None)

    bad = [dict(d=0), dict(d=9), dict(burnin=-1), dict(steps=0), dict(thin=0), dict(burnin=2**32),
           dict(burnin=1, steps=2, thin=2**32 - 1), dict(n=-1), dict(chain0=2**64 - 2, n=4), dict(chol=None),
           dict(out=None), dict(acc=None), dict(scale=float("nan")), dict(b=1), dict(k=-1)]
    for kw in bad:
        assert mh(**kw) == -1, kw
    assert mh(n=0) == 0                                 # nothing to run: no launch
    assert lib.mfb_mh_propose(None, 4, 2, 0, None, 1.0, None, 1, 1, p, None) == -1          # t >= 1 needs x, chol
    assert lib.mfb_mh_propose(None, 4, 2, 0, None, 1.0, None, 2**32, 1, p, None) == -1
    assert lib.mfb_mh_propose(None, 4, 9, 0, None, 1.0, None, 0, 1, p, None) == -1
    assert lib.mfb_mh_propose(None, 0, 2, 0, None, 1.0, None, 0, 1, p, None) == 0
    assert lib.mfb_mh_accept(p, p, p, p, 4, 2, 0, 0, 1, p, None) == -1                     # t = 0 has no decision
    assert lib.mfb_mh_accept(p, p, p, p, 4, 2, 0, 1, 1, None, None) == -1
    assert lib.mfb_mh_accept(p, p, p, p, 0, 2, 0, 1, 1, p, None) == 0
