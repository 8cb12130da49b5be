"""Host-side folding of multipole chains for classical MENT (no GPU): the inverse terms of integrate mode against
CompositeTransform.inverse, the 2-D screen rows against transform.forward, and the maps MENT refuses."""
import itertools

import pytest
import torch
import torch.nn as nn

import mentflow_b200 as mf
from mentflow_b200.simulate.simulate import _multipole_chain, multipole_inverse_terms, multipole_terms
from mentflow_b200.simulate.transform import (CompositeTransform, LinearTransform, MultipoleTransform,
                                              ProjectionTransform)


def _matrix(d, gen):
    return torch.randn(d, d, dtype=torch.float64, generator=gen) * 0.4 + torch.eye(d, dtype=torch.float64)


def _chain(d, order, skew, with_pre, with_post, gen, strength=0.8):
    pre = _matrix(d, gen) if with_pre else None
    post = _matrix(d, gen) if with_post else None
    kick = MultipoleTransform(order=order, strength=strength, skew=skew)
    stages = ([LinearTransform(pre)] if with_pre else []) + [kick] + ([LinearTransform(post)] if with_post else [])
    return CompositeTransform(*stages), pre, kick, post


def _fold_inverse(u, lin, imp, order):
    d = u.shape[1]
    z = torch.complex(u @ imp[:d], u @ imp[d:2 * d]) ** (order - 1)
    return u @ lin.T + z.real[:, None] * imp[2 * d:3 * d] + z.imag[:, None] * imp[3 * d:4 * d]


@pytest.mark.parametrize("d,order,skew", list(itertools.product([2, 4, 6], [3, 4, 5], [False, True])))
def test_multipole_inverse_terms_match_composite_inverse(d, order, skew):
    gen = torch.Generator().manual_seed(100 * d + 10 * order + int(skew))
    for with_pre, with_post in itertools.product([False, True], repeat=2):
        t, pre, kick, post = _chain(d, order, skew, with_pre, with_post, gen)
        u = torch.randn(300, d, dtype=torch.float64, generator=gen) * 1.5
        want = t.inverse(u)
        lin, imp = multipole_inverse_terms(pre, kick, post, d, dtype=torch.float64)
        assert lin.shape == (d, d) and imp.shape == (4 * d + 2,) and float(imp[4 * d]) == order
        got = _fold_inverse(u, lin, imp, order)
        assert float((got - want).abs().max()) <= 1e-12 * float(want.abs().max()), (with_pre, with_post)
        # the chain MENT reads from the transform gives the same terms
        pre_c, kick_c, post_c = _multipole_chain(t)
        lin_c, imp_c = multipole_inverse_terms(pre_c, kick_c, post_c, d, dtype=torch.float64)
        assert torch.allclose(lin_c, lin, rtol=1e-14, atol=1e-14) and torch.allclose(imp_c, imp, rtol=1e-14, atol=1e-14)


def test_multipole_inverse_terms_default_to_float32():
    gen = torch.Generator().manual_seed(3)
    _, pre, kick, post = _chain(4, 3, False, True, True, gen)
    lin, imp = multipole_inverse_terms(pre, kick, post, 4)
    assert lin.dtype == imp.dtype == torch.float32


@pytest.mark.parametrize("d,order,skew", [(4, 3, False), (4, 4, True), (4, 5, False), (6, 3, True), (6, 4, False),
                                          (6, 5, True), (2, 3, False), (2, 5, True)])
def test_2d_screen_rows_match_forward_then_project(d, order, skew):
    gen = torch.Generator().manual_seed(7 * d + order)
    t, pre, kick, post = _chain(d, order, skew, True, True, gen, strength=0.5)
    screen = mf.diagnostics.Histogram2D(axis=(0, 1) if d == 2 else (0, 2), edges=(torch.linspace(-3, 3, 9),
                                                                                torch.linspace(-3, 3, 7)))
    x = torch.randn(500, d, dtype=torch.float64, generator=gen)
    want = screen.project(t(x))
    rows = screen.projection_vectors(post.to(torch.float32), d, "cpu")
    terms = [multipole_terms(r, pre, kick, d) for r in rows]
    # the two rows of a screen share wa, wb and the order
    assert torch.equal(terms[0][1][:2 * d], terms[1][1][:2 * d]) and float(terms[0][1][2 * d + 2]) == order
    for axis, (w, mp) in enumerate(terms):
        w, mp = w.double(), mp.double()
        z = torch.complex(x @ mp[:d], x @ mp[d:2 * d]) ** (order - 1)
        u = x @ w + mp[2 * d] * z.real + mp[2 * d + 1] * z.imag
        assert float((u - want[:, axis]).abs().max()) <= 2e-6 * float(want[:, axis].abs().max()), axis


def _model(transforms, ndim=4, two_d=False):
    edges = torch.linspace(-4.0, 4.0, 17)
    if two_d:
        diag = mf.diagnostics.Histogram2D(axis=(0, 2), edges=(edges, edges))
        meas = torch.ones(16, 16)
    else:
        diag = mf.diagnostics.Histogram1D(axis=0, edges=edges)
        meas = torch.ones(16)
    return mf.ment.MENT(ndim=ndim, transforms=transforms, diagnostics=[[diag] for _ in transforms],
                        measurements=[[meas] for _ in transforms], prior=mf.prior.Gaussian(ndim=ndim, scale=1.0))


class _Custom(nn.Module):
    def forward(self, x):
        return 2.0 * x


@pytest.mark.parametrize("name,transform", [
    ("two kicks", CompositeTransform(MultipoleTransform(3, 0.5), LinearTransform(torch.eye(4)),
                                     MultipoleTransform(4, 0.5))),
    ("projection", ProjectionTransform(torch.tensor([1.0, 0.0, 0.0, 0.0]))),
    ("order 2", CompositeTransform(MultipoleTransform(2, 0.5), LinearTransform(torch.eye(4)))),
    ("order 6", MultipoleTransform(6, 0.5)),
    ("custom module", _Custom()),
    ("custom stage", CompositeTransform(LinearTransform(torch.eye(4)), _Custom())),
])
def test_pack_refuses_unsupported_maps(name, transform):
    model = _model([LinearTransform(torch.eye(4)), transform])
    with pytest.raises(NotImplementedError, match="MultipoleTransform"):
        model._pack(torch.device("cpu"))


def test_pack_refuses_a_kick_in_three_dimensions():
    model = _model([CompositeTransform(MultipoleTransform(3, 0.5), LinearTransform(torch.eye(3)))], ndim=3)
    with pytest.raises(NotImplementedError, match="D = 2 or D >= 4"):
        model._pack(torch.device("cpu"))


@pytest.mark.parametrize("two_d", [False, True])
def test_pack_rows_of_a_mixed_model(two_d):
    """Linear maps keep their plain projection rows and get order-0 multipole rows; a chain gets the rows of
    multipole_terms; a model without a kick carries no multipole rows at all."""
    gen = torch.Generator().manual_seed(11)
    lin = LinearTransform(_matrix(4, gen).float())
    chain, pre, kick, post = _chain(4, 4, True, True, True, gen)
    chain = CompositeTransform(*[LinearTransform(s.matrix.float()) if isinstance(s, LinearTransform) else s
                                 for s in chain.transforms])
    model = _model([lin, chain], two_d=two_d)
    pk = model._pack(torch.device("cpu"))
    proj, mp = (pk["proj2"], pk["mp2"]) if two_d else (pk["proj"], pk["mp"])
    assert pk["kicked"] and mp is not None and (pk["mp2"] if not two_d else pk["mp"]) is None
    lin_rows = (model.diagnostics[0][0].projection_vectors if two_d else model.diagnostics[0][0].projection_vector)(
        lin.matrix, 4, "cpu")
    assert torch.equal(proj[0], lin_rows) and not mp[0].any()
    assert float(mp[1].reshape(-1, 12)[0, 10]) == 4.0
    g1, g2 = model._groups(torch.device("cpu"))
    grp = g2 if two_d else g1
    assert (g1 if two_d else g2) is None and len(grp) == (5 if two_d else 4) and grp[-1] is mp
    linear_only = _model([lin, LinearTransform(_matrix(4, gen).float())], two_d=two_d)
    pk = linear_only._pack(torch.device("cpu"))
    assert not pk["kicked"] and pk["mp"] is None and pk["mp2"] is None
    g1, g2 = linear_only._groups(torch.device("cpu"))
    assert len(g2 if two_d else g1) == (4 if two_d else 3)
