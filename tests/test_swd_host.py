"""Sliced Wasserstein distance: refusals raised before anything needs a GPU, the host-side direction generation and the
reference's spelling of the class name."""
import math

import pytest
import torch

from mentflow_b200 import loss, ops


def test_cpu_tensors_are_refused_without_fallback():
    x, y = torch.randn(100, 3), torch.randn(80, 3)
    theta = loss.random_projections(3, 5).t().float().contiguous()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        loss.sliced_wasserstein_distance(x, y)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        loss.SlicedWassersteinDistance(y)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.swd_sort(y, theta)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.swd_wpp(x, theta, torch.randn(5, 80), 2)


@pytest.mark.parametrize("xs,ys", [((100,), (80, 3)), ((100, 3), (80,)), ((2, 100, 3), (80, 3)), ((100, 3), (80, 4)),
                                   ((100, 0), (80, 0)), ((100, 9), (80, 9)), ((0, 3), (80, 3)), ((100, 3), (0, 3))])
def test_bad_shapes_are_refused(xs, ys):
    x, y = torch.randn(xs), torch.randn(ys)
    with pytest.raises(ValueError):
        loss.sliced_wasserstein_distance(x, y)


def test_sizes_past_int32_are_refused():
    big = torch.empty(2 ** 31, 2, device="meta")
    with pytest.raises(ValueError, match="2\\^31"):
        loss.sliced_wasserstein_distance(big, torch.randn(10, 2))
    with pytest.raises(ValueError, match="2\\^31"):
        loss.sliced_wasserstein_distance(torch.randn(10, 2), big)
    with pytest.raises(ValueError, match="2\\^31"):
        loss.SlicedWassersteinDistance(big)


@pytest.mark.parametrize("p", [0.0, 0.999, -1.0, math.inf, math.nan])
def test_bad_p_is_refused(p):
    x, y = torch.randn(100, 3), torch.randn(80, 3)
    with pytest.raises(ValueError, match="p ="):
        loss.sliced_wasserstein_distance(x, y, p=p)
    with pytest.raises(ValueError, match="p ="):
        loss.SlicedWassersteinDistance(y, p=p)


@pytest.mark.parametrize("shape", [(4, 10), (3, 0), (30,), (10, 3)])
def test_projections_of_the_wrong_shape_are_refused(shape):
    x, y = torch.randn(100, 3), torch.randn(80, 3)
    with pytest.raises(ValueError, match="projections"):
        loss.sliced_wasserstein_distance(x, y, projections=torch.randn(shape))
    with pytest.raises(ValueError, match="projections"):
        loss.SlicedWassersteinDistance(y, projections=torch.randn(shape))


def test_reference_that_requires_grad_is_refused():
    x, y = torch.randn(100, 3), torch.randn(80, 3, requires_grad=True)
    with pytest.raises(ValueError, match="require grad"):
        loss.sliced_wasserstein_distance(x, y)
    with pytest.raises(ValueError, match="require grad"):
        loss.SlicedWassersteinDistance(y)
    with pytest.raises(ValueError, match="requires grad"):
        ops.swd_wpp(x, torch.randn(5, 3), torch.randn(5, 80, requires_grad=True), 2)


def test_sample_weights_are_not_accepted():
    x, y = torch.randn(100, 3), torch.randn(80, 3)
    with pytest.raises(TypeError):
        loss.sliced_wasserstein_distance(x, y, torch.full((100,), 0.01), torch.full((80,), 1 / 80))
    with pytest.raises(TypeError):
        loss.sliced_wasserstein_distance(x, y, a=torch.full((100,), 0.01))


def test_random_projections_are_unit_columns_and_follow_the_seed():
    a = loss.random_projections(6, 50, seed=7)
    assert a.shape == (6, 50) and a.dtype == torch.float64
    assert torch.allclose(a.norm(dim=0), torch.ones(50, dtype=torch.float64), rtol=0, atol=1e-15)
    assert torch.equal(a, loss.random_projections(6, 50, seed=7))
    assert not torch.equal(a, loss.random_projections(6, 50, seed=8))
    g = torch.randn(6, 50, generator=torch.Generator().manual_seed(7), dtype=torch.float64)
    assert torch.equal(a, g / g.norm(dim=0, keepdim=True))
    torch.manual_seed(3)
    b = loss.random_projections(4, 9)
    torch.manual_seed(3)
    assert torch.equal(b, loss.random_projections(4, 9))
    with pytest.raises(ValueError):
        loss.random_projections(3, 0)


def test_reference_spelling_is_an_alias():
    assert loss.SlicedWassersteindDistance is loss.SlicedWassersteinDistance
