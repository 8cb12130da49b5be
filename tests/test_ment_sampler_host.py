"""CPU checks of the test-suite's float64 stand-ins for classical MENT: the numpy Philox4x32-10 that the sampler's
draw-by-draw test replays (Random123 known-answer vectors), and the oracle's Lagrange interpolation against the scipy
interpolator the reference calls (ment.py:45-52), on non-uniform centres and exactly on them."""
import numpy as np
import pytest
import torch
from scipy.interpolate import RegularGridInterpolator

from mfb_testutil import philox4x32_10, philox_ment, sampler_uniforms
from oracle import hotpath as hp


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox4x32_10_known_answers(ctr, key, want):
    assert tuple(int(v) for v in philox4x32_10(ctr, key)) == want


def test_philox_ment_layout_splits_counter_and_seed_into_words():
    seed, counter = 0x0123456789ABCDEF, np.array([0, 2**32 - 1, 2**32, 2**40 + 7], dtype=np.uint64)
    got = philox_ment(counter, 3, seed)
    for n, c in enumerate(counter.tolist()):
        want = philox4x32_10((c & 0xFFFFFFFF, c >> 32, 3, 0), (seed & 0xFFFFFFFF, seed >> 32))
        assert np.array_equal(got[n], want)


def test_sampler_uniforms_are_53_bit_and_take_the_stream_words_in_order():
    uu, rnd = sampler_uniforms(seed=5, offset=2**32 - 2, size=4, d=8)
    assert uu.shape == (4,) and np.all((uu > 0) & (uu < 1))
    assert rnd.shape == (4, 16)
    r0 = philox_ment(np.uint64(2**32 - 2) + np.arange(4, dtype=np.uint64), 0, 5)
    assert np.array_equal(rnd[:, :2], r0[:, 2:])
    # words 2 .. 15 of D = 8 come from streams 1 .. 4 in order (the kernel also draws stream 5 and drops it)
    blocks = [philox_ment(np.uint64(2**32 - 2) + np.arange(4, dtype=np.uint64), 1 + b, 5) for b in range(4)]
    assert np.array_equal(rnd[:, 2:], np.concatenate(blocks, axis=1)[:, :14])


def _geometric_centres(n, lo=-3.0, ratio=1.35):
    steps = ratio ** np.arange(n - 1)
    return (lo + np.concatenate([[0.0], np.cumsum(steps)]) * (6.0 / steps.sum())).astype(np.float32)


def _edge_points(c):
    """The centres themselves, one fp32 ulp inside and outside both ends, and points between the centres."""
    c = c.astype(np.float32)
    inf = np.float32(np.inf)
    ends = [np.nextafter(c[0], -inf), np.nextafter(c[0], inf), np.nextafter(c[-1], -inf), np.nextafter(c[-1], inf)]
    mids = 0.5 * (c[:-1] + c[1:])
    return np.concatenate([c, np.array(ends, dtype=np.float32), mids.astype(np.float32), c - 7.0, c + 7.0])


@pytest.mark.parametrize("n", [2, 3, 9, 33])
def test_lagrange_interp_matches_scipy_on_non_uniform_centres(n):
    rng = np.random.default_rng(n)
    c = _geometric_centres(n)
    t = rng.random(n) + 0.1
    u = _edge_points(c)
    want = RegularGridInterpolator((c.astype(np.float64),), t, method="linear", bounds_error=False,
                                   fill_value=0.0)(u.astype(np.float64)[:, None])
    got = hp.lagrange_interp(torch.from_numpy(t), torch.from_numpy(c), torch.from_numpy(u)).numpy()
    assert np.allclose(got, want, rtol=1e-12, atol=0.0)
    assert np.count_nonzero(got) >= n + 2 and got[n + 0] == 0 and got[n + 3] == 0   # closed interval, zero outside


@pytest.mark.parametrize("nx,ny", [(2, 3), (7, 4), (12, 9)])
def test_lagrange_interp_2d_matches_scipy_on_non_uniform_centres(nx, ny):
    rng = np.random.default_rng(nx * ny)
    cx, cy = _geometric_centres(nx, -2.5, 1.4), _geometric_centres(ny, -3.5, 0.8)
    t = rng.random((nx, ny)) + 0.1
    px, py = _edge_points(cx), _edge_points(cy)
    uv = np.stack(np.meshgrid(px, py, indexing="ij"), -1).reshape(-1, 2)
    want = RegularGridInterpolator((cx.astype(np.float64), cy.astype(np.float64)), t, method="linear",
                                   bounds_error=False, fill_value=0.0)(uv.astype(np.float64))
    got = hp.lagrange_interp_2d(torch.from_numpy(t), torch.from_numpy(cx), torch.from_numpy(cy),
                                torch.from_numpy(uv)).numpy()
    assert np.allclose(got, want, rtol=1e-12, atol=1e-15)
    assert np.count_nonzero(got) > 0.2 * got.size
