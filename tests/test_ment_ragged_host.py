"""Host side of classical MENT with screens of different sizes (no GPU): the offsets checks of ops before any launch,
the argument checks of the ragged C entry points, the exported symbols, and the packing and persistence of a model
whose screens differ in size."""
import ctypes
import os
import re

import pytest
import torch

import mentflow_b200 as mf
from mentflow_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RAGGED = ("mfb_ment_prob_ragged", "mfb_ment_prob_grid_ragged", "mfb_ment_integrate_ragged", "mfb_ment_mh_ragged")


def _r1(sizes, d=3, offsets=None, device="cpu"):
    t = sum(sizes)
    off = [0]
    for b in sizes:
        off.append(off[-1] + b)
    return ops.RaggedTables1D(torch.zeros(len(sizes), d, device=device), torch.zeros(t, device=device),
                              torch.zeros(t, device=device), off if offsets is None else offsets)


def _r2(shapes, d=3, offsets2=None, device="cpu"):
    rows = [[0], [0], [0]]
    for bx, by in shapes:
        rows[0].append(rows[0][-1] + bx)
        rows[1].append(rows[1][-1] + by)
        rows[2].append(rows[2][-1] + bx * by)
    return ops.RaggedTables2D(torch.zeros(len(shapes), 2, d, device=device), torch.zeros(rows[0][-1], device=device),
                              torch.zeros(rows[1][-1], device=device), torch.zeros(rows[2][-1], device=device),
                              rows if offsets2 is None else offsets2)


def test_bad_offsets_are_refused_on_the_host():
    with pytest.raises(ValueError, match="at least 2 bins, table 1 has 1"):
        ops._ment_tables(_r1([4, 1, 3]), None, 3, "cpu")
    for bad in ([0, 4, 5], [0, 4, 5, 7, 8], [1, 4, 5, 8], [0, 4, 5, 9]):        # length, start, end
        with pytest.raises(ValueError, match="offsets"):
            ops._ment_tables(_r1([4, 1, 3], offsets=bad), None, 3, "cpu")
    with pytest.raises(ValueError, match="at least 2 bins, table 1 has -1"):     # decreasing
        ops._ment_tables(_r1([4, 3], offsets=[0, 8, 7]), None, 3, "cpu")
    with pytest.raises(ValueError, match=r"offsets2\[1\].*at least 2 bins, table 0 has 1"):
        ops._ment_tables(None, _r2([(3, 1), (4, 5)]), 3, "cpu")
    good = _r2([(3, 2), (4, 5)])
    with pytest.raises(ValueError, match=r"offsets2\[2\]"):
        ops._ment_tables(None, good._replace(offsets2=good.offsets2[:2] + [[0, 6, 27]]), 3, "cpu")
    with pytest.raises(ValueError, match="3 rows"):
        ops._ment_tables(None, good._replace(offsets2=good.offsets2[:2]), 3, "cpu")
    with pytest.raises(ValueError, match=r"coords and values \(T,\)"):
        ops._ment_tables(_r1([4, 3])._replace(values=torch.zeros(6)), None, 3, "cpu")


def test_totals_past_int32_are_refused_on_the_host():
    big = 2 ** 31 + 4
    r1 = ops.RaggedTables1D(torch.zeros(2, 3), torch.empty(big, device="meta"), torch.empty(big, device="meta"),
                            [0, 4, big])
    with pytest.raises(ValueError, match="int32"):
        ops._ment_tables(r1, None, 3, "cpu")
    n = 50_000                                    # one table of n x n values: 2.5e9 entries
    r2 = ops.RaggedTables2D(torch.zeros(1, 2, 3), torch.zeros(n), torch.zeros(n), torch.empty(n * n, device="meta"),
                            [[0, n], [0, n], [0, n * n]])
    with pytest.raises(ValueError, match="int32"):
        ops._ment_tables(None, r2, 3, "cpu")


def test_a_uniform_family_beside_a_ragged_one_is_passed_with_offsets_k_b():
    g1, off = ops._as_ragged1((torch.zeros(3, 2), torch.zeros(3, 7), torch.zeros(3, 7)))
    assert off == [0, 7, 14, 21] and g1.coords.shape == (21,) and g1.mp is None
    g2, off2 = ops._as_ragged2((torch.zeros(2, 2, 2), torch.zeros(2, 5), torch.zeros(2, 4), torch.zeros(2, 5, 4)))
    assert off2 == [0, 5, 10] + [0, 4, 8] + [0, 20, 40] and g2.values.shape == (40,)


def test_ragged_symbols_are_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "mentflow_b200.h")).read()
    declared = set(re.findall(r"\b(mfb_[a-z0-9_]+)\s*\(", header))
    lib = _lib.load()
    for name in RAGGED:
        assert name in declared and name in _lib.SIGNATURES and hasattr(lib, name)
    for name in RAGGED:         # as many arguments as the uniform sibling: b -> (offsets, total), (bx, by) -> offsets2
        uniform = _lib.SIGNATURES[name.replace("_ragged", "")][1]
        assert len(_lib.SIGNATURES[name][1]) == len(uniform)


def test_ragged_entry_points_check_their_arguments_before_any_launch():
    lib = _lib.load()
    p = ctypes.c_void_p(256)                    # never dereferenced: every call below is refused first
    f32 = (ctypes.c_float * 1)(0.0)
    i32 = (ctypes.c_int32 * 8)(*[2] * 8)
    host = ctypes.cast(i32, ctypes.c_void_p)
    hf = ctypes.cast(f32, ctypes.c_void_p)

    def prob(proj=p, coords=p, tables=p, k=2, off=p, total=6, mp=None, proj2=None, cx=None, cy=None, tab2=None,
             k2=0, off2=None, mp2=None, g=10):
        return lib.mfb_ment_prob_ragged(p, g, 3, proj, coords, tables, k, off, total, mp, proj2, cx, cy, tab2, k2,
                                        off2, mp2, 0.0, 0.0, p, None)

    assert prob(off=None) == -1                             # 1-D tables without offsets
    assert prob(total=3) == -1                              # fewer than 2 bins a table in all
    assert prob(k=-1) == -1
    assert prob(k2=1, proj2=p, cx=p, cy=p, tab2=p) == -1    # 2-D tables without offsets2
    assert prob(k2=1, proj2=p, cx=p, cy=None, tab2=p, off2=p) == -1
    assert prob(mp=None, mp2=p, k2=1, proj2=p, cx=p, cy=p, tab2=p, off2=p) == -1   # kicks need the 1-D rows too
    assert prob(k=0, off=None, total=0, g=0) == 0           # empty families, nothing to evaluate
    assert prob(total=60_000) == -2                         # past the 200 KB of shared memory: refused, no launch
    assert lib.mfb_ment_prob_grid_ragged(3, host, hf, hf, p, p, p, 2, p, 60_000, None, None, None, None, None, 0,
                                         None, None, 0.0, 0.0, p, None) == -2
    assert lib.mfb_ment_prob_grid_ragged(3, host, hf, hf, p, p, p, 2, None, 6, None, None, None, None, None, 0,
                                         None, None, 0.0, 0.0, p, None) == -1
    integ = lambda off, total: lib.mfb_ment_integrate_ragged(  # noqa: E731
        3, p, 4, 0, None, 0, -1, 2, host, hf, hf, p, None, p, p, p, 2, off, total, None, None, None, None, None, 0,
        None, None, 0.0, 0.0, p, None)
    assert integ(None, 6) == -1 and integ(p, 60_000) == -2
    mh = lambda off, total: lib.mfb_ment_mh_ragged(  # noqa: E731
        3, p, p, p, 2, off, total, None, None, None, None, None, 0, None, None, 0.0, 0.0, 0, 10, None, 1.0, p, 0, 1, 1,
        1, p, p, None)
    assert mh(None, 6) == -1 and mh(p, 60_000) == -2


def _model(device="cpu"):
    tfs = [mf.simulate.LinearTransform(torch.eye(3) * (1.0 + 0.1 * i)) for i in range(3)]
    h1 = lambda axis, b: mf.diagnostics.Histogram1D(axis=axis, edges=torch.linspace(-3, 3, b + 1), bandwidth=0.5)  # noqa: E731
    h2 = lambda bx, by: mf.diagnostics.Histogram2D(  # noqa: E731
        axis=(0, 1), edges=(torch.linspace(-3, 3, bx + 1), torch.linspace(-2, 2, by + 1)), bandwidth=(0.5, 0.5))
    diags = [[h1(0, 10), h2(5, 6)], [h1(1, 20)], [h1(2, 10), h2(7, 8)]]
    meas = [[torch.rand(10), torch.rand(5, 6)], [torch.rand(20)], [torch.rand(10), torch.rand(7, 8)]]
    return mf.ment.MENT(ndim=3, transforms=tfs, diagnostics=diags, measurements=meas, mode="integrate", device=device)


def test_a_model_of_mixed_sizes_packs_ragged_tables():
    model = _model()
    for row in model.lagrange_functions:
        for lf in row:
            lf.set_values(torch.rand(lf.values.shape))
    g1, g2 = model._groups(torch.device("cpu"))
    assert isinstance(g1, ops.RaggedTables1D) and isinstance(g2, ops.RaggedTables2D)
    assert g1.offsets == [0, 10, 30, 40] and g1.coords.shape == (40,) and g1.proj.shape == (3, 3)
    assert g2.offsets2 == [[0, 5, 12], [0, 6, 14], [0, 30, 86]] and g2.cx.shape == (12,) and g2.cy.shape == (14,)
    lfs = model.lagrange_functions
    assert torch.equal(g1.values, torch.cat([lfs[0][0].values, lfs[1][0].values, lfs[2][0].values]))
    assert torch.equal(g2.values, torch.cat([lfs[0][1].values.reshape(-1), lfs[2][1].values.reshape(-1)]))
    assert ops._as_ragged1(g1)[1] == g1.offsets                       # the host checks accept the packed layout
    assert ops._as_ragged2(g2)[1] == sum(g2.offsets2, [])


def test_equal_sizes_keep_the_stacked_tables():
    model = _model()
    model.diagnostics[1][0] = mf.diagnostics.Histogram1D(axis=1, edges=torch.linspace(-3, 3, 11), bandwidth=0.5)
    model.measurements[1][0] = torch.rand(10)
    model.diagnostics[2][1] = mf.diagnostics.Histogram2D(
        axis=(0, 1), edges=(torch.linspace(-3, 3, 6), torch.linspace(-2, 2, 7)), bandwidth=(0.5, 0.5))
    model.measurements[2][1] = torch.rand(5, 6)
    model.initialize_lagrange_functions()
    g1, g2 = model._groups(torch.device("cpu"))
    assert type(g1) is tuple and g1[1].shape == (3, 10) and g1[2].shape == (3, 10)
    assert type(g2) is tuple and g2[3].shape == (2, 5, 6)


def test_a_ragged_model_survives_save_and_load(tmp_path):
    model = _model()
    for row in model.lagrange_functions:
        for lf in row:
            lf.set_values(torch.rand(lf.values.shape))
    model.epoch = 3
    path = str(tmp_path / "ment.pt")
    model.save(path)
    other = _model()
    other.load(path, device="cpu")
    assert other.epoch == 3
    a, b = model._groups(torch.device("cpu")), other._groups(torch.device("cpu"))
    for x, y in zip(a, b):
        assert type(x) is type(y)
        for s, t in zip(x, y):
            assert (torch.equal(s, t) if isinstance(s, torch.Tensor) else s == t)
