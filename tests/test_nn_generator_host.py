"""NNGenerator host side: construction, default initialisation, checkpoint keys, refusals and the C entry points'
argument checks (all before any launch, so no GPU is needed)."""
import ctypes

import pytest
import torch
import torch.nn as nn

import mentflow_b200 as mf
from mentflow_b200 import _lib
from mentflow_b200.generate import NNGenerator, build_generator

MFB_E_BADARG, MFB_E_UNSUPPORTED = -1, -2


def sequential(din, dout, layers, hidden=64):
    mods = [nn.Linear(din, hidden), nn.Tanh()]
    for _ in range(layers - 1):
        mods += [nn.Linear(hidden, hidden), nn.Tanh()]
    return nn.Sequential(*mods, nn.Linear(hidden, dout))


@pytest.mark.parametrize("din,dout,layers", [(6, 6, 3), (2, 2, 1), (1, 8, 8), (8, 1, 2)])
def test_default_init_equals_nn_sequential_under_one_seed(din, dout, layers):
    torch.manual_seed(17)
    gen = NNGenerator(din, dout, layers, 64)
    torch.manual_seed(17)
    ref = sequential(din, dout, layers)
    ref_sd = ref.state_dict()
    sd = gen.state_dict()
    assert sorted(sd) == sorted("_network." + k for k in ref_sd)
    for k, v in ref_sd.items():
        assert torch.equal(sd["_network." + k], v), k
    assert gen.dim() == dout and gen.input_features == din and gen.output_features == dout
    assert gen.w_hid.shape == (layers - 1, 64, 64) and gen.b_hid.shape == (layers - 1, 64)


def test_state_dict_round_trip():
    torch.manual_seed(0)
    a = NNGenerator(6, 6, 3, 64)
    torch.manual_seed(1)
    b = NNGenerator(6, 6, 3, 64)
    assert not torch.equal(a.w_hid, b.w_hid)
    b.load_state_dict(a.state_dict())
    for pa, pb in zip(a.parameters(), b.parameters()):
        assert torch.equal(pa, pb)
    assert sorted(a.state_dict()) == sorted(f"_network.{m}.{f}" for m in (0, 2, 4, 6) for f in ("weight", "bias"))
    with pytest.raises(RuntimeError):
        b.load_state_dict({k: v for k, v in a.state_dict().items() if k != "_network.4.bias"})
    with pytest.raises(RuntimeError):
        b.load_state_dict(dict(a.state_dict(), **{"_network.8.weight": torch.zeros(1)}))


def test_build_generator_takes_the_common_options():
    gen = build_generator("nn", input_features=4, output_features=6, hidden_layers=2, hidden_units=64, transforms=5,
                          dropout=0.0, activation="tanh")
    assert isinstance(gen, NNGenerator) and gen.input_features == 4 and gen.dim() == 6
    with pytest.raises(TypeError, match="bins"):
        build_generator("nn", input_features=4, output_features=6, hidden_layers=2, hidden_units=64, bins=8)
    assert mf.generate.NNGenerator is NNGenerator


@pytest.mark.parametrize("kws", [
    dict(input_features=0, output_features=6, hidden_layers=3, hidden_units=64),
    dict(input_features=9, output_features=6, hidden_layers=3, hidden_units=64),
    dict(input_features=6, output_features=0, hidden_layers=3, hidden_units=64),
    dict(input_features=6, output_features=9, hidden_layers=3, hidden_units=64),
    dict(input_features=6, output_features=6, hidden_layers=0, hidden_units=64),
    dict(input_features=6, output_features=6, hidden_layers=9, hidden_units=64),
    dict(input_features=6, output_features=6, hidden_layers=3, hidden_units=32),
    dict(input_features=6, output_features=6, hidden_layers=3, hidden_units=64, dropout=0.1),
    dict(input_features=6, output_features=6, hidden_layers=3, hidden_units=64, activation="relu"),
])
def test_unsupported_configurations_are_refused_at_construction(kws):
    with pytest.raises(NotImplementedError):
        NNGenerator(**kws)


def test_cpu_tensors_are_refused_without_fallback():
    gen = NNGenerator(2, 2, 3, 64)
    z = gen.sample_base(10)
    assert z.shape == (10, 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gen(z)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        gen.sample(10)


def test_log_prob_is_none_and_there_is_no_inverse():
    gen = NNGenerator(2, 2, 3, 64)
    assert gen.log_prob(torch.zeros(3, 2)) is None
    with pytest.raises(NotImplementedError):
        gen.inverse(torch.zeros(3, 2))
    with pytest.raises(NotImplementedError):
        gen.inverse_steps(torch.zeros(3, 2))


def test_monte_carlo_entropy_without_log_prob_raises_value_error():
    est = mf.entropy.MonteCarloEntropyEstimator()
    with pytest.raises(ValueError, match="KNNEntropyEstimator"):
        est(torch.zeros(4, 2), None)


def test_c_entry_points_refuse_bad_arguments_before_any_launch():
    lib = _lib.load()
    assert lib.mfb_nn_supported(6, 6, 64, 3) == 1
    for bad in [(0, 6, 64, 3), (9, 6, 64, 3), (6, 0, 64, 3), (6, 9, 64, 3), (6, 6, 32, 3), (6, 6, 64, 0),
                (6, 6, 64, 9)]:
        assert lib.mfb_nn_supported(*bad) == 0, bad
        assert lib.mfb_nn_bwd_workspace_bytes(100, *bad) == 0, bad
    assert lib.mfb_nn_bwd_workspace_bytes(0, 6, 6, 64, 3) == 0
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)

    def fwd(z=p, n=10, din=6, dout=6, h=64, layers=3, w_hid=p, b_hid=p, w_in=p, x=p):
        return lib.mfb_nn_fwd(z, n, din, dout, h, layers, w_in, p, w_hid, b_hid, p, p, x, None)

    assert fwd(z=None) == MFB_E_BADARG
    assert fwd(x=None) == MFB_E_BADARG
    assert fwd(w_in=None) == MFB_E_BADARG
    assert fwd(n=0) == MFB_E_BADARG
    assert fwd(w_hid=None) == MFB_E_BADARG          # required when there is more than one layer
    assert fwd(din=9) == MFB_E_UNSUPPORTED
    assert fwd(dout=0) == MFB_E_UNSUPPORTED
    assert fwd(h=128) == MFB_E_UNSUPPORTED
    assert fwd(layers=9) == MFB_E_UNSUPPORTED

    def bwd(z=p, gx=p, n=10, din=6, dout=6, h=64, layers=3, w_hid=p, gw_hid=p, work=p, gw_in=p):
        return lib.mfb_nn_bwd(z, gx, n, din, dout, h, layers, p, p, w_hid, p, p, p, None, gw_in, p, gw_hid, p, p, p,
                              work, 1 << 30, None)

    assert bwd(z=None) == MFB_E_BADARG
    assert bwd(gx=None) == MFB_E_BADARG
    assert bwd(work=None) == MFB_E_BADARG
    assert bwd(gw_in=None) == MFB_E_BADARG
    assert bwd(n=0) == MFB_E_BADARG
    assert bwd(gw_hid=None) == MFB_E_BADARG
    assert bwd(din=0) == MFB_E_UNSUPPORTED
    assert bwd(dout=9) == MFB_E_UNSUPPORTED
    assert bwd(h=63) == MFB_E_UNSUPPORTED
    assert bwd(layers=0) == MFB_E_UNSUPPORTED
