"""``build_generator`` with the reference's signature (mentflow/generate/build.py:80-123)."""
import torch

from .base import GenerativeModel
from .nn import NNGenerator
from .nsf import NSFGenerator


def build_flow(name: str, input_features: int, output_features: int, hidden_layers: int, hidden_units: int,
               transforms: int, device=None, **kws) -> GenerativeModel:
    if name != "nsf":
        raise NotImplementedError(
            f"flow '{name}': only the neural spline flow ('nsf', the reference's configured generator, "
            "experiments/config/gen/flow.yaml:1) has CUDA kernels")
    bins = int(kws.pop("bins", 8))   # zuko.flows.NSF default; experiments/setup.py:120-121 passes 20
    passes = kws.pop("passes", None)  # zuko MAF option forwarded by **kws (generate/build.py:36-40): 2 = coupling layers
    if kws:
        raise TypeError(f"unsupported NSF options: {sorted(kws)}")
    return NSFGenerator(output_features, hidden_units=hidden_units, hidden_layers=hidden_layers,
                        transforms=transforms, bins=bins, device=device, passes=passes)


def build_nn(input_features: int, output_features: int, hidden_layers: int, hidden_units: int, transforms=None,
             dropout: float = 0.0, activation: str = "tanh", device=None, **kws) -> NNGenerator:
    """The reference's common generator options (``transforms`` is a flow option and is ignored) plus the network's
    ``dropout`` and ``activation``."""
    if kws:
        raise TypeError(f"unsupported NN generator options: {sorted(kws)}")
    return NNGenerator(input_features, output_features, hidden_layers=hidden_layers, hidden_units=hidden_units,
                       dropout=dropout, activation=activation, device=device)


def build_generator(name: str, device: torch.device = None, **kws) -> GenerativeModel:
    if name == "nn":
        return build_nn(device=device, **kws)
    if name in ("bpf", "ffjord", "gf", "gmm", "maf", "nag", "nsf", "sospf", "unaf"):
        return build_flow(name=name, device=device, **kws)
    raise ValueError(f"Invalid generative model name '{name}'")
