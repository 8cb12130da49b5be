"""Plain neural-network generator: a tanh MLP from base noise to particles, with no density.

Stands in for the reference's ``mentflow.generate.NNGenerator`` (the paper's baseline, ``build_generator("nn", ...)``).
That source is not available here; its architecture is restated from SURVEY.md row 14 and is unverified against the
reference:

* ``z ~ N(0, I_{input_features})``;
* ``x = W_out tanh(... tanh(W_2 tanh(W_1 z + b_1) + b_2) ...) + b_out``: ``Linear(Din, H)``, then
  ``hidden_layers - 1`` times ``Linear(H, H)``, each followed by tanh, then ``Linear(H, Dout)`` with no activation
  (the counting of the NSF conditioner);
* ``log_prob`` returns None;
* ``state_dict`` keys follow an ``nn.Sequential`` of those modules (``NNGenerator._KEY``).

Parameters are stored stacked per role (``w_in``, ``b_in``, ``w_hid``, ``b_hid``, ``w_out``, ``b_out``) in
``nn.Linear`` layout and run through the library's fused CUDA kernels (``ops.nn_forward``).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.nn as nn

from .. import ops
from .base import GenerativeModel

HIDDEN_UNITS = 64     # the one width the CUDA kernels are compiled for
MAX_FEATURES = 8
MAX_HIDDEN_LAYERS = 8


class NNGenerator(GenerativeModel):
    # Restated layer table (SURVEY.md row 14, unverified against the reference): hidden_layers + 1 Linears, Linear k
    # (0 = input, hidden_layers = output) is module 2k of an nn.Sequential stored as `_network`, with a Tanh after
    # every Linear but the last.
    _KEY = "_network.{module}.{field}"

    def __init__(self, input_features: int, output_features: int, hidden_layers: int, hidden_units: int,
                 dropout: float = 0.0, activation: str = "tanh", device=None) -> None:
        super().__init__()
        if float(dropout) != 0.0:
            raise NotImplementedError("the CUDA NN generator has no dropout (dropout must be 0)")
        if activation != "tanh":
            raise NotImplementedError(f"activation '{activation}': the CUDA NN generator is compiled for tanh only")
        if hidden_units != HIDDEN_UNITS:
            raise NotImplementedError(f"the CUDA NN generator is compiled for hidden_units={HIDDEN_UNITS}")
        if not (1 <= input_features <= MAX_FEATURES and 1 <= output_features <= MAX_FEATURES):
            raise NotImplementedError(f"the CUDA NN generator is compiled for 1..{MAX_FEATURES} input and output "
                                      "features")
        if not 1 <= hidden_layers <= MAX_HIDDEN_LAYERS:
            raise NotImplementedError(f"the CUDA NN generator is compiled for 1..{MAX_HIDDEN_LAYERS} hidden layers")
        self.input_features, self.output_features = int(input_features), int(output_features)
        self.hidden_layers, self.hidden_units = int(hidden_layers), int(hidden_units)
        Din, Dout, H, L = self.input_features, self.output_features, self.hidden_units, self.hidden_layers
        # default nn.Linear initialisation, drawn layer by layer in construction order
        first = nn.Linear(Din, H)
        hid = [nn.Linear(H, H) for _ in range(L - 1)]
        last = nn.Linear(H, Dout)
        self.w_in = nn.Parameter(first.weight.detach().clone())          # (H, Din)
        self.b_in = nn.Parameter(first.bias.detach().clone())            # (H,)
        self.w_hid = nn.Parameter(torch.stack([m.weight.detach() for m in hid]) if hid else torch.zeros(0, H, H))
        self.b_hid = nn.Parameter(torch.stack([m.bias.detach() for m in hid]) if hid else torch.zeros(0, H))
        self.w_out = nn.Parameter(last.weight.detach().clone())          # (Dout, H)
        self.b_out = nn.Parameter(last.bias.detach().clone())            # (Dout,)
        self._rng = None
        if device is not None:
            self.to(device)

    def dim(self) -> int:
        return self.output_features

    # nn.Sequential names in checkpoints ----------------------------------------------------
    def _items(self):
        """(state_dict key, stacked tensor, index into it) for every Linear's weight and bias."""
        L = self.hidden_layers
        linears = [(self.w_in, self.b_in, ())] + [(self.w_hid, self.b_hid, (l,)) for l in range(L - 1)] + \
            [(self.w_out, self.b_out, ())]
        for k, (w, b, idx) in enumerate(linears):
            yield self._KEY.format(module=2 * k, field="weight"), w, idx
            yield self._KEY.format(module=2 * k, field="bias"), b, idx

    def state_dict(self, *args, destination=None, prefix="", keep_vars=False, **kwargs):
        out = {} if destination is None else destination
        for name, tensor, idx in self._items():
            value = tensor[idx]
            out[prefix + name] = value if keep_vars else value.detach().clone()
        return out

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        missing = []
        known = set()
        with torch.no_grad():
            for name, tensor, idx in self._items():
                known.add(name)
                if name in state_dict:
                    tensor[idx].copy_(state_dict[name])
                else:
                    missing.append(name)
        unexpected = [k for k in state_dict if k not in known]
        if strict and (missing or unexpected):
            raise RuntimeError(f"state_dict mismatch: missing {missing[:4]}, unexpected {unexpected[:4]}")
        return torch.nn.modules.module._IncompatibleKeys(missing, unexpected)

    # sampling ------------------------------------------------------------------------------
    def sample_base(self, n: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """z ~ N(0, I_Din).  On a CUDA device the draw is the library's Philox kernel on torch's own generator state:
        bitwise ``torch.randn((n, Din), device=...)`` for the same seed, torch's generator moved on identically, and
        safe to capture in a CUDA graph."""
        dev = self.w_in.device
        if dev.type != "cuda":
            return torch.randn((int(n), self.input_features), dtype=torch.float32, device=dev)
        if out is None:
            out = torch.empty((int(n), self.input_features), dtype=torch.float32, device=dev)
        return self.rng(dev).normal_(out)

    def rng(self, device=None) -> "ops.PhiloxStream":
        dev = torch.device(device) if device is not None else self.w_in.device
        if self._rng is None or self._rng.device != dev:
            self._rng = ops.PhiloxStream(dev)
        return self._rng

    def forward(self, z: torch.Tensor) -> torch.Tensor:
        return ops.nn_forward(z, self.w_in, self.b_in, self.w_hid, self.b_hid, self.w_out, self.b_out)

    def forward_and_log_prob(self, z: torch.Tensor) -> Tuple[torch.Tensor, None]:
        return self.forward(z), None

    def sample(self, n: int) -> torch.Tensor:
        return self.forward(self.sample_base(n))

    def sample_and_log_prob(self, n: int) -> Tuple[torch.Tensor, None]:
        return self.sample(n), None

    def log_prob(self, x: torch.Tensor) -> None:
        """None: a plain network has no tractable density."""
        return None
