"""Neural spline flow generator on the CUDA kernels.

Stands in for ``mentflow.generate.WrappedZukoFlow`` around ``zuko.flows.NSF`` inverted by
``build_flow`` (generate/build.py:36-46, generate/flows/zuko.py:10-53): same methods
(``sample``, ``sample_base``, ``log_prob``, ``sample_and_log_prob``, ``forward``, ``inverse``,
``forward_steps``, ``inverse_steps``), sampling direction = one conditioner pass per layer.

Parameters are stored stacked over the flow's layers (one tensor per role, so the optimiser
touches 2*(2+L) tensors instead of 40) and exposed under zuko-style names in ``state_dict``:
``_flow.transform.transforms.{t}.hyper.{2l}.{weight,bias,mask}``.  (The exact key layout of
zuko 1.3.1 cannot be verified here -- zuko is not installable; SURVEY.md 8f-2.)
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from .. import ops
from .base import GenerativeModel


def layer_order(features: int, layer: int, passes: Optional[int] = None) -> List[int]:
    """Dependency order of layer ``layer``: natural for even layers, reversed for odd ones (zuko MAF without
    randperm), then grouped into ``passes`` classes, ``order // ceil(features / passes)`` (zuko
    MaskedAutoregressiveTransform).  passes = None or >= features: fully autoregressive; passes = 2: the
    coupling variant (the first half of the features gets unconditional splines, the second half is
    conditioned on the first)."""
    order = list(range(features))
    order = order if layer % 2 == 0 else order[::-1]
    if passes is not None:
        passes = min(max(int(passes), 1), features)
        group = -(-features // passes)
        order = [o // group for o in order]
    return order


def conditioner_masks(order: Sequence[int], total: int, hidden_units: int, hidden_layers: int):
    """Closed form of zuko's MaskedMLP masks for a strict autoregressive ordering.

    A unit/output of dependency class c may read the features whose order is smaller than c.
    With C distinct order values (C = D for a fully autoregressive layer, C = 2 for a coupling layer) hidden
    unit h has class 1 + h mod (C-1); output rows of feature i have class order[i];
    a connection a -> b exists iff class(a) <= class(b) (for inputs: order[j] < class(b)).
    Returns [mask_in (H, D), mask_hid (H, H) x (L-1), mask_out (D*total, H)] as bool tensors.
    """
    d = len(order)
    order_t = torch.as_tensor(list(order))
    classes = int(order_t.max()) + 1
    if d > 1 and classes > 1:
        hid_class = 1 + torch.arange(hidden_units) % (classes - 1)
    else:
        raise ValueError("a conditioned flow layer needs at least 2 features in 2 dependency classes")
    out_class = torch.repeat_interleave(order_t, total)
    masks = [order_t[None, :] < hid_class[:, None]]
    for _ in range(hidden_layers - 1):
        masks.append(hid_class[None, :] <= hid_class[:, None])
    masks.append(hid_class[None, :] <= out_class[:, None])
    return masks


class NSFGenerator(GenerativeModel):
    def __init__(self, features: int, hidden_units: int = 64, hidden_layers: int = 3, transforms: int = 5,
                 bins: int = 20, device=None, passes: Optional[int] = None) -> None:
        super().__init__()
        if hidden_units != 64:
            raise NotImplementedError("the CUDA conditioner is compiled for hidden_units=64")
        if not (2 <= features <= 6):
            raise NotImplementedError("the CUDA flow is compiled for 2..6 features")
        if 3 * bins - 1 > 64 or bins < 2:
            raise NotImplementedError("bins must satisfy 3*bins-1 <= 64")
        self.features, self.hidden_units, self.hidden_layers = features, hidden_units, hidden_layers
        self.transforms, self.bins = transforms, bins
        # zuko's `passes`: None / >= features = autoregressive (tcgen05 kernels); 2 = coupling layers (the fp32
        # CUDA-core kernels: the tensor-core operand images are laid out for strict orderings)
        self.passes = None if passes is None or int(passes) >= features else max(int(passes), 2)
        self.total = 3 * bins - 1
        T, H, L, D, P = transforms, hidden_units, hidden_layers, features, self.total
        # default nn.Linear initialisation, drawn layer by layer in construction order
        w_in, b_in, w_hid, b_hid, w_out, b_out = [], [], [], [], [], []
        for _ in range(T):
            lin = nn.Linear(D, H)
            w_in.append(lin.weight.detach()), b_in.append(lin.bias.detach())
            wh, bh = [], []
            for _ in range(L - 1):
                lin = nn.Linear(H, H)
                wh.append(lin.weight.detach()), bh.append(lin.bias.detach())
            w_hid.append(torch.stack(wh) if wh else torch.zeros(0, H, H))
            b_hid.append(torch.stack(bh) if bh else torch.zeros(0, H))
            lin = nn.Linear(H, D * P)
            w_out.append(lin.weight.detach()), b_out.append(lin.bias.detach())
        self.w_in = nn.Parameter(torch.stack(w_in))      # (T, H, D)
        self.b_in = nn.Parameter(torch.stack(b_in))      # (T, H)
        self.w_hid = nn.Parameter(torch.stack(w_hid))    # (T, L-1, H, H)
        self.b_hid = nn.Parameter(torch.stack(b_hid))    # (T, L-1, H)
        self.w_out = nn.Parameter(torch.stack(w_out))    # (T, D*P, H)
        self.b_out = nn.Parameter(torch.stack(b_out))    # (T, D*P)
        m_in, m_hid, m_out = [], [], []
        for t in range(T):
            masks = conditioner_masks(layer_order(D, t, self.passes), P, H, L)
            m_in.append(masks[0])
            m_hid.append(torch.stack(masks[1:-1]) if L > 1 else torch.zeros(0, H, H, dtype=torch.bool))
            m_out.append(masks[-1])
        self.register_buffer("m_in", torch.stack(m_in).float(), persistent=False)
        self.register_buffer("m_hid", torch.stack(m_hid).float(), persistent=False)
        self.register_buffer("m_out", torch.stack(m_out).float(), persistent=False)
        self._orders = [layer_order(D, t, self.passes) for t in range(T)]
        self._pack_key, self._pack_cache = None, None
        self._rng = None
        if device is not None:
            self.to(device)

    # ------------------------------------------------------------------ parameters
    def dim(self) -> int:
        return self.features

    def packed_pair(self):
        """(packed, packed_om) on a CUDA device: one kernel launch (``ops.PackParameters``), differentiable w.r.t.
        the six parameter tensors through one launch the other way."""
        dims = (self.transforms, self.features, self.hidden_units, self.hidden_layers, self.bins)
        return ops.PackParameters.apply(self.w_in, self.b_in, self.w_hid, self.b_hid, self.w_out, self.b_out,
                                        self.m_in, self.m_hid, self.m_out, dims)

    def packed_parameters(self) -> torch.Tensor:
        """(T, floats_per_layer) block in the kernels' layout: masked, transposed to [in][out],
        per-feature output blocks padded from 3*bins-1 to 64.  CUDA parameters: one launch of the packing kernel;
        CPU parameters (host-side tests of the layout): the same layout spelled in differentiable torch ops."""
        if self.w_in.is_cuda:
            return self.packed_pair()[0]
        T, H, D, P = self.transforms, self.hidden_units, self.features, self.total
        parts = [(self.w_in * self.m_in).transpose(1, 2).reshape(T, -1), self.b_in]
        if self.hidden_layers > 1:
            wh = (self.w_hid * self.m_hid).transpose(2, 3)             # (T, L-1, in, out)
            hid = torch.cat([wh.reshape(T, self.hidden_layers - 1, -1), self.b_hid], dim=2)
            parts.append(hid.reshape(T, -1))
        wo = (self.w_out * self.m_out).reshape(T, D, P, H).permute(0, 1, 3, 2)   # (T, D, in, P)
        wo = torch.nn.functional.pad(wo, (0, 64 - P))
        bo = torch.nn.functional.pad(self.b_out.reshape(T, D, P), (0, 64 - P))
        parts += [wo.reshape(T, -1), bo.reshape(T, -1)]
        return torch.cat(parts, dim=1).contiguous()

    def packed_parameters_om(self) -> torch.Tensor:
        """(T, floats) masked weights in out-major layout for the backward data-gradient kernels:
        W1 [64][D] | Wl [64][64] x (L-1) | Wout [D*64 (59->64 padded rows)][64]; detached (the
        parameter gradient flows through ``packed_parameters``)."""
        T, H, D, P = self.transforms, self.hidden_units, self.features, self.total
        if self.w_in.is_cuda:
            with torch.no_grad():
                return self.packed_pair()[1]
        with torch.no_grad():
            parts = [(self.w_in * self.m_in).reshape(T, -1)]
            if self.hidden_layers > 1:
                parts.append((self.w_hid * self.m_hid).reshape(T, -1))
            wo = (self.w_out * self.m_out).reshape(T, D, P, H)
            wo = torch.nn.functional.pad(wo, (0, 0, 0, 64 - P))
            parts.append(wo.reshape(T, -1))
            return torch.cat(parts, dim=1).contiguous()

    # zuko-style names in checkpoints ------------------------------------------------
    def _zuko_items(self):
        for t in range(self.transforms):
            base = f"_flow.transform.transforms.{t}.hyper."
            yield base + "0.weight", self.w_in, (t,), self.m_in
            yield base + "0.bias", self.b_in, (t,), None
            for l in range(self.hidden_layers - 1):
                yield base + f"{2 * (l + 1)}.weight", self.w_hid, (t, l), self.m_hid
                yield base + f"{2 * (l + 1)}.bias", self.b_hid, (t, l), None
            yield base + f"{2 * self.hidden_layers}.weight", self.w_out, (t,), self.m_out
            yield base + f"{2 * self.hidden_layers}.bias", self.b_out, (t,), None

    def state_dict(self, *args, destination=None, prefix="", keep_vars=False, **kwargs):
        out = {} if destination is None else destination
        for name, tensor, idx, mask in self._zuko_items():
            value = tensor[idx]
            out[prefix + name] = value if keep_vars else value.detach().clone()
            if mask is not None:
                out[prefix + name[:-len("weight")] + "mask"] = mask[idx].bool().clone()
        for t in range(self.transforms):
            out[prefix + f"_flow.transform.transforms.{t}.order"] = torch.tensor(self._orders[t])
        out[prefix + "_flow.base.loc"] = torch.zeros(self.features)
        out[prefix + "_flow.base.scale"] = torch.ones(self.features)
        return out

    # mentflow wraps the inverted flow, zuko.flows.Flow(flow.transform.inv, flow.base) (generate/build.py:44-46), and
    # zuko keeps the wrapped transform of a LazyInverse under `.transform`: checkpoints written by the reference
    # most likely carry `_flow.transform.transform.transforms.{t}...`.  zuko is not installable here, so both
    # spellings are accepted on load (SURVEY.md 8f-2: unverified against a real zuko 1.3.1 key list).
    _ZUKO_PREFIXES = ("_flow.transform.transforms.", "_flow.transform.transform.transforms.")

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        missing = []
        with torch.no_grad():
            for name, tensor, idx, _ in self._zuko_items():
                tail = name[len(self._ZUKO_PREFIXES[0]):]
                hit = next((p + tail for p in self._ZUKO_PREFIXES if p + tail in state_dict), None)
                if hit is not None:
                    tensor[idx].copy_(state_dict[hit])
                else:
                    missing.append(name)
        if strict and missing:
            raise RuntimeError(f"missing keys in state_dict: {missing[:4]} ...")
        return torch.nn.modules.module._IncompatibleKeys(missing, [])

    # ------------------------------------------------------------------ sampling direction
    def sample_base(self, n: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """z ~ N(0, I) (generate/flows/zuko.py:15-16).  On a CUDA device the draw is the library's
        Philox kernel on torch's own generator state: bitwise the tensor ``torch.randn((n, D),
        device=...)`` returns for the same seed, and torch's generator is moved on identically."""
        dev = self.w_in.device
        if dev.type != "cuda":
            return torch.randn((int(n), self.features), dtype=torch.float32, device=dev)
        if out is None:
            out = torch.empty((int(n), self.features), dtype=torch.float32, device=dev)
        return self.rng(dev).normal_(out)

    def rng(self, device=None) -> "ops.PhiloxStream":
        dev = torch.device(device) if device is not None else self.w_in.device
        if self._rng is None or self._rng.device != dev:
            self._rng = ops.PhiloxStream(dev)
        return self._rng

    def _packed_cached(self):
        """(packed parameters, tensor-core operand images) for the current weights, rebuilt only when a
        parameter tensor was modified (in-place version counters) or moved -- sampling / evaluation
        loops with fixed weights skip a dozen small kernels per call."""
        params = (self.w_in, self.b_in, self.w_hid, self.b_hid, self.w_out, self.b_out)
        key = tuple((p.data_ptr(), p._version) for p in params) + (ops.NSF_USE_TENSOR_CORES,)
        if self._pack_key != key:
            with torch.no_grad():
                packed = self.packed_parameters()
                images = ops.nsf_direction_images(ops.NSF_USE_TENSOR_CORES, packed, self._orders, self.hidden_units,
                                                  self.hidden_layers, self.bins)
            self._pack_key, self._pack_cache = key, (packed, images)
        return self._pack_cache

    def _run(self, z: torch.Tensor, want_logq: bool, want_steps: bool = False):
        need_grad = torch.is_grad_enabled() and (z.requires_grad or self.w_in.requires_grad)
        if not need_grad and z.is_cuda:
            packed, images = self._packed_cached()
            return ops.nsf_forward(z, packed, None, self._orders, self.hidden_units, self.hidden_layers, self.bins,
                                   want_logq, want_steps, images=images)
        if self.w_in.is_cuda:
            packed, packed_om = self.packed_pair()          # one launch for both layouts
        else:
            packed, packed_om = self.packed_parameters(), (self.packed_parameters_om() if need_grad else None)
        return ops.nsf_forward(z, packed, packed_om, self._orders, self.hidden_units,
                               self.hidden_layers, self.bins, want_logq, want_steps)

    def forward(self, z: torch.Tensor) -> torch.Tensor:
        return self._run(z, False)[0]

    def forward_and_log_prob(self, z: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        x, logq, _ = self._run(z, True)
        return x, logq

    def sample(self, n: int) -> torch.Tensor:
        return self.forward(self.sample_base(n))

    def sample_and_log_prob(self, n: int) -> Tuple[torch.Tensor, torch.Tensor]:
        return self.forward_and_log_prob(self.sample_base(n))

    def forward_steps(self, z: torch.Tensor) -> List[torch.Tensor]:
        with torch.no_grad():
            _, _, steps = self._run(z, False, want_steps=True)
        return steps

    # ------------------------------------------------------------------ density direction
    def _inverse(self, x: torch.Tensor, want_logq: bool, want_steps: bool):
        if x.is_cuda:
            packed, images = self._packed_cached()      # tensor-core operand images where the shape has them
        else:
            packed, images = self.packed_parameters(), None
        return ops.nsf_inverse(x, packed, self._orders, self.hidden_units, self.hidden_layers, self.bins, want_logq,
                               want_steps, images=images)

    def inverse(self, x: torch.Tensor) -> torch.Tensor:
        return self._inverse(x, False, False)[0]

    def inverse_steps(self, x: torch.Tensor) -> List[torch.Tensor]:
        with torch.no_grad():
            return self._inverse(x, False, True)[2]

    def log_prob(self, x: torch.Tensor) -> torch.Tensor:
        return self._inverse(x, True, False)[1]
