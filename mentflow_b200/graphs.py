"""CUDA-graph capture of the forward hot path for a fixed batch size.

The reference's trainer evaluates ``model.loss(batch_size)`` a few hundred times per epoch with the
same shapes (train/train.py:163-214, and the no-grad convergence test at :235-261).  One pass is
~25 kernel launches; at the reference's batch sizes (2.5e4-1e5 particles) the launches, not the
kernels, bound the rate (SURVEY.md 8f-1).  ``GraphedLoss`` captures one pass -- flow sample +
log-density, entropy, projections + KDE, discrepancies, loss -- into a CUDA graph and replays it.

Forward only (no autograd through a replay).  The capture is keyed on the generator's parameter
versions: after an optimiser step the next call re-captures.

Base noise that arrives in pinned host memory is copied in ``host_chunks`` pieces on a second
stream *inside* the graph, and the flow layers of piece c run while piece c+1 is still crossing
PCIe, so only the first piece's copy is exposed.
"""
from __future__ import annotations

from typing import Optional

import torch


class GraphedLoss:
    def __init__(self, model, batch_size: int, warmup: int = 2, host_chunks: int = 3) -> None:
        self.model = model
        self.batch_size = int(batch_size)
        self.warmup = max(1, int(warmup))
        self.host_chunks = max(1, int(host_chunks))
        self._host_graph = None
        self._host_key = None
        self._host_src = None
        self._host_out = None
        self._copy_stream = None
        gen = model.generator
        dev = next(gen.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("GraphedLoss needs a CUDA model; mentflow_b200 has no CPU fallback")
        self.device = dev
        from . import _lib
        # particles one launch of the flow kernel processes per pass over the SMs (one 128-row tile
        # per compute warpgroup, three per SM): pieces of whole waves leave no ragged tail per piece
        self._wave = max(1, _lib.load().mfb_sm_count()) * 3 * 128
        zdim = getattr(gen, "input_features", None) or gen.features   # the NN generator's noise is not x-sized
        self.z = torch.empty((self.batch_size, zdim), dtype=torch.float32, device=dev)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self._key = None
        self._held = None
        self.out = None
        # second capture with the base-noise draw inside (``__call__()`` without z): the library's Philox
        # kernel reads torch's generator state from a device tensor and advances it itself
        self._rng_graph: Optional[torch.cuda.CUDAGraph] = None
        self._rng_key = None
        self._rng_out = None
        self._rng = None

    def _step(self):
        gen = self.model.generator
        x, logq = gen.forward_and_log_prob(self.z)
        return self.model.loss_from_particles(x, logq)

    def _weights_key(self):
        # checked on every call: the parameter list is walked once per generator object, not per step
        gen = self.model.generator
        cached = getattr(self, "_param_list", None)
        if cached is None or cached[0] is not gen:
            cached = self._param_list = (gen, list(gen.parameters()))
        return tuple((p.data_ptr(), p._version) for p in cached[1]) + (float(self.model.penalty_parameter),)

    def _capture(self) -> None:
        gen = self.model.generator
        with torch.cuda.device(self.device), torch.no_grad():
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(self.warmup):
                    self._step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            # the packed weights / operand images are built during warm-up (outside the graph) and
            # must outlive it
            self._held = getattr(gen, "_pack_cache", None)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.out = self._step()
        self._key = self._weights_key()

    def _step_draw(self):
        self.model.generator.sample_base(self.batch_size, out=self.z)
        return self._step()

    def _capture_draw(self) -> None:
        gen = self.model.generator
        self._rng = gen.rng(self.device)
        with torch.cuda.device(self.device), torch.no_grad():
            rng_mark = self._rng.mark()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(self.warmup):
                    self._step_draw()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self._rng.rewind(rng_mark)     # the warm-up passes leave torch's random stream where it was
            self._held_rng = getattr(gen, "_pack_cache", None)
            self._rng.begin_capture()
            self._rng_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._rng_graph):
                self._rng_out = self._step_draw()
            self._rng_increment = self._rng.captured_increment
        self._rng_key = self._weights_key()

    # ---- pinned host input: chunked copies overlapped with the flow -------------------------------
    def _chunk_bounds(self):
        """Pieces of growing size (1 : 3 : 5 : 5 ...): only the first copy is exposed, so it is the
        small one (PCIe moves a piece about twice as fast as the flow consumes it).  Boundaries fall
        on whole waves of the flow kernel when the batch is large enough, else on 128-row tiles;
        either keeps every slice 16-byte aligned."""
        n, c = self.batch_size, self.host_chunks
        if c == 1 or n < 8 * 128:
            return [(0, n)]
        unit = getattr(self, "_wave", 128)
        if n < 4 * c * unit:
            unit = 128
        weights = ([1, 3] + [5] * (c - 2))[:c]
        total = sum(weights)
        bounds, a = [], 0
        for i, w in enumerate(weights):
            b = n if i == len(weights) - 1 else min(n, (a + n * w // total + unit - 1) // unit * unit)
            if b > a:
                bounds.append((a, b))
            a = b
        return bounds

    def _step_from_host(self, z_host):
        gen = self.model.generator
        cur = torch.cuda.current_stream()
        cp = self._copy_stream
        cp.wait_stream(cur)
        xs, lqs = [], []
        for a, b in self._chunk_bounds():
            with torch.cuda.stream(cp):
                self.z[a:b].copy_(z_host[a:b], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(cp)
            cur.wait_event(ev)
            x_c, lq_c = gen.forward_and_log_prob(self.z[a:b])
            xs.append(x_c)
            lqs.append(lq_c)
        cur.wait_stream(cp)
        if len(xs) == 1:
            x, logq = xs[0], lqs[0]
        else:   # a generator without a density returns log q = None
            x, logq = torch.cat(xs), (None if lqs[0] is None else torch.cat(lqs))
        return self.model.loss_from_particles(x, logq)

    def _capture_host(self, z_host) -> None:
        gen = self.model.generator
        with torch.cuda.device(self.device), torch.no_grad():
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(self.warmup):
                    self._step_from_host(z_host)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self._held_host = getattr(gen, "_pack_cache", None)
            self._host_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._host_graph):
                self._host_out = self._step_from_host(z_host)
        self._host_key = self._weights_key()
        self._host_src = z_host     # the graph reads this very buffer on every replay

    def __call__(self, z: Optional[torch.Tensor] = None):
        """(L, H, [D_k]) of one pass.  ``z``: base noise (device or pinned host tensor of shape
        (batch_size, D)); None draws it on the device.  A pinned host tensor is bound to the graph
        on first use: refill the same tensor for the following steps."""
        if z is not None and not z.is_cuda and z.is_pinned() and z.is_contiguous() and z.dtype == torch.float32:
            if (self._host_graph is None or self._host_key != self._weights_key()
                    or self._host_src is None or self._host_src.data_ptr() != z.data_ptr()):
                self._capture_host(z)
            self._host_graph.replay()
            return self._host_out
        if z is None:
            # sample on the device inside the graph: the call the reference makes, model.loss(batch_size)
            if self._rng_graph is None or self._rng_key != self._weights_key():
                self._capture_draw()
            self._rng.captured_increment = self._rng_increment
            self._rng.sync()
            self._rng_graph.replay()
            self._rng.consumed()
            return self._rng_out
        if self.graph is None or self._key != self._weights_key():
            self._capture()
        self.z.copy_(z, non_blocking=True)
        self.graph.replay()
        return self.out


class GraphedTrainStep:
    """``zero_grad(); loss, H, D = model.loss(n); loss.backward(); optimizer.step()`` -- the body of
    the reference's training loop (train/train.py:164-169) -- as ONE CUDA-graph replay.

    The optimiser must be capturable (``torch.optim.AdamW(..., capturable=True)``; add ``fused=True`` for
    one launch instead of sixteen): its step counter then lives on the device.  The learning rate is read
    by the captured kernels from wherever the optimiser keeps it: a *tensor* ``lr`` (``AdamW(lr=torch.tensor(
    1e-3, device=...))``) is followed live, so LR schedulers keep working between replays; a Python float
    is a constant of the graph, so the step is RE-CAPTURED whenever a param group's float ``lr`` (or the
    model's penalty parameter) changes -- ``lr_scheduler.step(loss)`` of the reference trainer
    (train/train.py:205-207) is therefore honoured either way.
    The warm-up passes a capture needs run real optimiser steps; parameters and optimiser state are
    snapshotted before and restored after them, so a (re-)capture leaves the training state exactly
    where the caller had it and every counted step is one replay.
    One difference from the reference loop: a non-finite loss cannot skip the update from inside a
    graph; ``step.finite`` (a device flag refreshed by every replay) lets the caller notice.
    """

    def __init__(self, model, optimizer, batch_size: int, warmup: int = 3) -> None:
        self.model, self.optimizer = model, optimizer
        self.batch_size = int(batch_size)
        dev = next(model.generator.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("GraphedTrainStep needs a CUDA model; mentflow_b200 has no CPU fallback")
        for group in optimizer.param_groups:
            if not group.get("capturable", False):
                raise ValueError("GraphedTrainStep needs an optimizer constructed with capturable=True")
        self.device = dev
        self._penalty = None
        self._lrs = None
        self._rng = None
        self._rng_increment = 0
        self.graph = None
        self.out = None
        self.finite = None
        self.warmup = max(3, int(warmup))

    def _float_lrs(self):
        """the Python-float learning rates a captured graph would bake in (tensor lrs are read live)"""
        return tuple(float(g["lr"]) for g in self.optimizer.param_groups if not torch.is_tensor(g["lr"]))

    def _snapshot(self):
        params = [p.detach().clone() for g in self.optimizer.param_groups for p in g["params"]]
        state = {}
        for p, st in self.optimizer.state.items():
            state[p] = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in st.items()}
        return params, state

    def _restore(self, snap) -> None:
        params, state = snap
        with torch.no_grad():
            i = 0
            for g in self.optimizer.param_groups:
                for p in g["params"]:
                    p.copy_(params[i])
                    i += 1
            for p, st in list(self.optimizer.state.items()):
                if p not in state:            # state created by the warm-up: back to "never stepped"
                    for k, v in st.items():
                        if torch.is_tensor(v):
                            v.zero_()
                    continue
                for k, v in st.items():
                    if torch.is_tensor(v):
                        v.copy_(state[p][k])
                    else:
                        st[k] = state[p][k]

    def _body(self):
        L, H, D = self.model.loss(self.batch_size)
        L.backward()
        self.optimizer.step()
        return L.detach(), H.detach() if torch.is_tensor(H) else H, [d.detach() for d in D]

    def _capture(self) -> None:
        gen = self.model.generator
        self._rng = gen.rng(self.device) if hasattr(gen, "rng") else None
        with torch.cuda.device(self.device):
            snap = self._snapshot()
            rng_mark = self._rng.mark() if self._rng is not None else None
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(self.warmup):
                    self.optimizer.zero_grad(set_to_none=True)
                    self._body()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self._restore(snap)
            if self._rng is not None:
                self._rng.rewind(rng_mark)
                self._rng.begin_capture()
            self.graph = torch.cuda.CUDAGraph()
            self.optimizer.zero_grad(set_to_none=True)
            with torch.cuda.graph(self.graph):
                self.out = self._body()
                self.finite = torch.isfinite(self.out[0])
            self._rng_increment = self._rng.captured_increment if self._rng is not None else 0
        self._penalty = float(self.model.penalty_parameter)
        self._lrs = self._float_lrs()

    def __call__(self):
        """One optimisation step; returns (L, H, [D_k]) of the batch it was taken on (static tensors,
        overwritten by the next call)."""
        if (self.graph is None or self._penalty != float(self.model.penalty_parameter)
                or self._lrs != self._float_lrs()):
            self._capture()     # penalty parameter and float learning rates are constants of the graph
        if self._rng is not None:
            self._rng.captured_increment = self._rng_increment
            self._rng.sync()
        self.graph.replay()
        if self._rng is not None:
            self._rng.consumed()
        return self.out
