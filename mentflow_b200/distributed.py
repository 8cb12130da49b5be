"""Particle sharding across GPUs (one process per GPU, ``torch.distributed``).

Particles are i.i.d. rows, so every op up to the per-bin sums is rank-local.  The only
exchange on the forward path is ONE small all-reduce of the *unnormalised* profile sums
(K*B floats, or exact 64-bit fixed-point integers for 2-D screens / histogram counts) and of
the entropy partial sums -- it has to happen before the non-linear normalisation and KL
(SURVEY.md 8e).  Gradients of the flow parameters are summed after backward
(``allreduce_gradients``).  The k-NN entropy estimator is the exception: its neighbours live in the
union batch, so it all-gathers the particles and its per-particle results (``ShardReducer.all_gather``).
The reference has no distributed code at all.
"""
from __future__ import annotations

from typing import Iterable, List, Optional

import torch
import torch.distributed as dist


def shard_sizes(total: int, world_size: int):
    """Split ``total`` particles as evenly as possible: the first ``total % world`` ranks get
    one extra particle."""
    base, extra = divmod(int(total), int(world_size))
    return [base + (1 if r < extra else 0) for r in range(world_size)]


def shard_slice(total: int, rank: int, world_size: int) -> slice:
    sizes = shard_sizes(total, world_size)
    start = sum(sizes[:rank])
    return slice(start, start + sizes[rank])


class ShardReducer:
    """Callable handed to the fused ops: ``n_global = reducer(partial_sums, n_local)`` sums the
    tensor in place over the group.  With ``equal_shards`` (every rank holds the same number of
    particles, the weak-scaling layout) the global count needs no communication and no host
    synchronisation."""

    def __init__(self, group: Optional[dist.ProcessGroup] = None, equal_shards: bool = True):
        self.group = group
        self.equal_shards = equal_shards
        self.calls = 0
        self.bytes = 0
        self._stash = None          # float64 partial sums waiting for a float32 all-reduce to ride on
        self._stash_result = None
        self.peer = None            # PeerExchange: cross-rank sum inside the KDE tail kernel (enable_peer_exchange)

    @property
    def world_size(self) -> int:
        return dist.get_world_size(self.group) if dist.is_initialized() else 1

    def enable_peer_exchange(self) -> bool:
        """Route the forward step's cross-rank sum through the fused NVLink kernel.  Returns False (and keeps the
        NCCL path) when the ranks do not share a node with peer access or have unequal shards."""
        if self.world_size == 1 or self.world_size > 8 or not self.equal_shards or dist.get_backend(self.group) != "nccl":
            return False
        try:
            peer = PeerExchange(self.group)
            # probe: allocate and map a small block now, so that a node without peer mapping (no NVLink / P2P,
            # symmetric memory unavailable) falls back to NCCL on every rank alike instead of failing mid-step
            peer.block_for(2, 2, 0, torch.device("cuda", torch.cuda.current_device()))
            ok = torch.ones(1, device="cuda")
        except Exception:
            peer, ok = None, torch.zeros(1, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)     # all ranks or none
        self.peer = peer if bool(ok.item()) else None
        return self.peer is not None

    def take_stash(self) -> Optional[torch.Tensor]:
        m, self._stash = self._stash, None
        return m

    def set_stash_result(self, values: torch.Tensor) -> None:
        self._stash_result = values

    # ---- one packed all-reduce per forward step (SURVEY 8e) --------------------------------------
    def stash(self, values: torch.Tensor) -> None:
        """Leave a small float64 vector of partial sums to be reduced together with the next float32
        tensor that offers room for it (``tail_floats``); ``pop_result`` returns the reduced vector."""
        self._stash, self._stash_result = values, None

    def tail_floats(self) -> int:
        return 0 if self._stash is None or self.world_size == 1 else 2 * self._stash.numel()

    def pop_result(self) -> Optional[torch.Tensor]:
        res, self._stash_result = self._stash_result, None
        return res

    def global_count(self, n_local: float) -> Optional[float]:
        """particles over all ranks if that is known without communication (equal shards)"""
        if self.world_size == 1:
            return float(n_local)
        return float(n_local) * self.world_size if self.equal_shards else None

    @property
    def rank(self) -> int:
        return dist.get_rank(self.group) if dist.is_initialized() else 0

    def shard_counts(self, n_local: int, device=None) -> List[int]:
        """Particles of every rank, in rank order.  With ``equal_shards`` (or one rank) this needs no communication;
        otherwise it all-gathers the counts (one small collective and a host synchronisation).  ``device``: where the
        count tensor lives for the collective (the CUDA device for NCCL)."""
        world = self.world_size
        if world == 1 or self.equal_shards:
            return [int(n_local)] * world
        mine = torch.tensor([int(n_local)], dtype=torch.int64, device=device)
        out = torch.empty(world, dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(out, mine, group=self.group)
        return [int(c) for c in out.tolist()]

    def all_gather(self, tensor: torch.Tensor, counts: Optional[List[int]] = None) -> torch.Tensor:
        """Every rank's ``tensor`` concatenated along dim 0 in rank order (the union batch, rank r's rows starting at
        the sum of the counts of ranks 0 .. r-1).  With ``equal_shards`` it is one ``all_gather_into_tensor`` and no
        host synchronisation, so a CUDA graph can capture it.  Unequal shards take the counts (``shard_counts``,
        gathered here when not given), gather rows padded to the largest count and drop the padding.  With one rank,
        the tensor itself."""
        world = self.world_size
        if world == 1:
            return tensor
        tensor = tensor.contiguous()
        rest = tuple(tensor.shape[1:])
        if self.equal_shards:
            out = torch.empty((world * tensor.shape[0],) + rest, dtype=tensor.dtype, device=tensor.device)
            dist.all_gather_into_tensor(out, tensor, group=self.group)
            return out
        if counts is None:
            counts = self.shard_counts(tensor.shape[0], tensor.device)
        m = max(counts)
        if m == 0:
            return tensor.new_empty((0,) + rest)
        padded = tensor
        if tensor.shape[0] != m:
            padded = tensor.new_zeros((m,) + rest)
            padded[:tensor.shape[0]] = tensor
        buf = torch.empty((world * m,) + rest, dtype=tensor.dtype, device=tensor.device)
        dist.all_gather_into_tensor(buf, padded, group=self.group)
        return torch.cat([buf[r * m:r * m + c] for r, c in enumerate(counts)])

    def __call__(self, tensor: torch.Tensor, n_local: float, flat: Optional[torch.Tensor] = None) -> float:
        """``flat``: a flat float32 buffer whose head is ``tensor`` and whose last ``tail_floats()`` entries
        are free for the stashed partial sums."""
        if self.world_size == 1:
            return float(n_local)
        if flat is not None and self._stash is not None:
            from . import ops
            tail = flat[flat.numel() - 2 * self._stash.numel():]
            ops.f64_split(self._stash, tail)
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
            self._stash_result, self._stash = ops.f64_join(tail), None
            tensor = flat
        else:
            dist.all_reduce(tensor, op=dist.ReduceOp.SUM, group=self.group)
        self.calls += 1
        self.bytes += tensor.numel() * tensor.element_size()
        if self.equal_shards or n_local == 0.0:
            return float(n_local) * self.world_size
        count = torch.tensor([float(n_local)], dtype=torch.float64, device=tensor.device)
        dist.all_reduce(count, op=dist.ReduceOp.SUM, group=self.group)
        return float(count.item())


class PeerExchange:
    """Peer-mapped ("symmetric") block of every rank for the fused KDE tail (``mfb_kde1d_finish_p2p``): the ranks
    add each other's unnormalised sums through NVLink loads inside the finish kernel instead of running an NCCL
    all-reduce between deposit and tail.  torch's symmetric-memory allocator provides the mapping (one CUDA VMM
    allocation per rank, imported by all peers); the kernel, its epoch protocol and the buffers' layout are the
    library's.  ``block_for`` is collective on first use for a given screen shape (all ranks run the same program)."""

    def __init__(self, group=None) -> None:
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        self._blocks = {}

    def block_for(self, k: int, b: int, tail: int, device):
        from . import _lib
        key = (int(k), int(b), int(tail), str(device))
        hit = self._blocks.get(key)
        if hit is None:
            import torch.distributed._symmetric_memory as symm_mem
            floats = int(_lib.load().mfb_kde1d_p2p_block_floats(k, b, tail))
            block = symm_mem.empty(floats, dtype=torch.float32, device=device)
            block.zero_()
            handle = symm_mem.rendezvous(block, self.group)
            ptrs = [int(p) for p in handle.buffer_ptrs]
            state = torch.zeros(4, dtype=torch.int32, device=device)
            torch.cuda.synchronize(device)
            dist.barrier(self.group)          # every block is zeroed before anybody's first epoch arrives
            hit = self._blocks[key] = (block, handle, ptrs, state)
        return hit


def shard_model(model, group: Optional[dist.ProcessGroup] = None, equal_shards: bool = True,
                peer_exchange: bool = True) -> ShardReducer:
    """Attach a reducer to a ``MENTFlow`` model (and its entropy estimator) so that
    ``model.loss(n_local)`` returns the loss of the *global* batch on every rank, or to a classical
    ``MENT`` model so that ``gauss_seidel_update`` draws ``n_samples`` particles over all ranks."""
    reducer = ShardReducer(group, equal_shards)
    model.reducer = reducer
    if getattr(model, "entropy_estimator", None) is not None and hasattr(model.entropy_estimator, "reducer"):
        model.entropy_estimator.reducer = reducer
    if hasattr(model, "shard") and hasattr(model, "gauss_seidel_update"):
        # classical MENT: every rank draws its slice of the n_samples particles (ment.py:319-326)
        world = reducer.world_size
        model.shard = (dist.get_rank(group) if world > 1 else 0, world)
        if world > 1:
            reducer.equal_shards = False if model.n_samples % world else reducer.equal_shards
    if peer_exchange:
        # forward step: cross-rank sum inside the KDE tail kernel over NVLink peer memory (NCCL stays the path for
        # gradients, 2-D screens, histogram counts, and whenever peer mapping is not available)
        reducer.enable_peer_exchange()
    return reducer


def allreduce_gradients(params: Iterable[torch.nn.Parameter], group: Optional[dist.ProcessGroup] = None) -> None:
    """Sum parameter gradients over ranks in one flattened all-reduce (636 KB for the 6-D flow).
    Every rank back-propagates the same replicated dL/dS through its own particles, so the
    plain SUM is the gradient of the global loss."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    offset = 0
    for g in grads:
        g.copy_(flat[offset:offset + g.numel()].view_as(g))
        offset += g.numel()
