"""Data-parallel host logic of the path (SURVEY 8e): one process per GPU, samples sharded
contiguously across ranks, weights / prototypes / prompts replicated.

Exactly two collectives exist on the path, both plain ``torch.distributed`` all-reduces
(NCCL over NVLink on the GPU box, gloo in the CPU tests):

  * prototype build: local keyed sums ``[K,512]`` fp32 + counts ``[K]`` int64 are summed
    over ranks, then divided (counts stay exact integers)      - models/proof.py:258-276
  * training step: the flat head-gradient bucket (``HeadStepRunner.flat_grads``,
    1.85 M fp32) is summed over ranks                            - models/proof.py:444

The reference has no working multi-GPU path (its ``nn.DataParallel`` wrap crashes,
models/proof.py:312-313 vs :248), so this module is new surface, not a mirror.
The graph / state-distance path is tiny (<= 60 nodes): every rank computes it redundantly
from the already all-reduced prototypes ("replicas only"), no collective.

Nothing here touches the CUDA library: the functions take the tensors the kernels
produced, so the same code runs under gloo on CPU tensors in ``tests/test_parallel_gloo.py``.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist


def world(group=None) -> Tuple[int, int]:
    """(rank, world_size); (0, 1) when torch.distributed is not initialised."""
    if not dist.is_available() or not dist.is_initialized():
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def shard_bounds(n_rows: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous [begin, end) slice of ``n_rows`` samples owned by ``rank``: the first
    ``n_rows % world_size`` ranks get one extra row (ragged batches keep every row exactly once)."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError(f"bad rank/world_size {rank}/{world_size}")
    base, extra = divmod(int(n_rows), world_size)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def shard_rows(t: torch.Tensor, rank: int, world_size: int) -> torch.Tensor:
    b, e = shard_bounds(t.shape[0], rank, world_size)
    return t[b:e]


def allreduce_prototype_sums(sums: torch.Tensor, counts: torch.Tensor, group=None):
    """In-place sum over ranks of the local keyed sums (fp32) and counts (int64).
    Counts are integers, so the global per-class counts are exact whatever the reduction order."""
    if counts.dtype != torch.int64:
        raise TypeError("counts must be int64")
    _, ws = world(group)
    if ws > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    return sums, counts


def allreduce_gradients(flat_grads: torch.Tensor, group=None, average: bool = False,
                        async_op: bool = False):
    """Sum (or mean) of the flat gradient bucket over ranks, in place.  The head's outputs are
    per-sample and every loss the learner uses is a batch mean, so callers that scale their
    cotangents by 1/global_batch want ``average=False`` (plain sum)."""
    _, ws = world(group)
    if ws == 1:
        return None
    work = dist.all_reduce(flat_grads, op=dist.ReduceOp.SUM, group=group, async_op=async_op)
    if average:
        if async_op:
            work.wait()
            work = None
        flat_grads.div_(ws)
    return work


def gather_slices(send: torch.Tensor, gathered: torch.Tensor, group=None):
    """One exchange of ``ops.ShardedLosses``: every rank's ``send`` slice into ``gathered`` in rank order
    (``all_gather_into_tensor``; the collective does no arithmetic, the next loss phase folds in rank order)."""
    _, ws = world(group)
    if ws == 1:
        gathered.copy_(send)
        return
    dist.all_gather_into_tensor(gathered, send, group=group)


def allreduce_batch_means(text_sum: torch.Tensor, proto_sum: torch.Tensor, local_rows: int, group=None):
    """PROOF ``Proof_Net.forward`` returns batch MEANS of the text / prototype rows
    (utils/inc_net.py:458-459); under data parallelism the exact single-GPU value needs the sums
    over all shards divided by the global batch.  Takes per-shard SUMS, returns global means."""
    n = torch.tensor([local_rows], dtype=torch.int64, device=text_sum.device)
    _, ws = world(group)
    if ws > 1:
        dist.all_reduce(text_sum, group=group)
        dist.all_reduce(proto_sum, group=group)
        dist.all_reduce(n, group=group)
    g = float(n.item())
    return text_sum / g, proto_sum / g


class _PeerExchange:
    """Health of a peer-memory exchange: ``_lib``, ``_hf`` (the rendezvoused flag array), ``rank`` and ``_what`` are set
    by the subclass."""

    def status(self, stream=None) -> int:
        """Synchronises ``stream`` and returns this rank's exchange status: 0 = every exchange so far completed;
        otherwise ``1 + (phase << 8) + (peer << 16)`` of the first wait that ran past the deadline
        (``TEAM_PEER_TIMEOUT_S``, default 1800 s) - the buffer then does NOT hold the exchanged data."""
        import ctypes as C
        from . import capi
        st = (stream or torch.cuda.current_stream()).cuda_stream
        out = C.c_uint32(0)
        capi.check(self._lib.team_peer_allreduce_status(int(self._hf.buffer_ptrs[self.rank]), st, C.byref(out)),
                   "team_peer_allreduce_status")
        return int(out.value)

    def check(self, stream=None):
        s = self.status(stream)
        if s:
            raise RuntimeError(f"{self._what} on rank {self.rank}: peer {(s >> 16) & 0xff} did not arrive at barrier "
                               f"{(s >> 8) & 0xff} before the deadline (TEAM_PEER_TIMEOUT_S)")


class PeerAllReduce(_PeerExchange):
    """In-place sum over the ranks of ONE fp32 buffer per GPU by a single kernel over NVLink peer memory
    (``team_peer_allreduce_f32``: two-shot, rank-ordered sum, graph-capturable) instead of an NCCL ring/tree,
    whose latency dominates at the size of the head's gradient buffer (7.4 MB).

    ``buffer`` is allocated in torch symmetric memory and mapped by every rank; hand it to
    ``HeadStepRunner(grad_buffer=...)`` so the backward writes the gradients straight into it.  torch.distributed
    (NCCL) is only used for the rendezvous that exchanges the memory handles."""

    _what = "peer all-reduce"

    def __init__(self, numel: int, device, group=None, multicast: bool = True):
        import ctypes as C
        import torch.distributed._symmetric_memory as symm
        from . import capi
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerAllReduce needs an initialised process group")
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        if self.world > 8:
            raise ValueError("PeerAllReduce: one NVSwitch box (<= 8 ranks)")
        if numel % 4:
            raise ValueError("PeerAllReduce: numel must be a multiple of 4")
        self._lib = capi.lib()
        self.numel = numel
        self.buffer = symm.empty(numel, dtype=torch.float32, device=device)
        self._flags = symm.empty(self._lib.team_peer_allreduce_flag_bytes() // 4, dtype=torch.int32, device=device)
        self.buffer.zero_()
        self._flags.zero_()
        self._hb = symm.rendezvous(self.buffer, self.group)
        self._hf = symm.rendezvous(self._flags, self.group)
        torch.cuda.synchronize(device)
        dist.barrier(self.group)                     # every rank has zeroed its flags before anyone signals
        vp8 = C.c_void_p * self.world
        self._bufs = vp8(*[int(p) for p in self._hb.buffer_ptrs])
        self._flgs = vp8(*[int(p) for p in self._hf.buffer_ptrs])
        # measured: the switch-side reduction (multimem) wins from 4 ranks up; at 2 ranks plain peer loads are faster
        mc = int(getattr(self._hb, "multicast_ptr", 0) or 0) if (multicast and self.world >= 4) else 0
        ok = torch.tensor([1 if mc else 0], device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)      # all ranks take the same path
        self.multicast_ptr = mc if int(ok.item()) else 0

    def comm_struct(self, split_at: int):
        """ctypes ``team_peer_comm`` for ``team_head_grads.comm``: the backward then sums ``buffer[:split_at]`` over the
        ranks on a side stream as soon as it is final and ``buffer[split_at:]`` after its last kernel."""
        from . import capi
        c = capi.PeerComm()
        for r in range(self.world):
            c.bufs[r] = int(self._hb.buffer_ptrs[r])
            c.flags[r] = int(self._hf.buffer_ptrs[r])
        c.multicast = self.multicast_ptr or None
        c.rank, c.world, c.n_total, c.split_at = self.rank, self.world, self.numel, int(split_at)
        return c

    def __call__(self, stream=None):
        """Enqueue the all-reduce of ``buffer`` on ``stream`` (default: the current stream); capturable."""
        from . import capi
        st = (stream or torch.cuda.current_stream()).cuda_stream
        capi.check(self._lib.team_peer_allreduce_f32(self._bufs, self._flgs, self.multicast_ptr or None, self.rank, self.world,
                                                        self.numel, st),
                   "team_peer_allreduce_f32")


class PeerAllGather(_PeerExchange):
    """All-gathers of fixed-size byte slices, one per rank in rank order, by a single kernel over NVLink peer memory
    (``team_peer_allgather``: bit-exact, graph-capturable): the exchanges between the phases of ``ops.ShardedLosses``
    inside a captured training step, where an eager NCCL call cannot sit.

    ``slice_bytes[p]`` is the size of one rank's slice of exchange ``p`` (a multiple of 16).  ``gathered[p]`` (uint8,
    ``world * slice_bytes[p]`` bytes, torch symmetric memory) is the rank's gathered buffer and ``send[p]`` its slot
    ``rank`` of it: whatever the caller writes there is what every rank finds in slot ``rank`` after ``self(p)``.
    Hand ``gathered`` to ``ops.ShardedLosses(gathered=...)`` so the loss phases write their slices in place.
    torch.distributed (NCCL) is only used for the rendezvous that exchanges the memory handles."""

    _what = "peer all-gather"

    def __init__(self, slice_bytes, device, group=None, multicast: bool = True):
        import ctypes as C
        import torch.distributed._symmetric_memory as symm
        from . import capi
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerAllGather needs an initialised process group")
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        if self.world > 8:
            raise ValueError("PeerAllGather: one NVSwitch box (<= 8 ranks)")
        self.slice_bytes = [int(n) for n in slice_bytes]
        if any(n <= 0 or n % 16 for n in self.slice_bytes):
            raise ValueError(f"PeerAllGather: slice sizes {self.slice_bytes} must be positive multiples of 16 bytes")
        self._lib = capi.lib()
        self.gathered = [symm.empty(self.world * n, dtype=torch.uint8, device=device) for n in self.slice_bytes]
        self.send = [g[self.rank * n:(self.rank + 1) * n] for g, n in zip(self.gathered, self.slice_bytes)]
        self._flags = symm.empty(self._lib.team_peer_allreduce_flag_bytes() // 4, dtype=torch.int32, device=device)
        for g in self.gathered:
            g.zero_()
        self._flags.zero_()
        self._hg = [symm.rendezvous(g, self.group) for g in self.gathered]
        self._hf = symm.rendezvous(self._flags, self.group)
        torch.cuda.synchronize(device)
        dist.barrier(self.group)                     # every rank has zeroed its flags before anyone signals
        vp8 = C.c_void_p * self.world
        self._bufs = [vp8(*[int(p) for p in h.buffer_ptrs]) for h in self._hg]
        self._flgs = vp8(*[int(p) for p in self._hf.buffer_ptrs])
        # the all-reduce's policy: multicast from 4 ranks up, and only when every buffer of every rank has the mapping
        mc = [int(getattr(h, "multicast_ptr", 0) or 0) if (multicast and self.world >= 4) else 0 for h in self._hg]
        ok = torch.tensor([1 if all(mc) else 0], device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)      # all ranks take the same path
        self.multicast_ptrs = mc if int(ok.item()) else [0] * len(mc)

    def __call__(self, p: int, stream=None):
        """Enqueue exchange ``p`` on ``stream`` (default: the current stream); capturable.  ``send[p]`` must be final."""
        from . import capi
        st = (stream or torch.cuda.current_stream()).cuda_stream
        capi.check(self._lib.team_peer_allgather(self._bufs[p], self._flgs, self.multicast_ptrs[p] or None, self.rank,
                                                 self.world, self.slice_bytes[p], st),
                   "team_peer_allgather")
