"""One process per GPU (torch.distributed): the two tools over sharded inputs (SURVEY.md 8(e)).

profile : read batches are sharded across ranks, the packed reference is replicated; ONE all-reduce (sum) of the int64
          accumulator vector (< 10 KB) -- NCCL over NVLink on GPUs, gloo in the CPU tests; Java's int wrap-around is
          applied after the reduction (it commutes with addition mod 2^32).
pileup  : contiguous read ranges (genome regions) per rank and no bulk collective.  The exchange step is one
          all-gather of a (valid, contig, end) triple per rank: the exclusive prefix-max of the shards' maximum
          (contig, alignment end) is each shard's carry-in, so all shards run at the same time.  The boundary clusters
          (head partial of shard s + open cluster of shard s-1) are merged by `sharding.merge_pileup_shards` where the
          cluster list is consumed.
The compute calls are parameters so that the host logic can be tested on CPU with a stand-in backend.
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence, Tuple

import numpy as np

from .sharding import merge_pileup_shards

Key = Optional[Tuple[int, int]]


def _rank_key(order: Optional[Sequence[int]]) -> Callable:
    """(contig, end) -> what orders it: (position of the contig in `order`, end).  Contigs `order` does not list come
    after the listed ones in FASTA order (Context.set_contig_order); order=None: FASTA order."""
    if order is None:
        return lambda k: k
    rank = {int(c): i for i, c in enumerate(order)}
    return lambda k: (rank.get(k[0], len(rank) + k[0]), k[1])


def exclusive_prefix_max(keys: Sequence[Key], order: Optional[Sequence[int]] = None) -> list:
    """keys[r] = (contig, end) maximum of shard r or None -> carry-in of every shard (None for shard 0 / empty prefix).
    Contigs are FASTA indices, compared by their position in `order` (the records' contig order, e.g.
    BamBatcher.contig_order; None: FASTA order)."""
    rk = _rank_key(order)
    out, best = [], None
    for k in keys:
        out.append(best)
        if k is not None and (best is None or rk(k) > rk(best)):
            best = k
    return out


class _KeyGather:
    """In-flight all-gather of one (valid, contig, end) triple per rank."""

    def __init__(self, local: Key, group=None, device=None, order=None):
        import torch
        import torch.distributed as dist
        self.group = group
        self.order = order
        world = dist.get_world_size(group)
        self.t = torch.tensor([1 if local is not None else 0, local[0] if local else 0, local[1] if local else 0],
                              dtype=torch.int64, device=device)
        self.got = torch.empty(world * 3, dtype=torch.int64, device=device)
        self.work = dist.all_gather_into_tensor(self.got, self.t, group=group, async_op=True)

    def keys(self) -> list:
        self.work.wait()
        flat = self.got.tolist()          # device -> host (synchronises the collective's stream)
        return [(int(flat[k + 1]), int(flat[k + 2])) if flat[k] else None for k in range(0, len(flat), 3)]

    def carry(self) -> Key:
        import torch.distributed as dist
        return exclusive_prefix_max(self.keys(), self.order)[dist.get_rank(self.group)]


def all_gather_keys_async(local: Key, group=None, device=None, order=None) -> _KeyGather:
    """Start the exchange; call .carry() when the carry-in is needed (other work can be queued in between).  order: the
    records' contig order (exclusive_prefix_max)."""
    return _KeyGather(local, group, device, order)


def all_gather_keys(local: Key, group=None, device=None) -> list:
    return _KeyGather(local, group, device).keys()


def gather_keys_device(key_tensor, group=None):
    """All-gather of the 1-element device key tensors of Context.pileup_max_key_tensor.  Nothing comes back to the host:
    the call is enqueued (the current stream waits for the collective) and the gathered keys stay in HBM, where
    pileup_run(carry_keys=(ptr, rank)) takes the maximum of the first `rank` of them as this shard's carry-in."""
    import torch
    import torch.distributed as dist
    out = torch.empty(dist.get_world_size(group), dtype=torch.int64, device=key_tensor.device)
    dist.all_gather_into_tensor(out, key_tensor, group=group)
    return out


def sharded_pileup_carry(local_key: Key, group=None, device=None, order=None) -> Key:
    """The carry-in of this rank's region: one all-gather of 3 scalars per rank + a prefix-max on the host (contigs
    compared in the records' contig order `order`, FASTA order when None)."""
    import torch.distributed as dist
    keys = all_gather_keys(local_key, group, device)
    return exclusive_prefix_max(keys, order)[dist.get_rank(group)]


def sharded_pileup(local_batch, max_key_fn: Callable, pileup_fn: Callable, read_offset: int, group=None, device=None,
                   gather_to: Optional[int] = 0, order=None):
    """Region-sharded T>C pileup.  max_key_fn(batch) -> Key; pileup_fn(batch, carry) -> result dict (Context.pileup).
    order: the records' contig order when it is not the FASTA's (BamBatcher.contig_order; the contexts behind
    max_key_fn / pileup_fn need the same order, Context.set_contig_order).
    Returns (local result, merged whole-stream result on rank `gather_to` else None)."""
    import torch.distributed as dist
    carry = sharded_pileup_carry(max_key_fn(local_batch), group, device, order)
    res = pileup_fn(local_batch, carry)
    merged = None
    if gather_to is not None:
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        # only the boundary pieces and the closed clusters the consumer wants travel; object collective = host path
        payload = (read_offset, res)
        got = [None] * world if rank == gather_to else None
        dist.gather_object(payload, got, dst=gather_to, group=group)
        if rank == gather_to:
            got.sort(key=lambda x: x[0])
            merged = merge_pileup_shards([g[1] for g in got], [g[0] for g in got])
    return res, merged


def allreduce_profile(acc, group=None):
    """Sum the int64 accumulator vectors of all ranks in place (torch tensor on the backend's device)."""
    import torch.distributed as dist
    dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
    return acc
