"""Multi-GPU plumbing around ``torch.distributed``, one process per GPU (NCCL on a GPU machine, gloo in the CPU tests).

- Independent problems (SURVEY.md section 8e: stripe solves on different matrices / the two sides of a plaid alternation
  share nothing) are dealt to the ranks round-robin; results and device timings are combined with one small collective.
- ONE stripe solve over several GPUs runs inside the library (``cp.partition_stripe_sharded``, NCCL owned by the
  library); ``library_communicator`` creates that communicator from the host framework's process group.
"""
from __future__ import annotations

from typing import List, Sequence

import numpy as np
import torch
import torch.distributed as dist


def my_problems(n_problems: int, rank: int, world: int) -> List[int]:
    """Round-robin assignment of independent problems to ranks (weak scaling: n_problems = c * world)."""
    return list(range(rank, n_problems, world))


def max_over_ranks(values: Sequence[float], device="cpu") -> List[float]:
    """Element-wise MAX over ranks (the step time of a multi-GPU run is the slowest rank's)."""
    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def gather_split_vectors(local: dict, n_problems: int, K: int, device="cpu") -> np.ndarray:
    """All ranks contribute {problem index: spl[K+1]}; every rank gets the (n_problems, K+1) table."""
    table = torch.zeros((n_problems, K + 1), dtype=torch.int64, device=device)
    for idx, spl in local.items():
        table[idx] = torch.as_tensor(np.asarray(spl, dtype=np.int64), device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(table, op=dist.ReduceOp.SUM)  # disjoint rows: SUM == gather
    return table.cpu().numpy()


def library_communicator(cp, dist_mod, rank: int, world: int):
    """Creates the library-owned NCCL communicator (``cp.Communicator``) on every rank: rank 0 makes the 128-byte id, the
    ranks receive it through the host framework's own process group (any transport would do -- the id is just bytes)."""
    uid = [cp.Communicator.unique_id() if rank == 0 else None]
    if world > 1:
        dist_mod.broadcast_object_list(uid, src=0)
    return cp.Communicator(uid[0], rank, world)
