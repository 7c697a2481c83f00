"""The N > 1 path on CPU: world_size-2 gloo run of the host-side sharding logic (problem assignment,
max-over-ranks timing, split-vector gathering) with the CPU oracle standing in for the per-rank solve."""
import os
import sys

import numpy as np
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist

    import chainb200 as cp
    import pyoracle as ref
    from chainb200 import parallel, synth

    dist.init_process_group("gloo", rank=rank, world_size=world)
    n_problems, K = 4, 8
    mine = parallel.my_problems(n_problems, rank, world)
    mtd = cp.LazyBisectCostBottleneckSplitter(cp.AffineConnectivityModel(0, 10, 1, 100), 0.01)
    local = {i: ref.partition_stripe(synth.erdos_renyi(400 + 100 * i, 6), K, mtd).spl for i in mine}
    table = parallel.gather_split_vectors(local, n_problems, K)
    t = parallel.max_over_ranks([float(rank + 1), 10.0 - rank])
    if rank == 0:
        out.put((mine, table.tolist(), t))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_sharding_gloo():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    mine, table, t = out.get(timeout=300)
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    assert mine == [0, 2]
    assert t == [2.0, 10.0]
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import chainb200 as cp
    import pyoracle as ref
    from chainb200 import synth

    mtd = cp.LazyBisectCostBottleneckSplitter(cp.AffineConnectivityModel(0, 10, 1, 100), 0.01)
    for i in range(4):
        exp = ref.partition_stripe(synth.erdos_renyi(400 + 100 * i, 6), 8, mtd).spl
        assert table[i] == exp.tolist()


# ---------------------------------------------------------------------------------------------------
# The sharded link construction of csrc/sharded.cu as a host model over gloo: every rank owns the block of CSC positions
# cpb_shard_range gives it, links inside the block come from the block alone, the per-row "last position" array travels
# down the ranks once (send / recv), the shards are all-gathered.  The result must be the link array of the whole matrix
# (the reference's cch[], LazyBisectCostBottleneckSplitter.jl:165-175, position-valued).
# ---------------------------------------------------------------------------------------------------
def _links_model(rowval, lo, hi, carry_in, m):
    """links of positions [lo, hi) given the last position (+1) of every row left of lo; also returns the outgoing carry"""
    last = carry_in.copy()
    out = np.zeros(hi - lo, dtype=np.int64)
    for q in range(lo, hi):
        r = rowval[q] - 1
        out[q - lo] = last[r]
        last[r] = q + 1
    return out, last


def _shard_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as dist

    import chainb200 as cp
    from chainb200 import synth

    dist.init_process_group("gloo", rank=rank, world_size=world)
    A = synth.rmat(9, 16 << 9)
    N, m = A.nnz, A.m
    lo, hi = cp.shard_range(N, rank, world)
    cnt = cp.shard_range(N, 0, world)[1]
    carry = torch.zeros(m, dtype=torch.int64)
    if rank > 0:
        dist.recv(carry, src=rank - 1)
    links, carry_out = _links_model(A.rowval, lo, hi, carry.numpy(), m)
    if rank + 1 < world:
        dist.send(torch.from_numpy(carry_out), dst=rank + 1)
    shard = torch.zeros(cnt, dtype=torch.int64)
    shard[: hi - lo] = torch.from_numpy(links)
    full = torch.zeros(cnt * world, dtype=torch.int64)
    dist.all_gather_into_tensor(full, shard)
    if rank == 0:
        out.put(full[:N].tolist())
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_link_construction_protocol_gloo():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    full = out.get(timeout=300)
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    for p in (ROOT,):
        if p not in sys.path:
            sys.path.insert(0, p)
    from chainb200 import synth

    A = synth.rmat(9, 16 << 9)
    exp, _ = _links_model(A.rowval, 0, A.nnz, np.zeros(A.m, dtype=np.int64), A.m)
    assert full == exp.tolist()


def test_shard_ranges_partition_the_positions():
    for p in (ROOT,):
        if p not in sys.path:
            sys.path.insert(0, p)
    import chainb200 as cp

    for N in (0, 1, 5, 1000, 263_000_001):
        for world in (1, 2, 3, 8, 16):
            blocks = [cp.shard_range(N, r, world) for r in range(world)]
            assert blocks[0][0] == 0 and blocks[-1][1] == N
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(world - 1))
            cnt = blocks[0][1] - blocks[0][0] if N else 0
            assert all(hi - lo <= max(cnt, 0) for lo, hi in blocks) and (cnt % 4 == 0 or world == 1 or N < 4 * world)
