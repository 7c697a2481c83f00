"""The two new sharded constructions of csrc/sharded.cu as host models over gloo (2 and 3 ranks, CPU only):

  * the A + I link blocks of the monotonized symmetric model: per-rank "diagonal present" flags combined with a MAX
    all-reduce, every rank's block [img(q_lo), img(q_hi)) of A + I positions, the block's virtual diagonals, the carried
    "last position" array and a gather of blocks of different sizes by one broadcast per rank -- compared with the links of
    the whole A + I (a virtual diagonal appended to every column that lacks one, SparseColorArrays.jl:87-91);
  * the sharded adjointpattern: row histograms all-gathered, every entry routed to the rank owning its position in the
    transpose, one contiguous slice per destination, scattered there -- compared with adjointpattern (util.jl:67-95).

The inputs include a column that straddles a block boundary with its diagonal on one side only, a boundary right after a
virtual diagonal, leading / inner / trailing empty columns, and rectangular patterns for the transpose."""
import os
import sys

import numpy as np
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _paths():
    for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)


def _square_cases():
    import chainb200 as cp
    from chainb200 import synth

    rng = np.random.default_rng(7)
    # 6 x 6, 8 nonzeros: leading empty column, no diagonal in columns 0..4, column 4 empty; with two ranks the boundary at
    # position 4 is the first element of column 3 -- right after column 2's virtual diagonal, which stays with rank 0
    m1 = cp.SparseMatrixCSC(6, 6, np.array([0, 0, 2, 4, 6, 6, 8]) + 1, np.array([0, 3, 0, 4, 0, 5, 2, 5]) + 1)
    # 7 x 7, 12 nonzeros: column 0 (no diagonal) straddles position 4, column 3 straddles position 8 with its diagonal in
    # the upper part only, empty columns inside and at the end (their diagonals trail the last element)
    m2 = cp.SparseMatrixCSC(7, 7, np.array([0, 5, 6, 6, 12, 12, 12, 12]) + 1, np.array([1, 2, 3, 4, 5, 1, 0, 1, 2, 3, 5, 6]) + 1)
    empty = cp.SparseMatrixCSC(3, 3, np.ones(4, dtype=np.int64), np.zeros(0, dtype=np.int64))
    from helpers import sprand

    return [m1, m2, empty, sprand(rng, 40, 40, 0.1), synth.laplacian5(6), synth.banded(50, 3), synth.erdos_renyi(300, 4)]


def _rect_cases():
    from helpers import sprand

    rng = np.random.default_rng(11)
    return _square_cases() + [sprand(rng, 30, 17, 0.15), sprand(rng, 9, 41, 0.2), sprand(rng, 5, 3, 0.0)]


def _links(rows, lo, hi, carry_in):
    """links (1 + position of the previous entry of the row, 0 = none) of positions [lo, hi) and the outgoing carry"""
    last = carry_in.copy()
    out = np.zeros(hi - lo, dtype=np.int64)
    for q in range(lo, hi):
        out[q - lo] = last[rows[q]]
        last[rows[q]] = q + 1
    return out, last


def _aug_direct(A):
    """0-based rows of A + I in column order (a virtual diagonal at the end of every column that lacks one)"""
    pos, row = A.colptr - 1, A.rowval - 1
    out = []
    for j in range(A.n):
        r = list(row[pos[j]:pos[j + 1]])
        if j not in r:
            r.append(j)
        out += r
    return np.array(out, dtype=np.int64)


def _img_bounds(pos, addscan, N, world, cnt):
    """A + I block boundaries: rank 0 starts at 0, img(q) = q + addscan[c(q)], img(N) = N2"""
    N2 = N + int(addscan[-1])
    out = [0]
    for r in range(1, world + 1):
        q = min(N, r * cnt)
        if q >= N:
            out.append(N2)
        else:
            c = int(np.searchsorted(pos, q, side="right")) - 1  # the largest c with pos[c] <= q: a non-empty column
            out.append(q + int(addscan[c]))
    return out


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    _paths()
    import torch
    import torch.distributed as dist

    import chainb200 as cp

    dist.init_process_group("gloo", rank=rank, world_size=world)
    results = {"aug": [], "bounds": [], "tr": []}
    # ---- A + I link blocks --------------------------------------------------------------------------------------------
    for A in _square_cases():
        pos, row, n, m, N = A.colptr - 1, A.rowval - 1, A.n, A.m, A.nnz
        lo, hi = cp.shard_range(N, rank, world)
        cnt = cp.shard_range(N, 0, world)[1]
        present = torch.zeros(max(n, 1), dtype=torch.uint8)
        for j in range(n):  # the columns that intersect the block
            a, b = max(pos[j], lo), min(pos[j + 1], hi)
            if a < b and j in row[a:b]:
                present[j] = 1
        dist.all_reduce(present, op=dist.ReduceOp.MAX)
        add = np.array([0 if present[j] else 1 for j in range(n)] + [0], dtype=np.int64)
        addscan = np.concatenate([[0], np.cumsum(add)[:-1]])
        bnd = _img_bounds(pos, addscan, N, world, cnt)
        b_lo, b_hi = bnd[rank], bnd[rank + 1]
        row2 = np.full(b_hi - b_lo, -1, dtype=np.int64)
        for q in range(lo, hi):
            c = int(np.searchsorted(pos, q, side="right")) - 1
            row2[q + addscan[c] - b_lo] = row[q]
        for j in range(n):
            if add[j]:
                d = pos[j + 1] + addscan[j + 1] - 1  # pos2[j + 1] - 1
                if b_lo <= d < b_hi:
                    row2[d - b_lo] = j
        assert (row2 >= 0).all()
        # links of the block with the "last position" carry travelling down the ranks (chain form)
        carry = torch.zeros(max(m, 1), dtype=torch.int64)
        if rank > 0:
            dist.recv(carry, src=rank - 1)
        full_rows = np.zeros(bnd[-1], dtype=np.int64)
        full_rows[b_lo:b_hi] = row2
        links, carry_out = _links(full_rows, b_lo, b_hi, carry.numpy()[:m] if m else np.zeros(0, dtype=np.int64))
        if rank + 1 < world:
            c_out = torch.zeros(max(m, 1), dtype=torch.int64)
            c_out[:m] = torch.from_numpy(carry_out)
            dist.send(c_out, dst=rank + 1)
        # the blocks differ in size: one broadcast per rank at its offset
        prev = torch.zeros(max(bnd[-1], 1), dtype=torch.int64)
        prev[b_lo:b_hi] = torch.from_numpy(links)
        for r in range(world):
            if bnd[r + 1] > bnd[r]:
                seg = prev[bnd[r]:bnd[r + 1]].clone()
                dist.broadcast(seg, src=r)
                prev[bnd[r]:bnd[r + 1]] = seg
        results["aug"].append(prev[: bnd[-1]].tolist())
        results["bounds"].append(bnd)
    # ---- sharded transpose ----------------------------------------------------------------------------------------------
    for A in _rect_cases():
        pos, row, n, m, N = A.colptr - 1, A.rowval - 1, A.n, A.m, A.nnz
        lo, hi = cp.shard_range(N, rank, world)
        cnt = cp.shard_range(N, 0, world)[1]
        col = np.searchsorted(pos, np.arange(lo, hi), side="right") - 1
        brow = row[lo:hi]
        order = np.argsort(brow, kind="stable")  # (row, column) order of the block
        srow, scol = brow[order], col[order]
        hist = torch.from_numpy(np.bincount(brow, minlength=m).astype(np.int64))
        allh = [torch.zeros(m, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(allh, hist)
        allh = np.stack([h.numpy() for h in allh])
        tot, below = allh.sum(0), allh[:rank].sum(0)
        colptrT = np.concatenate([[0], np.cumsum(tot)])
        lstart = np.concatenate([[0], np.cumsum(allh[rank])[:-1]]) if m else np.zeros(0, dtype=np.int64)
        dst = colptrT[srow] + below[srow] + (np.arange(hi - lo) - lstart[srow])
        assert (np.diff(dst) > 0).all()  # the positions increase along the sorted block: one slice per destination
        starts = [min(N, d * cnt) for d in range(world + 1)]
        off = np.searchsorted(dst, starts, side="left")
        counts = torch.from_numpy((off[1:] - off[:-1]).astype(np.int64))
        allc = [torch.zeros(world, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(allc, counts)
        allc = np.stack([c.numpy() for c in allc])  # row s: what rank s sends to every rank
        assert allc[:, rank].sum() == hi - lo
        pairs = np.stack([dst, scol], axis=1).astype(np.int64)
        reqs, bufs = [], {}
        for d in range(world):
            if d != rank and allc[rank, d]:
                reqs.append(dist.isend(torch.from_numpy(np.ascontiguousarray(pairs[off[d]:off[d + 1]])), dst=d))
        for s in range(world):
            if s != rank and allc[s, rank]:
                bufs[s] = torch.zeros((int(allc[s, rank]), 2), dtype=torch.int64)
                reqs.append(dist.irecv(bufs[s], src=s))
        for rq in reqs:
            rq.wait()
        bufs[rank] = torch.from_numpy(pairs[off[rank]:off[rank + 1]])
        blk = np.full(hi - lo, -1, dtype=np.int64)
        for s in range(world):
            if s in bufs and len(bufs[s]):
                p = bufs[s].numpy()
                blk[p[:, 0] - lo] = p[:, 1]
        assert (blk >= 0).all()
        shard = torch.zeros(max(cnt, 1), dtype=torch.int64)
        shard[: hi - lo] = torch.from_numpy(blk)
        full = [torch.zeros(max(cnt, 1), dtype=torch.int64) for _ in range(world)]
        dist.all_gather(full, shard)
        rowT = np.concatenate([f.numpy() for f in full])[:N] if N else np.zeros(0, dtype=np.int64)
        results["tr"].append((colptrT.tolist(), rowT.tolist()))
    if rank == 0:
        out.put(results)
    dist.barrier()
    dist.destroy_process_group()


def _run(world, port_base):
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = port_base + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = out.get(timeout=300)
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    return res


def _check(res, world):
    _paths()
    import chainb200 as cp
    import pyoracle as ref

    for A, got, bnd in zip(_square_cases(), res["aug"], res["bounds"]):
        rows2 = _aug_direct(A)
        exp, _ = _links(rows2, 0, len(rows2), np.zeros(A.m, dtype=np.int64))
        assert got == exp.tolist(), (A.m, A.n, world)
        assert bnd[0] == 0 and bnd[-1] == len(rows2) and all(a <= b for a, b in zip(bnd, bnd[1:]))
    for A, (colptrT, rowT) in zip(_rect_cases(), res["tr"]):
        B = ref.adjointpattern(A)
        assert colptrT == (B.colptr - 1).tolist() and rowT == (B.rowval - 1).tolist(), (A.m, A.n, world)
    # the block rule pinned on the hand-made cases
    m1, m2 = _square_cases()[:2]
    cnt = cp.shard_range(m1.nnz, 0, world)[1]
    if world == 2:
        # m1: A + I = [d0 | 0 3 d1 | 0 4 d2 | 0 5 d3 | d4 | 2 5]; rank 0 owns A positions 0..3 -> A + I 0..6 (d2 included)
        assert res["bounds"][0] == [0, 7, 13]
        assert cnt == 4
    if world == 3:
        # m2: A + I = [1 2 3 4 5 d0 | 1 | d2 | 0 1 2 3 5 6 | d4 d5 d6]; A blocks [0,4) [4,8) [8,12) -> d0 with rank 1, the
        # trailing diagonals with rank 2
        assert res["bounds"][1] == [0, 4, 10, 17]


def test_sharded_aug_links_and_transpose_two_ranks_gloo():
    _check(_run(2, 33500), 2)


def test_sharded_aug_links_and_transpose_three_ranks_gloo():
    _check(_run(3, 35600), 3)
