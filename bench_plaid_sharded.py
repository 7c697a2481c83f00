"""C5 (configs[4]: partition_plaid(AlternatingPartitioner(LazyBisect(MonotonizedSymmetric(0,0,1,100,90), 0.1) x2)) on the
8M-vertex random geometric graph, K = 256) on one GPU and sharded over N GPUs through the C ABI, in one call.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29514 \\
        bench_plaid_sharded.py [--steps 5] [--warmup 2] [--out result.json]

(also runs as a plain process: a world of one).  Reports, max over ranks, with L2 flushed before every timed step as
bench.py does, device events around a device synchronise:
  * single_gpu_ms: cp.partition_plaid with the pattern resident on each GPU (the transpose built inside the step);
  * sharded_ms: cp.partition_plaid_sharded with the ShardedMatrix resident (the sharded transpose inside the step);
  * e2e_ms: cp.partition_plaid_sharded from pageable Int64 host arrays (each rank uploads only its block), host clock;
  * phases from cp.profile_get() and the collective bytes (cp.sharded_stats(), last solve), and an `identical` flag over all
    ranks (sharded == single GPU == end to end).
Writes nothing unless --out is given."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import chainb200 as cp  # noqa: E402
from chainb200 import parallel, workloads  # noqa: E402


def card():
    name, limit = torch.cuda.get_device_name(), None
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        limit = float(q.stdout.strip().splitlines()[0])
    except Exception:
        pass
    return {"device": name, "power_limit_w": limit}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    cp.init(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        cp.synchronize()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush_l2():
        flush.zero_()
        torch.cuda.synchronize()

    W = workloads.WORKLOADS["C5"]
    M, _ = W.make(args.scale, True)
    K = min(256, max(2, M.n // 64))
    sym = cp.LazyBisectCostBottleneckSplitter(cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 90), 0.1)
    meth = cp.AlternatingPartitioner(sym, sym)
    comm = parallel.library_communicator(cp, dist, rank, world)

    def timed(fn, before=None):
        for _ in range(args.warmup):
            res = fn()
        barrier()
        if before:
            before()
        ms = []
        for _ in range(args.steps):
            flush_l2()
            barrier()
            cp.timer_start()
            res = fn()
            ms.append(cp.timer_stop())
        barrier()
        return res, ms

    # ---- one GPU, pattern resident ----
    dM = cp.device_matrix(M)
    single, single_ms = timed(lambda: W.call(cp, dM, None))
    dM.close()
    # ---- sharded, ShardedMatrix resident (every rank: the column offsets + its block of rowval) ----
    sA = cp.ShardedMatrix(M, comm)

    def profile_on():
        cp.profile_enable(True)
        cp.profile_reset()

    shard, shard_ms = timed(lambda: cp.partition_plaid_sharded(sA, K, meth), profile_on)
    prof = cp.profile_get()
    stats = cp.sharded_stats()
    cp.profile_enable(False)
    sA.close()
    # ---- end to end from pageable Int64 host arrays ----
    for _ in range(args.warmup):
        cp.partition_plaid_sharded(M, K, meth, comm=comm)
    e2e_ms = []
    for _ in range(args.steps):
        flush_l2()
        barrier()
        t0 = time.perf_counter()
        e2e = cp.partition_plaid_sharded(M, K, meth, comm=comm)
        cp.synchronize()
        e2e_ms.append((time.perf_counter() - t0) * 1e3)
    barrier()
    same = W.same(single, shard) and W.same(shard, e2e)
    flags = torch.tensor([int(same)], device="cuda")
    if dist is not None:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    med = [float(np.median(single_ms)), float(np.median(shard_ms)), float(np.median(e2e_ms))]
    mx = parallel.max_over_ranks(med, device="cuda") if dist is not None else med
    comm.close()
    if dist is not None:
        dist.destroy_process_group()
    if rank != 0:
        return 0
    line = {"workload": "C5", "title": W.title, "world": world, **W.sizes(M), "K": K, "steps": args.steps, "warmup": args.warmup,
            **card(), "timing": "median over steps of each rank, max over ranks; CUDA events on the library stream (e2e: host clock); "
                                "256 MiB written before every step to flush L2",
            "single_gpu_ms": mx[0], "sharded_ms": mx[1], "e2e_ms": mx[2], "speedup_sharded_vs_single": mx[0] / mx[1] if mx[1] else None,
            "identical": bool(flags.item()),
            "phases_ms_per_step": {nm: round(v["ms"] / args.steps, 4) for nm, v in prof.items()},
            "collectives_last_solve": stats}
    print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(line, f, indent=1)
    return 0 if line["identical"] else 1


if __name__ == "__main__":
    sys.exit(main())
