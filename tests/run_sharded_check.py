"""(-m gpu suites cannot start several ranks; this script is the N-GPU check, run by hand / by the round's GPU calls.)
Run under torchrun on N GPUs of one box:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29512 tests/run_sharded_check.py
Checks that the library's sharded solve (cp.partition_stripe_sharded: links by blocks of CSC positions, the bisection's
threshold tree over the ranks) returns the single-GPU / CPU-oracle split vector, and times it against one GPU (resident
matrices, max over ranks)."""
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import chainb200 as cp  # noqa: E402
from chainb200 import parallel, synth, synth_torch  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    cp.init(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    f = cp.AffineConnectivityModel(0, 10, 1, 100)
    sym = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 4)
    n2 = int(os.environ.get("CPB_SHARD_N", 1_000_000))
    # (name, matrix, K, method, compare with the CPU oracle too)
    cases = [("small ER", synth.erdos_renyi(30000, 10), 16, cp.BisectCostBottleneckSplitter(f, 0.01), True),
             ("RGG, LazyBisect(sym)", synth.random_geometric(20000), 32, cp.LazyBisectCostBottleneckSplitter(sym, 0.1), True),
             ("R-MAT 14", synth.rmat(14, 16 << 14), 128, cp.LazyBisectCostBottleneckSplitter(f, 0.01), True),
             ("banded", synth.banded(3000, 20), 5, cp.LazyBisectCostBottleneckSplitter(cp.AffineConnectivityModel(0.0, 3.0, 1.0, 7.0), 0.05), True),
             ("empty", cp.SparseMatrixCSC(4, 3, [1, 1, 1, 1], np.zeros(0, dtype=np.int64)), 2, cp.LazyBisectCostBottleneckSplitter(f, 0.1), True),
             (f"C2: ER n={n2}, K=64, BisectCost eps=0.01", synth_torch.erdos_renyi(n2, 10), 64, cp.BisectCostBottleneckSplitter(f, 0.01), False),
             ("R-MAT scale 20, K=1024, LazyBisect eps=0.01", synth_torch.rmat(20, 16 << 20), 1024, cp.LazyBisectCostBottleneckSplitter(f, 0.01), False)]
    ok = True
    # the C-ABI sharded solve with the library-owned communicator (csrc/sharded.cu)
    comm = parallel.library_communicator(cp, dist, rank, world)
    for name, A, K, mtd, check_cpu in cases:
        single = cp.partition_stripe(A, K, mtd)
        shard = cp.partition_stripe_sharded(A, K, mtd, comm=comm)
        sh = cp.ShardedMatrix(A, comm)
        shard2 = cp.partition_stripe_sharded(sh, K, mtd)
        stats = cp.sharded_stats()
        same = np.array_equal(single.spl, shard.spl) and np.array_equal(single.spl, shard2.spl)
        if check_cpu and rank == 0:
            import pyoracle as ref

            same = same and np.array_equal(ref.partition_stripe(A, K, mtd).spl, shard.spl)
        # one GPU on a resident device matrix vs all ranks on the resident sharded matrix (max over ranks)
        dA = cp.device_matrix(A)
        times = {}
        for label, fn in (("single_gpu_ms", lambda: cp.partition_stripe(dA, K, mtd)), ("sharded_ms", lambda: cp.partition_stripe_sharded(sh, K, mtd))):
            best = 1e9
            for _ in range(5):
                dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                cp.synchronize()
                best = min(best, (time.perf_counter() - t0) * 1e3)
            times[label] = parallel.max_over_ranks([best], device="cuda")[0]
        dA.close()
        sh.close()
        flags = torch.tensor([int(same)], device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        ok = ok and bool(flags.item())
        if rank == 0:
            print(json.dumps({"case": name, "world": world, "identical_on_all_ranks": bool(flags.item()), **times, "stats": stats}), flush=True)
    comm.close()
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
