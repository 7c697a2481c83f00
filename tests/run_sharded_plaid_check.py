"""(-m gpu suites cannot start several ranks; this script is the N-GPU check of the sharded partition_plaid pieces.)
Run under torchrun on N GPUs of one box:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29513 tests/run_sharded_plaid_check.py
Checks on every rank, through the C ABI with the library-owned communicator (csrc/sharded.cu):
  * the sharded monotonized-symmetric stripe solve and partition_plaid_sharded equal the single-GPU results (and the CPU
    oracle's at small sizes);
  * each rank's block of the sharded transpose (ShardedMatrix.adjointpattern().to_host_block()) equals its block of
    adjointpattern(A)."""
import json
import os
import sys

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
    comm = parallel.library_communicator(cp, dist, rank, world)
    aff = cp.AffineConnectivityModel(0, 10, 1, 100)
    sym = cp.LazyBisectCostBottleneckSplitter(cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 90), 0.1)
    sym4 = cp.BisectCostBottleneckSplitter(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 7, 4), 0.01)
    z = np.zeros(0, dtype=np.int64)
    n5 = int(os.environ.get("CPB_SHARD_N", 1_000_000))
    cases = [("RGG 20000, C5 shape", synth.random_geometric(20000), 32, sym, True),
             ("ER 30000 (diagonals missing)", synth.erdos_renyi(30000, 10), 16, sym4, True),
             ("R-MAT 14 (heavy rows)", synth.rmat(14, 16 << 14), 128, sym, True),
             ("banded 3000", synth.banded(3000, 20), 5, sym4, True),
             ("laplacian5 40", synth.laplacian5(40), 7, sym, True),
             ("fewer nonzeros than ranks", cp.SparseMatrixCSC(6, 6, np.array([1, 1, 1, 1, 3, 3, 3]), np.array([1, 4])), 3, sym, True),
             ("empty 3x3", cp.SparseMatrixCSC(3, 3, np.ones(4, dtype=np.int64), z), 2, sym, True),
             (f"RGG {n5}, K=256", synth_torch.random_geometric(n5), 256, sym, False)]
    ok = True
    for name, A, K, mtd, check_cpu in cases:
        same = True
        # the monotonized-symmetric stripe solve
        single = cp.partition_stripe(A, K, mtd)
        shard = cp.partition_stripe_sharded(A, K, mtd, comm=comm)
        same = same and np.array_equal(single.spl, shard.spl)
        # plaid: alternating (C5) and a disjoint connectivity / symmetric pair
        for meth in (cp.AlternatingPartitioner(mtd, mtd), cp.DisjointPartitioner(cp.LazyBisectCostBottleneckSplitter(aff, 0.01), mtd)):
            Ps, Fs = cp.partition_plaid(A, K, meth)
            Pd, Fd = cp.partition_plaid_sharded(A, K, meth, comm=comm)
            same = same and np.array_equal(Ps.spl, Pd.spl) and np.array_equal(Fs.spl, Fd.spl)
            if check_cpu and rank == 0:
                import pyoracle as ref

                Pr, Fr = ref.partition_plaid(A, K, meth)
                same = same and np.array_equal(Pr.spl, Pd.spl) and np.array_equal(Fr.spl, Fd.spl)
        # the sharded transpose, block by block
        S = cp.ShardedMatrix(A, comm)
        T = S.adjointpattern()
        colptr, rowval, lo, hi = T.to_host_block()
        B = cp.adjointpattern(A)
        same = same and (lo, hi) == cp.shard_range(A.nnz, rank, world)
        same = same and np.array_equal(colptr, B.colptr) and np.array_equal(rowval, B.rowval[lo:hi])
        T.close()
        S.close()
        flags = torch.tensor([int(same)], device="cuda")
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        ok = ok and bool(flags.item())
        if rank == 0:
            print(json.dumps({"case": name, "world": world, "n": int(A.n), "nnz": int(A.nnz), "K": K,
                              "identical_on_all_ranks": bool(flags.item()), "cpu_oracle_checked": check_cpu}), flush=True)
    comm.close()
    dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
