"""bench.py's N > 1 leg: ONE headline problem sharded over the ranks (strong scaling), plus the replica throughput.

Sharded solve = ``cp.partition_stripe_sharded`` -> ``cpb_partition_stripe_sharded`` (C ABI, library-owned NCCL
communicator): column blocks of the link construction with a last-position carry, all-gather of the link shards,
the threshold tree of every bisection round split over the ranks.  Every rank passes the same host matrix; each
uploads only its own column block of ``rowval``.
"""
import json
import time

import numpy as np


def run_sharded(cp, dist, W, M, extra, args, rank, world, local_rank, barrier, flush_l2, sampler, config, metric, unit):
    import torch

    from chainb200 import parallel

    K = min(1024, max(2, M.n // 64))
    from chainb200.workloads import AFF

    mtd = cp.LazyBisectCostBottleneckSplitter(AFF, 0.01)
    comm = parallel.library_communicator(cp, dist, rank, world)
    warm = max(args.warmup, 3)
    # ---- resident: the pattern already in HBM on every rank (each rank holds its column block + the offsets) ----
    sh = cp.ShardedMatrix(M, comm)
    for _ in range(warm):
        res = cp.partition_stripe_sharded(sh, K, mtd)
    cp.profile_enable(True)
    cp.profile_reset()
    sampler.active.set()
    barrier()
    dev_ms = 0.0
    for _ in range(args.steps):
        flush_l2()
        barrier()
        cp.timer_start()
        res = cp.partition_stripe_sharded(sh, K, mtd)
        dev_ms += cp.timer_stop()
    barrier()
    launches = cp.launch_count()
    prof = cp.profile_get()
    phases = cp.sharded_stats()
    cp.profile_enable(False)
    sh.close()
    # ---- e2e: host arrays -> every rank uploads its block, solves, reads the split vector back ----
    for _ in range(2):
        cp.partition_stripe_sharded(M, K, mtd, comm=comm)
    e2e_samples = []
    for _ in range(args.steps):
        flush_l2()
        barrier()
        t0 = time.perf_counter()
        res2 = cp.partition_stripe_sharded(M, K, mtd, comm=comm)
        cp.synchronize()
        e2e_samples.append((time.perf_counter() - t0) * 1e3)
    barrier()
    sampler.active.clear()
    e2e_ms = float(np.sum(e2e_samples))
    # ---- single-GPU time of the same problem on rank 0's GPU, for the in-run strong-scaling ratio ----
    single_ms = None
    same = bool(np.array_equal(res.spl, res2.spl))
    if rank == 0:
        dM = cp.device_matrix(M)
        one = W.call(cp, dM, extra)
        s = 0.0
        for _ in range(3):
            flush_l2()
            cp.timer_start()
            one = W.call(cp, dM, extra)
            s += cp.timer_stop()
        single_ms = s / 3
        dM.close()
        same = same and bool(np.array_equal(one.spl, res.spl))
    flags = torch.tensor([int(same)], device="cuda")
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    dev_ms_max, e2e_ms_max = parallel.max_over_ranks([dev_ms, e2e_ms], device="cuda")
    comm.close()
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    if rank != 0:
        return None
    from bench import dump_outputs, rooflines

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    roofs = rooflines(prof, dev_ms, args.steps, "C3")
    value = args.steps / (dev_ms_max / 1e3)
    return {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic", "config": {**config, **W.sizes(M), "K": K, "parallelism": f"one problem over {world} GPUs: column blocks of build_links + threshold sets of the bisection"},
            "e2e": {"value": args.steps / (e2e_ms_max / 1e3), "unit": unit, "ms_per_step": e2e_ms_max / args.steps,
                    "median_ms_per_step": float(np.median(e2e_samples)), "host_memory": "pageable",
                    "h2d_bytes_per_step": int((M.nnz // world + 2 * (M.n + 1)) * 8), "d2h_bytes_per_step": int((K + 1) * 8)},
            "gpu_launches": int(launches), "roofline": roofs[0] if roofs else None, "roofline_all_kernels": roofs,
            "sharded": {**phases, "single_gpu_ms_same_run": single_ms, "speedup_vs_single_gpu": (single_ms / (dev_ms_max / args.steps)) if single_ms else None,
                        "identical_on_all_ranks_and_to_single_gpu": bool(flags.item())},
            "cpu_baseline": None, "clocks": sampler.summary(),
            "phases_ms_per_step": {nm: round(v["ms"] / args.steps, 4) for nm, v in prof.items()}, "parity": "identical to the single-GPU split vector (checked in-run)"}
