#!/usr/bin/env python
"""bench_batch.py -- batched BisectIndex / Flip solves (partition_stripe_batch) against the same problems solved one call at a
time, on one GPU.  One JSON line per row to stdout (and to the file --out names); every batch vector is asserted identical
to the single call's.  Rows (Erdos-Renyi n = m = 10^6, ~10 nonzeros per column, the C2 matrix of bench.py):

  single       one problem through cpb_partition_stripe and through a batch of one, alternating (the oracle prebuilt):
               what a batch costs a lone problem (descriptor upload, the oracle read from the table)
  k_sweep      BisectIndex(AffineConnectivityModel(0,10,1,100)) for K = 2..65: 64 sequential calls vs one batch
  copies       B in {1, 8, 32, 128, 512} copies of BisectIndex(connectivity), K = 64: B x the single call vs one batch
  flip         the Flip rows of bench_next.py (FlipBisectCost(secondary connectivity, 0.01) and FlipBisectIndex(secondary
               edge cut), Pi = Equi(A', 64)) sequentially vs as one batch of two

Oracles are built before the timed windows (their construction is the same for both forms), so the times are the solves.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import chainb200 as cp  # noqa: E402
import pyoracle as ref  # noqa: E402
from chainb200 import synth_torch  # noqa: E402

SPLIT_BISECT_INDEX, SPLIT_FLIP_BISECT_COST, SPLIT_LAZY_FLIP_BISECT_COST, SPLIT_FLIP_BISECT_INDEX = 12, 6, 7, 13


def single(ocl, method, eps, K):
    out = np.empty(K + 1, dtype=np.int64)
    con = cp.types.CConstraint()
    cp.api._check(cp.load_library().cpb_partition_stripe(ocl._h, method, ctypes.byref(con), eps, K, out.ctypes.data))
    return out


def batch(ocls, methods, eps, Ks):
    B = len(ocls)
    outs = [np.empty(K + 1, dtype=np.int64) for K in Ks]
    f = (ctypes.c_void_p * B)(*[o._h.value for o in ocls])
    m, e, k = np.array(methods, dtype=np.int32), np.array(eps, dtype=np.float64), np.array(Ks, dtype=np.int64)
    spl = (ctypes.c_void_p * B)(*[o.ctypes.data for o in outs])
    cp.api._check(cp.load_library().cpb_partition_stripe_batch(B, f, m.ctypes.data, e.ctypes.data, k.ctypes.data, spl))
    return outs


def wall(fn):
    cp.synchronize()
    t0 = time.perf_counter()
    out = fn()
    cp.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers still stand; say what is missing
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--copies", default="1,8,32,128,512")
    args = ap.parse_args()
    cp.init(0)
    lines = []

    def emit(line):
        lines.append(line)
        print(json.dumps(line), flush=True)

    cap = cp.partition_stripe_batch_capacity()
    emit({"row": "device", "gpu": gpu_info(), "batch_kernel_max_active_clusters": cap})
    A = synth_torch.erdos_renyi(args.n, 10)
    dA = cp.device_matrix(A)
    net = cp.AffineConnectivityModel(0, 10, 1, 100)
    o_net = cp.oracle_stripe(net, dA)
    Pi = ref.partition_stripe(ref.adjointpattern(A), 64, cp.EquiSplitter())
    o_sc = cp.oracle_stripe(cp.AffineSecondaryConnectivityModel(0, 10, 1, 0, 100), dA, Pi)
    o_se = cp.oracle_stripe(cp.AffineSecondaryEdgeCutModel(0, 10, 1, 100), dA, Pi)

    # single problems: the one-call path against a batch of one, alternating
    for name, ocl, method, eps in (("bisect_index", o_net, SPLIT_BISECT_INDEX, 0.0), ("secondary_conn FlipBisectCost 0.01", o_sc, SPLIT_FLIP_BISECT_COST, 0.01),
                                   ("secondary_edge FlipBisectIndex", o_se, SPLIT_FLIP_BISECT_INDEX, 0.0)):
        want = single(ocl, method, eps, 64)
        assert np.array_equal(batch([ocl], [method], [eps], [64])[0], want)
        ts, tb = [], []
        for _ in range(args.reps):
            t, g = wall(lambda: single(ocl, method, eps, 64)); ts.append(t); assert np.array_equal(g, want)
            t, g = wall(lambda: batch([ocl], [method], [eps], [64])); tb.append(t); assert np.array_equal(g[0], want)
        emit({"row": "single", "case": name, "K": 64, "single_call_ms": ts, "batch_of_one_ms": tb,
              "single_call_median_ms": float(np.median(ts)), "batch_of_one_median_ms": float(np.median(tb)), "identical": True})

    # K sweep 2..65 on one oracle
    Ks = list(range(2, 66))
    seq = [single(o_net, SPLIT_BISECT_INDEX, 0.0, K) for K in Ks]
    t_seq, seq = wall(lambda: [single(o_net, SPLIT_BISECT_INDEX, 0.0, K) for K in Ks])
    batch([o_net] * len(Ks), [SPLIT_BISECT_INDEX] * len(Ks), [0.0] * len(Ks), Ks)
    t_bat, got = wall(lambda: batch([o_net] * len(Ks), [SPLIT_BISECT_INDEX] * len(Ks), [0.0] * len(Ks), Ks))
    same = all(np.array_equal(a, b) for a, b in zip(seq, got))
    assert same
    emit({"row": "k_sweep", "case": "BisectIndex(AffineConnectivityModel(0,10,1,100)), K = 2..65", "n": A.n, "nnz": A.nnz, "B": len(Ks),
          "sequential_ms": t_seq, "batch_ms": t_bat, "speedup": t_seq / t_bat, "identical": same})

    # B copies of the C2-size problem
    want = single(o_net, SPLIT_BISECT_INDEX, 0.0, 64)
    t_one = min(wall(lambda: single(o_net, SPLIT_BISECT_INDEX, 0.0, 64))[0] for _ in range(args.reps))
    for B in [int(b) for b in args.copies.split(",")]:
        call = lambda: batch([o_net] * B, [SPLIT_BISECT_INDEX] * B, [0.0] * B, [64] * B)
        call()
        t_bat, got = min((wall(call) for _ in range(max(1, args.reps // 2))), key=lambda x: x[0])
        same = all(np.array_equal(g, want) for g in got)
        assert same
        emit({"row": "copies", "case": "BisectIndex(connectivity), K = 64", "B": B, "single_call_ms": t_one, "sequential_ms_est": B * t_one,
              "batch_ms": t_bat, "problems_per_s_batch": B / t_bat * 1e3, "problems_per_s_sequential": 1e3 / t_one,
              "speedup": B * t_one / t_bat, "identical": same, "note": "sequential_ms_est = B x the best single call"})

    # the Flip rows of bench_next.py as one batch
    flips = [(o_sc, SPLIT_FLIP_BISECT_COST, 0.01), (o_se, SPLIT_FLIP_BISECT_INDEX, 0.0)]
    seq = [single(o, m, e, 64) for o, m, e in flips]
    t_seq, seq = wall(lambda: [single(o, m, e, 64) for o, m, e in flips])
    t_bat, got = wall(lambda: batch([o for o, _, _ in flips], [m for _, m, _ in flips], [e for _, _, e in flips], [64, 64]))
    same = all(np.array_equal(a, b) for a, b in zip(seq, got))
    r = [ref.partition_stripe(A, 64, cp.FlipBisectCostBottleneckSplitter(cp.AffineSecondaryConnectivityModel(0, 10, 1, 0, 100), 0.01), Pi).spl,
         ref.partition_stripe(A, 64, cp.FlipBisectIndexBottleneckSplitter(cp.AffineSecondaryEdgeCutModel(0, 10, 1, 100)), Pi).spl]
    same = same and all(np.array_equal(a, b) for a, b in zip(got, r))
    assert same
    emit({"row": "flip", "case": "FlipBisectCost(secondary conn, 0.01) + FlipBisectIndex(secondary edge), K = 64", "B": 2,
          "sequential_ms": t_seq, "batch_ms": t_bat, "speedup": t_seq / t_bat, "identical_to_single_and_cpu_oracle": same})

    for o in (o_net, o_sc, o_se):
        o.close()
    dA.close()
    if args.out is None:
        return
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        for line in lines:
            fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
