#!/usr/bin/env python
"""bench_weight_constrained.py -- constrained splitters with a count weight on one GPU, each beside the CPU oracle.

partition_stripe(B, K, method(ConstrainedCost(nets, AffineConnectivityModel(0, 0, 0, 1), w_max))) on banded n = 2^14
(synth.banded(2^14, 16, 4), the input of bench_next.py's constrained rows), K in {4, 8, 16}, method in DynamicTotalSplitter,
DynamicBottleneckSplitter and ConvexTotalSplitter.  The weight is the part's number of distinct rows; w_max is the weight of the
first ceil(1.5 n / K) columns, so the windows are about as wide as bench_next.py's VertexCount rows (w_max = ceil(1.5 n / K)).

Per case, one JSON line: the public call with the pattern resident in HBM (best of --reps), the weight_windows phase of that
call (CUDA events, profiling on, a separate run), the single-threaded CPU oracle on the same input (tests/weighted_oracle.py),
and whether the split vectors are identical (asserted).  The device name and power limit are recorded with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import chainb200 as cp  # noqa: E402
import pyoracle as ref  # noqa: E402
import weighted_oracle as wref  # noqa: E402  (the CPU oracle's constrained splitters with a count weight)
from chainb200 import synth  # noqa: E402


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
        return {"device": name, "power_limit": power}
    except Exception as e:  # the numbers are still reported; say why the device line is missing
        return {"device": "unknown", "power_limit": "unknown", "error": str(e)}


def timed(fn, reps):
    best, out = None, None
    for _ in range(reps):
        cp.synchronize()
        t0 = time.perf_counter()
        out = fn()
        cp.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 14)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--Ks", default="4,8,16")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()
    cp.init(0)
    info = device_info()
    B = synth.banded(args.n, 16, 4)
    dB = cp.device_matrix(B)
    f = cp.AffineConnectivityModel(0, 0, 0, 1)
    w = cp.AffineConnectivityModel(0, 0, 0, 1)
    lines = []
    for K in [int(k) for k in args.Ks.split(",")]:
        width = int(np.ceil(1.5 * B.n / K))
        w_max = int(ref.oracle_query(w, B, [1], [1 + width])[0])
        for mk in (cp.DynamicTotalSplitter, cp.DynamicBottleneckSplitter, cp.ConvexTotalSplitter):
            mtd = mk(cp.ConstrainedCost(f, w, w_max))
            cp.partition_stripe(dB, K, mtd)  # warm-up: module load, pools
            t_res, g = timed(lambda: cp.partition_stripe(dB, K, mtd), args.reps)
            cp.profile_reset()
            cp.profile_enable(True)
            cp.partition_stripe(dB, K, mtd)
            cp.synchronize()
            prof = cp.profile_get()
            cp.profile_enable(False)
            t0 = time.perf_counter()
            r = wref.partition_stripe(B, K, mtd)
            t_cpu = (time.perf_counter() - t0) * 1e3
            same = bool(np.array_equal(g.spl, r.spl))
            ww = prof.get("weight_windows", {})
            line = {"case": f"{mk.__name__}(ConstrainedCost(nets, nets, w_max))", "n": B.n, "nnz": B.nnz, "K": K, "window_columns": width,
                    "w_max": w_max, "gpu_resident_ms": t_res, "weight_windows_ms": ww.get("ms"), "weight_windows_bytes": ww.get("bytes"),
                    "dp_layer_ms": prof.get("dp_layer", {}).get("ms"), "oracle_stripe_ms": prof.get("oracle_stripe", {}).get("ms"),
                    "cpu_oracle_ms": t_cpu, "identical": same, **info}
            lines.append(line)
            print(json.dumps(line), flush=True)
            assert same, (mk.__name__, K, g.spl, r.spl)
    dB.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
