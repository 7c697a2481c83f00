#!/usr/bin/env python
"""bench.py -- the hot path of ChainPartitioners.jl on B200, measured per the driver contract.

Headline workload: BASELINE.json configs[2] (C3) -- R-MAT scale 24 (16M x 16M, ~2.6e8 nonzeros), K = 1024,
``partition_stripe(A, 1024, LazyBisectCostBottleneckSplitter(AffineConnectivityModel(0,10,1,100), 0.01))``.
It is the largest configuration that fits one GPU and the only one whose working set (1 GB link array) exceeds
the 126 MB L2, i.e. the one the HBM roofline is about; configs[1] (C2, last round's headline) and the other
configurations are measured too and reported in the ``configs`` array of the same JSON line, each with its own
resident / end-to-end time, dominant-kernel roofline, CPU-oracle time and bit-exact comparison.

A "step" is one full partition_stripe: link construction (the cost oracle's build) and the bisection probes.
``value``  times it with the CSC pattern already resident in HBM (CUDA events on the library stream);
``e2e``    times the public call with PAGEABLE host colptr/rowval (what a Julia ``Array`` is): host->device copies
           inside the timed region, split vector read back; ``e2e_pinned`` is the same from pinned host memory.
N > 1:     ONE C3 problem sharded over the N ranks behind the C ABI (library-owned NCCL communicator):
           column blocks of the link construction, threshold sets of the bisection -> strong scaling
           (``sharded`` holds the phase times and collective bytes; ``replicas`` the independent-problem throughput).

``--impl reference`` times the reference's CPU algorithm for the same call on the host cores: the C++
restatement in oracle/ (Julia is not installed in this image, so the reference itself cannot run; kind = "port",
single-threaded because the reference is).

``--dump-outputs DIR`` writes the split vectors the last timed step returned as ``DIR/<name>.npy`` (float64). The
inputs come from seeded generators, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

HEADLINE = os.environ.get("CPB_BENCH_HEADLINE", "C3")
SCALE = float(os.environ.get("CPB_BENCH_SCALE", "1.0"))  # < 1 shrinks every workload (debugging only; the line says so)
METRIC = "partition_stripe throughput (LazyBisectCostBottleneckSplitter, R-MAT scale 24, K=1024)"
UNIT = "partitions/s"

NOTES = {
    "k_probe_stream": "greedy feasibility probes of the most likely thresholds of the bisection tree, one 8-CTA cluster each; "
                      "bytes = ONE pass over the link array per launch (SURVEY 8d G4) although every threshold streams it",
    "k_probe_ring": "streaming probes, link array staged through a shared-memory ring by 1-D bulk copies (cp.async.bulk + mbarrier); "
                    "bytes = ONE pass over the link array per launch (SURVEY 8d G4)",
    "k_lt_fill": "build_links: every nonzero takes a slot of its row's segment through an atomic cursor and stores its position",
    "k_lt_link": "build_links: every slot scans its row segment for the largest position below its own and writes the link",
    "k_lt_count": "build_links: row histogram (one atomic per nonzero)",
    "k_rs_scatter": "stable radix scatter of (row, position) pairs inside build_links (rows heavier than 128 nonzeros)",
    "k_os_pass": "build_links (rows heavier than 128 nonzeros): one-sweep stable radix pass on packed (row, position) pairs, one read + one write "
                 "per 8-bit pass, tile prefixes by decoupled look-back (csrc/onesweep.cu)",
    "k_os_hist": "build_links: digit histograms of all radix passes in one sweep over the rows",
    "k_link_prev": "links from the row-sorted pairs + windowed scatter back into column order",
    "k_wm_level": "one bit level of the wavelet-matrix dominance index",
    "k_expand_columns": "column of every nonzero from the offsets (marks + running maximum per tile)",
    "k_window_hist": "pack_stripe: suffix histograms of link distance per column window",
    "k_cost_table": "pack_stripe: window cost table c(j, j') for j' - j <= w_max",
}


def load_traffic():
    """profiles/traffic.json: measured dram bytes per launch (ncu --set full), written by tools/ncu_to_traffic.py."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()
        self.active = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            if self.active.is_set():
                try:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([x.strip() for x in out.split(",")])
                except Exception:
                    pass
            self.stop_flag.wait(0.02)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def release_memory():
    gc.collect()
    try:
        import torch

        if torch.cuda.is_available():
            torch.cuda.empty_cache()
    except Exception:
        pass
    try:
        import chainb200 as cp

        cp.trim_memory()
    except Exception:
        pass


def peak_bandwidth():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return peak, src


def rooflines(prof, step_ms_total, steps, key):
    """Per-kernel achieved GB/s from the library's CUDA-event profile (algorithmic bytes per launch, SURVEY 8d)."""
    peak, peak_src = peak_bandwidth()
    traffic = load_traffic()
    tkey = traffic.get(key, {})
    kernels = {nm: v for nm, v in prof.items() if nm.startswith("k_") and v["ms"] > 0 and v["bytes"] > 0}
    out = []
    for nm in sorted(kernels, key=lambda nm: -kernels[nm]["ms"]):
        k = kernels[nm]
        ach = (k["bytes"] / 1e9) / (k["ms"] / 1e3)
        out.append({"bound": "hbm", "kernel": nm, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": tkey.get(nm), "traffic_source": traffic.get("_source") if nm in tkey else None, "peak_source": peak_src,
                    "launches_per_step": k["launches"] / max(steps, 1), "avg_launch_us": 1e3 * k["ms"] / max(k["launches"], 1),
                    "algorithmic_bytes_per_launch": k["bytes"] / max(k["launches"], 1), "share_of_step": k["ms"] / max(step_ms_total, 1e-9),
                    "note": NOTES.get(nm, "")})
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, res):
    """Writes what a caller of the timed call receives: the split vector ``spl`` of partition_stripe / pack_stripe, or
    ``Pi_spl`` and ``Phi_spl`` of partition_plaid's (Pi, Phi).  float64 holds every 1-based index exactly."""
    parts = [("Pi_spl", res[0]), ("Phi_spl", res[1])] if isinstance(res, tuple) else [("spl", res)]
    arrays = {name: np.asarray(p.spl, dtype=np.float64) for name, p in parts}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def time_workload(cp, w, M, extra, steps, warmup, flush_l2, e2e_steps=None, pinned=False):
    """-> dict(resident ms/step, e2e ms/step on pageable host arrays, profile, results)."""
    import torch

    dM = cp.device_matrix(M)
    for _ in range(max(warmup, 1)):
        w.call(cp, dM, extra)
    w.call(cp, M, extra)
    cp.synchronize()
    cp.profile_enable(True)
    cp.profile_reset()
    dev_ms = 0.0
    res = None
    for _ in range(steps):
        flush_l2()
        cp.timer_start()
        res = w.call(cp, dM, extra)
        dev_ms += cp.timer_stop()
    launches = cp.launch_count()
    prof = cp.profile_get()
    cp.profile_enable(False)
    stats = None
    try:
        stats = cp.bisect_stats()
    except Exception:
        pass
    dM.close()
    e2e_steps = steps if e2e_steps is None else e2e_steps
    samples = []
    res2 = None
    for _ in range(e2e_steps):
        flush_l2()
        t0 = time.perf_counter()
        res2 = w.call(cp, M, extra)
        cp.synchronize()
        samples.append((time.perf_counter() - t0) * 1e3)
    out = {"dev_ms": dev_ms, "steps": steps, "launches": int(launches), "prof": prof, "res": res, "res_e2e": res2, "e2e_samples": samples, "bisection": stats}
    if pinned:
        cpin = torch.from_numpy(M.colptr).pin_memory()
        rpin = torch.from_numpy(M.rowval).pin_memory()
        Mp = cp.SparseMatrixCSC(M.m, M.n, cpin.numpy(), rpin.numpy())
        w.call(cp, Mp, extra)
        ps = []
        for _ in range(max(3, min(e2e_steps, 10))):
            flush_l2()
            t0 = time.perf_counter()
            w.call(cp, Mp, extra)
            cp.synchronize()
            ps.append((time.perf_counter() - t0) * 1e3)
        out["pinned_samples"] = ps
        del Mp, cpin, rpin
    return out


def query_throughput(cp, ref, A, f, rank):
    """Cost-oracle queries/s (the other half of BASELINE.json's metric): Q = 2^24 uniform random (j <= j') pairs and the
    same pairs sorted, device-resident, on the dominance index; the CPU oracle's rate on a bounded sample beside it."""
    import torch

    Q = 1 << 24
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    qa = torch.randint(1, A.n + 2, (Q,), device="cuda", generator=g, dtype=torch.int64)
    qb = torch.randint(1, A.n + 2, (Q,), device="cuda", generator=g, dtype=torch.int64)
    qj, qjp = torch.minimum(qa, qb).contiguous(), torch.maximum(qa, qb).contiguous()
    del qa, qb
    order = torch.argsort(qj * (A.n + 2) + qjp)
    sj, sjp = qj[order].contiguous(), qjp[order].contiguous()
    del order
    qout = torch.empty(Q, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    dA = cp.device_matrix(A)
    ocl = cp.oracle_stripe(f, dA)
    ocl.query_device(qj.data_ptr(), qjp.data_ptr(), qout.data_ptr(), Q)  # builds the dominance index, warms up
    cp.synchronize()
    out = {"Q": Q}
    for name, (a, b) in (("random", (qj, qjp)), ("sorted", (sj, sjp))):
        ms = 0.0
        for _ in range(3):
            cp.timer_start()
            ocl.query_device(a.data_ptr(), b.data_ptr(), qout.data_ptr(), Q)
            ms += cp.timer_stop()
        out[name + "_queries_per_s"] = 3 * Q / (ms / 1e3)
    if ref is not None:
        nchk = 1 << 12
        ocl.query_device(qj.data_ptr(), qjp.data_ptr(), qout.data_ptr(), Q)
        cp.synchronize()
        got = qout[:nchk].cpu().numpy()
        hj, hjp = qj.cpu().numpy(), qjp.cpu().numpy()
        t0 = time.perf_counter()
        exp = ref.oracle_query(f, A, hj[:nchk], hjp[:nchk], hint=cp.SparseHint())
        t1 = time.perf_counter()
        big = 1 << 20
        ref.oracle_query(f, A, hj[:big], hjp[:big], hint=cp.SparseHint())
        t2 = time.perf_counter()
        out["identical_to_cpu_oracle"] = bool(np.array_equal(got, exp))
        out["cpu_queries_per_s"] = (big - nchk) / max((t2 - t1) - (t1 - t0), 1e-9)
        out["cpu_sample"] = f"{big} of the random pairs through the restated b-ary DominanceCount (SparseHint), build time subtracted, 1 thread"
    ocl.close()
    dA.close()
    return out


def config_entry(cp, ref, key, M, extra, steps, flush_l2, with_cpu=True):
    from chainb200.workloads import WORKLOADS

    w = WORKLOADS[key]
    t = time_workload(cp, w, M, extra, steps, 1, flush_l2, e2e_steps=steps)
    roofs = rooflines(t["prof"], t["dev_ms"], steps, key)
    entry = {"workload": w.title, **w.sizes(M), **w.describe(t["res"]), "ms_per_step": t["dev_ms"] / steps, "e2e_ms": float(np.mean(t["e2e_samples"])),
             "e2e_median_ms": float(np.median(t["e2e_samples"])), "e2e_host_memory": "pageable", "h2d_bytes": int((M.nnz + M.n + 1) * 8),
             "gpu_launches_per_step": t["launches"] / steps, "roofline": roofs[0] if roofs else None,
             "phases_ms_per_step": {nm: round(v["ms"] / steps, 4) for nm, v in t["prof"].items()}}
    if t["bisection"] and key in ("C2", "C3", "C5"):
        entry["bisection"] = t["bisection"]
    if with_cpu and ref is not None:
        t0 = time.perf_counter()
        exp = w.call(ref, M, extra)
        cpu_ms = (time.perf_counter() - t0) * 1e3
        entry["cpu_baseline"] = {"ms": cpu_ms, "cores": 1, "kind": "port", "sample": "full workload x1, C++ restatement of the Julia reference, 1 thread"}
        entry["identical"] = bool(w.same(t["res"], exp) and w.same(t["res_e2e"], exp))
        entry["speedup_e2e_vs_cpu"] = cpu_ms / entry["e2e_ms"]
    return entry


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--configs", default=os.environ.get("CPB_BENCH_CONFIGS", "all"), help="all | none | comma list of C1,C2,C4a,C4b,C5 (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the split vectors of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    from chainb200.workloads import WORKLOADS, AFF

    W = WORKLOADS[HEADLINE]
    config = {"workload": W.title + (f" [scaled by {SCALE}]" if SCALE != 1.0 else ""),
              "why_this_workload": "largest single-GPU configuration of BASELINE.json and the only one whose working set exceeds L2; "
                                   "configs[1] and the others are in `configs`",
              "l2": "inputs larger than L2 (1 GB link array); a 256 MiB write also flushes L2 between timed steps"}

    import torch

    have_cuda = torch.cuda.is_available()

    if args.impl == "reference":
        if rank != 0:
            return 0
        import pyoracle as ref

        if have_cuda:
            torch.cuda.set_device(local_rank)
        M, extra = W.make(SCALE, have_cuda)
        release_memory()
        steps = args.steps
        t0 = time.perf_counter()
        secs = [0.0, 0.0]
        for _ in range(steps):
            res = W.call(ref, M, extra)
            secs[0] += ref.last_seconds[0]
            secs[1] += ref.last_seconds[1]
        per = (time.perf_counter() - t0) / steps
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, res)
        v = 1.0 / per
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": 0,
                "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                                 "sample": f"full workload x{steps} (probe_init {secs[0]/steps*1e3:.0f} ms + probes {secs[1]/steps*1e3:.0f} ms per step); "
                                           "C++ restatement of the Julia reference (fused probe_init/probe of LazyBisectCostBottleneckSplitter.jl:140-258), 1 thread "
                                           "(the reference has no threads)"},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import chainb200 as cp

    if not have_cuda:
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    cp.init(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        cp.synchronize()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush_l2():
        flush.zero_()
        torch.cuda.synchronize()

    M, extra = W.make(SCALE, True)
    release_memory()
    sampler = ClockSampler(local_rank)
    sampler.start()

    if world > 1:
        from bench_sharded import run_sharded

        line = run_sharded(cp, dist, W, M, extra, args, rank, world, local_rank, barrier, flush_l2, sampler, config, METRIC, UNIT)
        if rank == 0:
            print(json.dumps(line))
        dist.destroy_process_group()
        return 0

    warm = max(args.warmup, 3)
    sampler.active.set()
    t = time_workload(cp, W, M, extra, args.steps, warm, flush_l2, e2e_steps=args.steps, pinned=True)
    sampler.active.clear()
    dev_ms, e2e_ms = t["dev_ms"], float(np.sum(t["e2e_samples"]))
    assert W.same(t["res"], t["res_e2e"])
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, t["res"])
    value = args.steps / (dev_ms / 1e3)
    e2e_value = args.steps / (e2e_ms / 1e3)
    roofs = rooflines(t["prof"], dev_ms, args.steps, HEADLINE)

    import pyoracle as ref

    t0 = time.perf_counter()
    exp = W.call(ref, M, extra)
    cpu_s = time.perf_counter() - t0
    identical = bool(W.same(t["res"], exp))
    assert identical, "GPU result differs from the CPU oracle"
    cpu = {"value": 1.0 / cpu_s, "unit": UNIT, "cores": 1, "kind": "port",
           "sample": f"full workload x1 ({cpu_s:.2f} s: probe_init {ref.last_seconds[0]*1e3:.0f} ms + probes {ref.last_seconds[1]*1e3:.0f} ms); "
                     "C++ restatement of the Julia reference, single thread (the reference has no threads)"}
    sizes = W.sizes(M)
    h2d = int((M.nnz + M.n + 1) * 8)
    K = int(W.describe(t["res"]).get("K", W.describe(t["res"]).get("chunks", 0)))
    del M
    release_memory()

    configs = []
    want = [] if args.configs == "none" else (["C1", "C2", "C4a", "C4b", "C5"] if args.configs == "all" else args.configs.split(","))
    queries = None
    cache = {}
    for key in want:
        w = WORKLOADS[key]
        ck = "C4" if key.startswith("C4") else key
        if ck not in cache:
            cache.clear()
            release_memory()
            cache[ck] = w.make(SCALE, True)
            release_memory()
        Mk, ek = cache[ck]
        entry = {"config": key, **config_entry(cp, ref, key, Mk, ek, args.steps, flush_l2)}
        if key == "C2":
            queries = query_throughput(cp, ref, Mk, AFF, rank)
            entry["oracle_queries"] = queries
        configs.append(entry)
    cache.clear()
    release_memory()
    sampler.stop_flag.set()
    sampler.join(timeout=2)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": warm,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic", "config": {**config, **sizes, "K": K},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms / args.steps, "median_ms_per_step": float(np.median(t["e2e_samples"])),
                    "max_ms": float(np.max(t["e2e_samples"])), "host_memory": "pageable (numpy arrays, what a Julia ccall hands over)",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int((K + 1) * 8)},
            "e2e_pinned": {"ms_per_step": float(np.mean(t["pinned_samples"])), "median_ms_per_step": float(np.median(t["pinned_samples"])),
                           "note": "same public call from pinned host arrays (not the headline)"},
            "oracle_queries_per_s": queries["random_queries_per_s"] if queries else None,
            "gpu_launches": t["launches"], "roofline": roofs[0] if roofs else None, "roofline_all_kernels": roofs, "cpu_baseline": cpu,
            "clocks": sampler.summary(), "phases_ms_per_step": {nm: round(v["ms"] / args.steps, 4) for nm, v in t["prof"].items()},
            "bisection": t["bisection"], "parity": "split vector identical to the CPU oracle", "configs": configs}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
