"""The splitters past K = 1024 (-m gpu): the branches the device code takes on the number of parts.

- The planner's upper bound on the optimal bottleneck (k_ub_splits / k_ub_count / k_ub_prepare / k_ub_apply on the
  streaming path, k_ub_index on the dominance-index path) decides results: the prewalk settles every threshold at or above
  ub (1 + eps)^2 as feasible without probing it, so a bound below the optimum c* changes the split vector.  k_ub_prepare
  and k_ub_apply walk the parts in chunks of 1024 threads, refinement runs only for K <= 4096 and n >= 4 K (and an
  unbalanced first partition), and the streaming bound is not computed at all above K = 65535.  Each case asserts which
  branch ran: the bound is >= c* (the BisectIndex optimum) where it exists and 0 where it does not, and the
  CPB_UB_DEBUG refinement lines appear or not.
- The per-threshold split vectors of k_probe_stream / k_bisect_round / k_bisect_index ((K + 2) ints per node, filled by
  blockDim-strided loops), K at and above n on the streaming path, and the DP pointer table with K >= n.
- The partition-aware models with many row parts: the part-id sort runs one 8-bit pass (K <= 256), one 10-bit pass
  (257 <= K <= 1024), two 8-bit passes (1025) and two 10-bit passes (65537), and row parts without rows or without
  nonzeros are queried and solved over.
- The sharded (emulated) streaming solve at K > 1024.

Every split vector is compared with the CPU oracle; where the oracle is slow its answers are computed on a thread pool
(ctypes releases the GIL) while the device runs.  Costs are integers or exactly representable Float64 sums far below
2^53."""
import concurrent.futures
import functools
import os

import numpy as np
import pytest

import chainb200 as cp
from chainb200 import synth

pytestmark = pytest.mark.gpu

AFF = cp.AffineConnectivityModel(0, 10, 1, 100)
F64 = cp.AffineConnectivityModel(0.5, 10.0, 1.0, 100.0)  # dyadic coefficients: every cost is an exact Float64 sum
SYM = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 4)
EPS = 0.01
UB_KMAX = 4096       # bisect.cu: the planner refines its bound for K <= UB_KMAX and n >= 4 K
UB_STREAM_KMAX = 65535  # bisect.cu: the streaming bound's counting grid has K blocks in y


@pytest.fixture(scope="module")
def pool():
    with concurrent.futures.ThreadPoolExecutor(max_workers=max(2, min(16, os.cpu_count() or 2))) as ex:
        yield ex


def exact_bottleneck(dA, K, f, Pi=None):
    """c* = bottleneck of the exact splitter (k_bisect_index)."""
    g = cp.partition_stripe(dA, K, cp.BisectIndexBottleneckSplitter(f), Pi)
    return cp.bottleneck_value(dA, g, f, Pi)


def certified_bottleneck(monkeypatch, dA, K, f, grid):
    """c* where k_bisect_index is too slow (it walks K parts per probe, hundreds of probes: 100 s at K = 16 384 on ER
    300 000): LazyBisect with eps = 1e-9 on the dominance index, without the planner (CPB_BISECT_PLAN=0: no upper bound is
    computed or used).  Every cost lies on a grid of spacing `grid`; the final bracket (c_lo, c_hi] is narrower than the
    grid and holds the result's bottleneck, which is then the only grid point above an infeasible threshold that a feasible
    partition reaches: the optimum."""
    with monkeypatch.context() as mp:
        mp.setenv("CPB_BISECT_PLAN", "0")
        mp.setenv("CPB_PROBE_STREAM", "0")
        g = cp.partition_stripe(dA, K, cp.LazyBisectCostBottleneckSplitter(f, 1e-9))
        st = cp.bisect_stats()
    v = cp.bottleneck_value(dA, g, f)
    assert st["plan_upper_bound"] == 0 and st["c_hi_final"] - st["c_lo_final"] < grid, st
    assert st["c_lo_final"] <= v <= st["c_hi_final"], (v, st)
    return v


def solve_with_stats(capfd, dA, K, mtd):
    """-> (split partition, bisect_stats(), number of '[cpb ub] step' lines the solve printed)."""
    capfd.readouterr()
    g = cp.partition_stripe(dA, K, mtd)
    st = cp.bisect_stats()
    err = capfd.readouterr().err
    return g, st, sum(1 for line in err.splitlines() if line.startswith("[cpb ub] step"))


def check_bisection(dA, K, f, g, st, c_star, stream):
    """The bound's branch and value, and the eps-bisection's bottleneck against the optimum."""
    ub = st["plan_upper_bound"]
    if K == 1 or (stream and K > UB_STREAM_KMAX):
        assert ub == 0, (K, ub)
    else:
        assert ub >= c_star > 0, (K, ub, c_star)
    v = cp.bottleneck_value(dA, g, f)
    assert c_star <= v <= c_star * (1 + EPS), (K, v, c_star)


# ------------------------------------------------------------------------------------------ streaming bisection, K > 1024
def half_banded(n, d=10):
    """n x n: the first n / 2 columns hold d random rows, column j >= n / 2 holds rows j .. j + d - 1 (mod n).  The first
    bounding partition counts every pin as a new net, so it gives the banded half far too few columns: the part costs are
    unbalanced (the costliest ~1.8x the mean share) with no column heavy enough to be a part on its own, and refinement runs."""
    rng = np.random.default_rng(n)
    h = n // 2
    c1, r1 = np.repeat(np.arange(h), d), rng.integers(0, n, h * d)
    c2 = np.repeat(np.arange(h, n), d)
    r2 = (c2 + np.tile(np.arange(d), n - h)) % n
    return synth._from_pairs(n, n, np.concatenate([r1, r2]), np.concatenate([c1, c2]))


def banded_hub(n, d=10, hub=100):
    """n x n banded (column j holds rows j .. j + d - 1 mod n) except the last column, which holds `hub` random rows.  The
    first bounding partition's LAST part holds the hub and is by far its costliest (the banded parts cost ~0.12 of their
    pin-counting weight): up to K = 4097 the bound is decided by part K - 1 alone, and every other part costs less than
    the optimum (the hub column on its own).  A bound that misses the last part falls below c*."""
    rng = np.random.default_rng(n)
    c = np.repeat(np.arange(n - 1), d)
    r = (c + np.tile(np.arange(d), n - 1)) % n
    return synth._from_pairs(n, n, np.concatenate([r, rng.choice(n, hub, replace=False)]), np.concatenate([c, np.full(hub, n - 1)]))


@functools.lru_cache(maxsize=None)
def stream_input(name):
    if name == "er300k":
        return synth.erdos_renyi(300_000, 10)
    if name == "rmat18":  # skewed degrees; at K >= 1023 the costliest first part is one hub column: the bound is exact
        return synth.rmat(18, 16 << 18)
    if name == "hub16":  # refinement runs for every K <= UB_KMAX
        return banded_hub(1 << 16)
    if name == "mixed13":  # n = 8192: n / 4 = 2048 < UB_KMAX separates the n >= 4 K condition from K <= UB_KMAX
        return half_banded(1 << 13)
    raise ValueError(name)


def stream_ks(n):
    return sorted({K for K in (1023, 1024, 1025, 2048, 4096, 4097, n // 4, n // 4 + 1, 65535, 65536, 70000) if K <= n})


STREAM_MODELS = [("conn-int", AFF, 1), ("conn-f64", F64, 0.5), ("monosym", SYM, 1)]  # (name, model, cost grid)


@pytest.mark.parametrize("mname,f,grid", STREAM_MODELS, ids=[m[0] for m in STREAM_MODELS])
@pytest.mark.parametrize("name", ["er300k", "rmat18", "hub16", "mixed13"])
def test_streaming_bisection_large_k(ref, pool, monkeypatch, capfd, name, mname, f, grid):
    """LazyBisect and BisectCost through k_probe_stream at K on both sides of the 1024-thread chunks of k_ub_prepare /
    k_ub_apply, of UB_KMAX = 4096, of n / 4 and of the 65535 limit of the streaming bound: split vectors equal the oracle's,
    the bound is >= c* (0 above 65535), and the refinement steps print exactly where they run (always inside the limits
    on the unbalanced inputs, never above UB_KMAX or below n = 4 K)."""
    monkeypatch.setenv("CPB_UB_DEBUG", "1")
    A = stream_input(name)
    dA = cp.device_matrix(A)
    Ks = stream_ks(A.n)
    unbalanced = name in ("hub16", "mixed13")
    mks = (cp.LazyBisectCostBottleneckSplitter, cp.BisectCostBottleneckSplitter)
    want = {(K, mk): pool.submit(ref.partition_stripe, A, K, mk(f, EPS)) for K in Ks for mk in mks}
    for K in Ks:
        c_star = certified_bottleneck(monkeypatch, dA, K, f, grid) if K <= UB_STREAM_KMAX else None
        for mk in mks:
            g, st, steps = solve_with_stats(capfd, dA, K, mk(f, EPS))
            tag = (name, K, mname, mk.__name__)
            assert np.array_equal(g.spl, want[K, mk].result().spl), tag
            if c_star is None:
                assert st["plan_upper_bound"] == 0, tag
            else:
                check_bisection(dA, K, f, g, st, c_star, True)
            if K > UB_KMAX or A.n < 4 * K:
                assert steps == 0, tag
            elif unbalanced:
                assert steps >= 1, tag
    dA.close()


def test_streaming_bisection_k_at_and_above_n(ref, capfd, monkeypatch):
    """K in {n - 1, n, n + 1, 2 n + 3} on a few thousand columns: empty trailing parts, every column its own part, and the
    probes' stop once every column is placed; the bound exists (K <= 65535) but is never refined (n < 4 K)."""
    monkeypatch.setenv("CPB_UB_DEBUG", "1")
    A = synth.erdos_renyi(3000, 6)
    dA = cp.device_matrix(A)
    n = A.n
    for f in (AFF, F64, SYM):
        for K in (n - 1, n, n + 1, 2 * n + 3):
            c_star = exact_bottleneck(dA, K, f)
            for mk in (cp.LazyBisectCostBottleneckSplitter, cp.BisectCostBottleneckSplitter):
                mtd = mk(f, EPS)
                g, st, steps = solve_with_stats(capfd, dA, K, mtd)
                assert np.array_equal(g.spl, ref.partition_stripe(A, K, mtd).spl), (K, f, mk.__name__)
                assert steps == 0
                check_bisection(dA, K, f, g, st, c_star, True)
    dA.close()


# ------------------------------------------------------------------------------------------ dominance-index bisection
@functools.lru_cache(maxsize=None)
def er50k():
    return synth.erdos_renyi(50_000, 10)


INDEX_MODELS = [("work", cp.AffineWorkModel(0, 10, 1)), ("envelope", cp.AffineEnvelopeModel(0, 10, 1, 1)), ("conn", AFF)]


@pytest.mark.parametrize("name,f", INDEX_MODELS, ids=[m[0] for m in INDEX_MODELS])
def test_index_bisection_large_k(ref, pool, monkeypatch, name, f):
    """k_bisect_round and k_ub_index (CPB_PROBE_STREAM=0: connectivity too) at K in {1025, 4097, 65536} (the last above
    n = 50 000): split vectors equal the oracle's, the index bound exists at every K >= 2 and is >= c*."""
    monkeypatch.setenv("CPB_PROBE_STREAM", "0")
    A = er50k()
    dA = cp.device_matrix(A)
    mks = (cp.LazyBisectCostBottleneckSplitter, cp.BisectCostBottleneckSplitter)
    Ks = (1025, 4097, 65536)
    want = {(K, mk): pool.submit(ref.partition_stripe, A, K, mk(f, EPS)) for K in Ks for mk in mks}
    for K in Ks:
        c_star = exact_bottleneck(dA, K, f)
        for mk in mks:
            g = cp.partition_stripe(dA, K, mk(f, EPS))
            st = cp.bisect_stats()
            assert np.array_equal(g.spl, want[K, mk].result().spl), (name, K, mk.__name__)
            check_bisection(dA, K, f, g, st, c_star, False)
    dA.close()


def test_bisect_index_large_k(ref, pool):
    """k_bisect_index (one cluster walks K parts per probe) at K = 1025 and 5000 against the oracle's BisectIndex."""
    A = er50k()
    dA = cp.device_matrix(A)
    cases = [(K, f) for K in (1025, 5000) for f in (AFF, cp.AffineWorkModel(0, 10, 1))]
    want = {(K, i): pool.submit(ref.partition_stripe, A, K, cp.BisectIndexBottleneckSplitter(f)) for i, (K, f) in enumerate(cases)}
    for i, (K, f) in enumerate(cases):
        g = cp.partition_stripe(dA, K, cp.BisectIndexBottleneckSplitter(f))
        assert np.array_equal(g.spl, want[K, i].result().spl), (K, f)
    dA.close()


# ------------------------------------------------------------------------------------------ partition-aware models, many row parts
PART_MODELS = [("prim-conn", cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6)), ("sec-conn", cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6)),
               ("prim-edge", cp.AffinePrimaryEdgeCutModel(0, 2, 1, 5)), ("sec-edge", cp.AffineSecondaryEdgeCutModel(0, 2, 1, 5))]


def sort_passes(K):
    """(passes, digit width) of the part-id sort: radix_sort_impl's choice for bits_for(K - 1) key bits."""
    bits = max(1, int(K - 1).bit_length())
    p8, p10 = -(-bits // 8), -(-bits // 10)
    return (p10, 10) if p10 < p8 else (p8, 8)


@functools.lru_cache(maxsize=None)
def banded_rows_matrix():
    """20 000 x 20 000, five nonzeros per column, rows 6001..9000 empty: the row parts there hold rows but no nonzeros."""
    A = synth.erdos_renyi(20_000, 5)
    keep = (A.rowval <= 6000) | (A.rowval > 9000)
    cols = np.repeat(np.arange(1, A.n + 1), np.diff(A.colptr))
    return cp.SparseMatrixCSC.from_coo(A.m, A.n, A.rowval[keep], cols[keep])


def row_partition(m, K, zero_width=()):
    """Rows 1..m in K nearly equal parts; the parts in `zero_width` (1-based) hold no rows."""
    spl = 1 + (np.arange(K + 1, dtype=np.int64) * m) // K
    for k in zero_width:
        spl[k] = spl[k - 1]  # part k empty, part k + 1 takes its rows
    return cp.SplitPartition(K, spl)


def part_cases():
    """name -> (matrix, row partition).  The last has fewer rows (3000) than parts: 62 537 of its parts are empty."""
    A = banded_rows_matrix()
    out = {}
    for K in (255, 256, 257, 1025):
        out[f"K{K}"] = (A, row_partition(A.m, K, zero_width=(2, K // 2, K // 2 + 1, K - 1)))
    out["K65537-m3000"] = (synth.erdos_renyi(4000, 5, m=3000), row_partition(3000, 65537))
    return out


def nonzeros_per_part(A, Pi):
    part = np.searchsorted(Pi.spl, A.rowval, side="right")  # 1-based part of every nonzero
    return np.bincount(part, minlength=Pi.K + 1)[1:]


def bound_reference(A, K, f, Pi):
    """bound_stripe's (c_lo, c_hi) for the partition-aware Int64 models, from the reference's formulas (PrimaryConnectivity-
    Costs.jl:31-42, PrimaryEdgeCutCosts.jl:29-40, SecondaryConnectivityCosts.jl:44-65, SecondaryEdgeCutCosts.jl:43-60) in
    exact integers."""
    c = [int(x) for x in f.coef]
    n, N = A.n, A.nnz
    if f.kind == cp.MODEL_PRIMCONN:
        nets = len(np.unique(A.rowval))
        return c[0] + (c[1] * n + c[2] * N) // K, c[0] + c[1] * n + c[2] * N + max(c[3], c[4]) * nets
    if f.kind == cp.MODEL_PRIMEDGE:
        return c[0] + (c[1] * n + min(c[2], c[3]) * N) // K, c[0] + c[1] * n + max(c[2], c[3]) * N
    size = np.diff(Pi.spl).astype(np.int64)
    pins = nonzeros_per_part(A, Pi)
    top = min(K, Pi.K)
    if f.kind == cp.MODEL_SECEDGE:
        lo = c[0] + size * c[1] + pins * min(c[2], c[3])
        hi = c[0] + size * c[1] + pins * max(c[2], c[3])
    else:
        cols = np.repeat(np.arange(A.n), np.diff(A.colptr))
        part = np.searchsorted(Pi.spl, A.rowval, side="right") - 1
        heads = np.bincount(np.unique(part * A.n + cols) // A.n, minlength=Pi.K)  # columns with a nonzero in the part
        lo = c[0] + size * c[1] + pins * c[2]
        hi = lo + heads * c[4]
    return max(0, int(lo[:top].max())), max(0, int(hi[:top].max()))


def part_queries(rng, A, Pi):
    """Random (j, j', k) over every part, plus every empty part (no rows, or rows without nonzeros) with random ranges."""
    K, n = Pi.K, A.n
    j = rng.integers(1, n + 2, 3000)
    jp = rng.integers(1, n + 2, 3000)
    k = rng.integers(1, K + 1, 3000)
    empty = np.flatnonzero(nonzeros_per_part(A, Pi) == 0) + 1
    if len(empty) > 3000:
        empty = rng.choice(empty, 3000, replace=False)
    ej = rng.integers(1, n + 2, len(empty))
    ejp = rng.integers(1, n + 2, len(empty))
    j, jp = np.concatenate([j, ej, [1, 1]]), np.concatenate([jp, ejp, [n + 1, n + 1]])
    k = np.concatenate([k, empty, [1, K]])
    return np.minimum(j, jp), np.maximum(j, jp), k, empty


def part_methods(f):
    if f.kind in (cp.MODEL_SECCONN, cp.MODEL_SECEDGE):
        return [cp.FlipBisectIndexBottleneckSplitter(f), cp.FlipBisectCostBottleneckSplitter(f, 0.1), cp.FlipBisectCostBottleneckSplitter(f, 0.001),
                cp.LazyFlipBisectCostBottleneckSplitter(f, 0.1), cp.LazyFlipBisectCostBottleneckSplitter(f, 0.001)]
    return [cp.BisectIndexBottleneckSplitter(f), cp.BisectCostBottleneckSplitter(f, 0.1), cp.BisectCostBottleneckSplitter(f, 0.01),
            cp.LazyBisectCostBottleneckSplitter(f, 0.01)]


PART_CASES = ["K255", "K256", "K257", "K1025", "K65537-m3000"]


@pytest.mark.parametrize("case", PART_CASES)
@pytest.mark.parametrize("name,f", PART_MODELS, ids=[m[0] for m in PART_MODELS])
def test_partition_aware_many_row_parts(ref, pool, case, name, f):
    """Primary / secondary connectivity and edge-cut models with K row parts: the part-id sort's passes and digit width
    (profile of k_rs_hist / rs_scan), oracle queries over every part (empty ones included), bound_stripe, bottleneck_value /
    total_value, and the BisectIndex / BisectCost / Flip splitters with K column parts."""
    A, Pi = part_cases()[case]
    K = Pi.K
    rng = np.random.default_rng(K + len(name))
    j, jp, k, empty = part_queries(rng, A, Pi)
    assert len(empty) > 0
    mtds = part_methods(f)
    if K > 4096:  # the oracle's BisectIndex over 65 537 parts takes minutes (measured); its device form runs in the streaming tests
        mtds = [m for m in mtds if not isinstance(m, cp.BisectIndexBottleneckSplitter)]
    want_q = pool.submit(ref.oracle_query, f, A, j, jp, k, Pi=Pi)
    want = [pool.submit(ref.partition_stripe, A, K, mtd, Pi) for mtd in mtds]
    dA = cp.device_matrix(A)
    ocl = cp.oracle_stripe(f, dA, Pi)
    cp.profile_enable(True)
    cp.profile_reset()
    try:
        got = ocl.query(j, jp, k)
        prof = cp.profile_get()
    finally:
        cp.profile_enable(False)
        cp.profile_reset()
    passes, db = sort_passes(K)
    tiles = -(-A.nnz // 8192)  # RS_TILE pairs per tile
    assert prof["k_rs_hist"]["launches"] == passes and prof["k_rs_scatter"]["launches"] == passes, (case, prof.get("k_rs_hist"))
    assert prof["rs_scan"]["bytes"] == passes * (1 << db) * tiles * 8, (case, db, prof.get("rs_scan"))
    assert np.array_equal(got, want_q.result()), (case, name, np.flatnonzero(got != want_q.result())[:10])
    assert cp.bound_stripe(dA, K, ocl) == bound_reference(A, K, f, Pi), (case, name)
    ocl.close()
    for mtd, w in zip(mtds, want):
        r = w.result()
        g = cp.partition_stripe(dA, K, mtd, Pi)
        assert np.array_equal(g.spl, r.spl), (case, name, type(mtd).__name__)
        for P in (g, cp.partition_stripe(A, K, cp.EquiSplitter())):
            assert cp.bottleneck_value(dA, P, f, Pi) == ref.bottleneck_value(A, P, f, Pi), (case, name)
            assert cp.total_value(dA, P, f, Pi) == ref.total_value(A, P, f, Pi), (case, name)
    dA.close()


# ------------------------------------------------------------------------------------------ DP layers with K >= n
def test_dynamic_splitters_k_at_and_above_n(ref):
    """DynamicBottleneck / DynamicTotal with K in {n - 1, n, n + 1, 2 n}: the pointer table's rows for layers past n and
    k_dp_unravel through them, against the oracle."""
    for A in (synth.erdos_renyi(300, 4), synth.rmat(8, 4 << 8)):
        n = A.n
        for f in (AFF, F64):
            for K in (n - 1, n, n + 1, 2 * n):
                for mk in (cp.DynamicBottleneckSplitter, cp.DynamicTotalSplitter):
                    g, r = cp.partition_stripe(A, K, mk(f)), ref.partition_stripe(A, K, mk(f))
                    assert np.array_equal(g.spl, r.spl), (n, K, f, mk.__name__)


def test_dynamic_bottleneck_matches_bisect_index_at_k2000():
    """n = 20 000, K = 2000 (too large for the oracle's DP): the device DP's bottleneck equals the exact splitter's."""
    A = synth.erdos_renyi(20_000, 10)
    dA = cp.device_matrix(A)
    for f in (AFF, F64):
        d = cp.partition_stripe(dA, 2000, cp.DynamicBottleneckSplitter(f))
        assert cp.bottleneck_value(dA, d, f) == exact_bottleneck(dA, 2000, f), f
    dA.close()


# ------------------------------------------------------------------------------------------ sharded emulation
def test_sharded_emulated_large_k(ref, pool):
    """partition_stripe_sharded_emulated at worlds 2 and 3 with K in {1025, 4097}: the ranks' rounds carry K + 2 split
    points per threshold."""
    A = synth.erdos_renyi(100_000, 10)
    runs = [(K, mk(f, EPS)) for K in (1025, 4097) for f in (AFF, F64) for mk in (cp.LazyBisectCostBottleneckSplitter, cp.BisectCostBottleneckSplitter)]
    want = [pool.submit(ref.partition_stripe, A, K, mtd) for K, mtd in runs]
    for (K, mtd), w in zip(runs, want):
        exp = w.result().spl
        for world in (2, 3):
            assert np.array_equal(cp.partition_stripe_sharded_emulated(A, K, mtd, world).spl, exp), (K, type(mtd).__name__, world)
