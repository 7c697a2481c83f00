"""GPU parity tests proper (-m gpu): every call goes through the C ABI of libchainb200.so and is
compared bit-for-bit with the CPU oracle on the same inputs (split vectors and integer counts exact,
Float64 costs identical because both sides evaluate the same left-to-right sums without FMA)."""
import numpy as np
import pytest

import chainb200 as cp
from chainb200 import synth
from helpers import sprand

pytestmark = pytest.mark.gpu

AFF = cp.AffineConnectivityModel(0, 10, 1, 100)


def rand_pairs(rng, n, Q):
    j = rng.integers(1, n + 2, Q)
    jp = rng.integers(1, n + 2, Q)
    return np.minimum(j, jp), np.maximum(j, jp)


def small_matrices(fixtures):
    rng = np.random.default_rng(100)
    mats = list(fixtures.values())
    mats += [sprand(rng, m, n, p) for (m, n, p) in [(1, 1, 1.0), (1, 5, 0.5), (5, 1, 0.5), (3, 3, 0.0), (8, 8, 0.5), (40, 30, 0.2),
                                                    (30, 40, 0.2), (300, 300, 0.02), (257, 225, 0.1), (1000, 1000, 0.01)]]
    return mats


def test_adjointpattern(ref, fixtures):
    for A in small_matrices(fixtures) + [synth.erdos_renyi(20000, 10)]:
        g = cp.adjointpattern(A)
        r = ref.adjointpattern(A)
        assert np.array_equal(g.colptr, r.colptr) and np.array_equal(g.rowval, r.rowval)
        assert (g.m, g.n) == (A.n, A.m)


def test_int32_indexed_matrix(ref, fixtures):
    """cpb_matrix_create_i32 (SparseMatrixCSC{Tv, Int32}): the same device matrix as the Int64 form, and the same errors."""
    for A in small_matrices(fixtures) + [synth.erdos_renyi(20000, 10)]:
        d = cp.device_matrix_i32(A.m, A.n, A.colptr.astype(np.int32), A.rowval.astype(np.int32))
        B = d.to_host()
        assert (B.m, B.n) == (A.m, A.n) and np.array_equal(B.colptr, A.colptr) and np.array_equal(B.rowval, A.rowval)
        mtd = cp.LazyBisectCostBottleneckSplitter(AFF, 0.01)
        assert np.array_equal(cp.partition_stripe(d, 4, mtd).spl, ref.partition_stripe(A, 4, mtd).spl)
        d.close()
    with pytest.raises(cp.CpbError):
        cp.device_matrix_i32(2, 2, np.array([1, 2, 3], dtype=np.int32), np.array([1, 3], dtype=np.int32))  # row 3 of 2
    with pytest.raises(cp.CpbError):
        cp.device_matrix_i32(2, 2, np.array([1, 3, 2], dtype=np.int32), np.array([1, 2], dtype=np.int32))  # colptr not monotone


def test_color_arrays(ref, fixtures):
    rng = np.random.default_rng(101)
    for A in small_matrices(fixtures) + [synth.laplacian5(40), synth.erdos_renyi(5000, 10)]:
        j, jp = rand_pairs(rng, A.n, 500)
        j = np.concatenate([j, [1, 1, A.n + 1]])
        jp = np.concatenate([jp, [1, A.n + 1, A.n + 1]])
        assert np.array_equal(cp.pincount(A).query(j, jp), ref.pincount(A, j, jp))
        assert np.array_equal(cp.netcount(A).query(j, jp), ref.netcount(A, j, jp))
        assert np.array_equal(cp.selfnetcount(A).query(j, jp), ref.selfnetcount(A, j, jp))
        if A.m == A.n:
            assert np.array_equal(cp.dianetcount(A).query(j, jp), ref.dianetcount(A, j, jp))
            assert np.array_equal(cp.selfpincount(A).query(j, jp), ref.selfpincount(A, j, jp))


def test_link_construction_paths(ref, monkeypatch):
    """build_links has two forms -- per-row segments filled through atomic cursors (rows of <= 128 nonzeros) and the
    stable radix sort (heavier rows): net / dia-net counts and the streaming bisection must not depend on which ran."""
    rng = np.random.default_rng(102)
    light = synth.erdos_renyi(20000, 10)
    dense_row = sprand(rng, 300, 300, 0.1)
    rows = [np.unique(np.concatenate([dense_row.rowval[dense_row.colptr[j] - 1:dense_row.colptr[j + 1] - 1], [7]])) for j in range(dense_row.n)]
    heavy = cp.SparseMatrixCSC(300, 300, np.cumsum([1] + [len(r) for r in rows]), np.concatenate(rows))  # row 7 holds 300 nonzeros
    for A in (light, heavy):
        j, jp = rand_pairs(rng, A.n, 400)
        want_net, want_dia = ref.netcount(A, j, jp), ref.dianetcount(A, j, jp)
        mtd = cp.LazyBisectCostBottleneckSplitter(AFF, 0.01)
        want_spl = ref.partition_stripe(A, 8, mtd).spl
        for force_sort, windowed in ((False, False), (True, False), (True, True)):
            if force_sort:
                monkeypatch.setenv("CPB_NO_ROW_SEGMENTS", "1")
            else:
                monkeypatch.delenv("CPB_NO_ROW_SEGMENTS", raising=False)
            # the sort form scatters the links either directly or (large inputs) after grouping them by destination window
            monkeypatch.setenv("CPB_WINDOWED_SCATTER_MIN", "1" if windowed else "0")
            assert np.array_equal(cp.netcount(A).query(j, jp), want_net)
            assert np.array_equal(cp.dianetcount(A).query(j, jp), want_dia)
            assert np.array_equal(cp.partition_stripe(A, 8, mtd).spl, want_spl)
    monkeypatch.delenv("CPB_NO_ROW_SEGMENTS", raising=False)
    monkeypatch.delenv("CPB_WINDOWED_SCATTER_MIN", raising=False)


MODELS = [
    cp.AffineWorkModel(0, 10, 1),
    cp.AffineConnectivityModel(0, 10, 1, 100),
    cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0),
    cp.AffineEnvelopeModel(1, 2, 3, 4),
]
SQUARE = [
    cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 90),
    cp.AffineMonotonizedSymmetricConnectivityModel(10, 10, 10, 100, 2),
    cp.AffineSymmetricConnectivityModel(1, 2, 3, 4, 5),
    cp.AffineHyperedgeCutModel(0, 1, 2, 3, 4),
    cp.AffineSymmetricEdgeCutModel(10, 10, 10, 100),
    cp.AffineSymmetricEdgeCutModel(0.5, 1.0, 1.0, 2.5),
]


def test_oracle_queries(ref, fixtures):
    rng = np.random.default_rng(102)
    for A in small_matrices(fixtures) + [synth.laplacian5(48)]:
        j, jp = rand_pairs(rng, A.n, 400)
        for mdl in MODELS + (SQUARE if A.m == A.n else [cp.AffineHyperedgeCutModel(0, 1, 2, 3, 4)]):
            if mdl.kind == cp.MODEL_ENVELOPE:
                keep = j < jp
                jj, jjp = j[keep], jp[keep]
            else:
                jj, jjp = j, jp
            if len(jj) == 0:
                continue
            ocl = cp.oracle_stripe(mdl, A)
            got = ocl.query(jj, jjp)
            ocl.close()
            exp = ref.oracle_query(mdl, A, jj, jjp)
            assert np.array_equal(got, exp), (mdl, A)


def test_column_block_oracle(ref, fixtures):
    rng = np.random.default_rng(103)
    mdl = cp.ColumnBlockComponentCostModel(int, 3, lambda w: 1 + w)
    for A in [fixtures["Pajek/GD99_c"], fixtures["LPnetlib/lp_blend"]]:
        j = rng.integers(1, A.n + 1, 300)
        jp = np.minimum(j + rng.integers(0, 9, 300), A.n + 1)
        ocl = cp.oracle_stripe(mdl, A, w_tab=8)
        got = ocl.query(j, jp)
        ocl.close()
        assert np.array_equal(got, ref.oracle_query(mdl, A, j, jp))


def test_column_block_oracle_wider_than_table(ref, fixtures):
    """ADVICE r1: a ConstrainedCost shrinks the tabulated widths to w_tab < n; queries wider than the table must not read
    past it -- they are infeasible under the constraint and come back as +Inf, the others equal the CPU oracle."""
    rng = np.random.default_rng(1031)
    A = fixtures["LPnetlib/lp_blend"]
    mdl = cp.ColumnBlockComponentCostModel(int, 3, lambda w: 1 + w)
    con = cp.ConstrainedCost(mdl, cp.VertexCount(), 5)
    j = rng.integers(1, A.n + 1, 2000)
    jp = np.minimum(j + rng.integers(0, A.n, 2000), A.n + 1)  # most of them far wider than the 5-column window
    ocl = cp.oracle_stripe(con, A)
    got = ocl.query(j, jp)
    ocl.close()
    wide = (jp - j) > 5
    assert np.all(np.isinf(got[wide])) and wide.sum() > 1000
    assert np.array_equal(got[~wide], ref.oracle_query(mdl, A, j[~wide], jp[~wide]))
    raw = cp.oracle_stripe(mdl, A, w_tab=4)  # an explicit short table, no constraint: still no out-of-bounds read
    got = raw.query(j, jp)
    raw.close()
    assert np.all(np.isinf(got[(jp - j) > 4]))


def test_envelope_bound_is_the_oracle_form(ref, fixtures):
    """ADVICE r1: partition_stripe(Bisect*) reaches bound_stripe(A, K, ocl) (EnvelopeCosts.jl:30-42): c_hi = ocl(1, n + 1) summed
    left to right, c_lo = alpha + fld(c_hi - alpha, K) -- for Float64 models with alpha != 0 that differs from the model form
    by roundings, and an empty pattern has a bound (no `extrema of an empty collection`)."""
    f = cp.AffineEnvelopeModel(0.1, 0.7, 0.3, 1.9)
    for A in [fixtures["LPnetlib/lp_blend"], fixtures["Pajek/GD99_c"], cp.SparseMatrixCSC(5, 4, [1, 1, 1, 1, 1], np.zeros(0, dtype=np.int64))]:
        for K in (1, 3, 7):
            assert cp.bound_stripe(A, K, f) == ref.bound_stripe(A, K, f, via_oracle=True), (A.n, K)
        if A.nnz:
            for mtd in (cp.BisectCostBottleneckSplitter(f, 0.01), cp.LazyBisectCostBottleneckSplitter(f, 0.01)):
                assert np.array_equal(cp.partition_stripe(A, 5, mtd).spl, ref.partition_stripe(A, 5, mtd).spl)


def test_prewalk_never_skips_the_last_feasible_probe(ref):
    """Fuzzer find (seed 41): bound_stripe's lower bound alpha + fld(c_hi - alpha, K) is not a bound for the envelope model (it
    can exceed the optimum), so the bisection can end on its INITIAL c_lo after feasible probes only -- the probe that ends
    the loop is then the last feasible one and must run for real even when the planner's bound already says "feasible"."""
    import json
    import os

    d = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "envelope_prewalk_case.json")))
    A = cp.SparseMatrixCSC(d["m"], d["n"], d["colptr"], np.array(d["rowval"], dtype=np.int64))
    f = cp.AffineEnvelopeModel(1.5, 1.0, 1.5, 3.0)
    for eps in (0.3, 0.1, 0.01, 0.001):
        for K in (2, 5, 9):
            for mk in (cp.BisectCostBottleneckSplitter, cp.LazyBisectCostBottleneckSplitter):
                g, r = cp.partition_stripe(A, K, mk(f, eps)), ref.partition_stripe(A, K, mk(f, eps))
                assert np.array_equal(g.spl, r.spl), (eps, K, mk.__name__, g.spl, r.spl)


def test_refusals_named_by_the_round1_review(fixtures):
    """ADVICE r1: (1) a work model with a negative beta shrinks as the part grows -- the reference's windowed search is path
    dependent there, the device refuses instead of answering differently; (2) the device-array query entry point has no part
    index and must not answer for part 1 on the row-partition-aware models."""
    import torch

    A = fixtures["LPnetlib/lp_blend"]
    for mtd in (cp.BisectCostBottleneckSplitter(cp.AffineWorkModel(100, -1, 0), 0.01), cp.LazyBisectCostBottleneckSplitter(cp.AffineWorkModel(100, 0, -1), 0.01),
                cp.BisectIndexBottleneckSplitter(cp.AffineWorkModel(100, -1, 0))):
        with pytest.raises(cp.CpbError) as e:
            cp.partition_stripe(A, 4, mtd)
        assert e.value.code == -2
    B = fixtures["Pajek/GD99_c"]
    m = B.m
    Pi = cp.SplitPartition(3, np.array([1, 1 + m // 3, 1 + 2 * m // 3, m + 1], dtype=np.int64))  # a row partition
    ocl = cp.oracle_stripe(cp.AffinePrimaryConnectivityModel(0, 1, 1, 1, 3), B, Pi)
    d = torch.ones(4, dtype=torch.int64, device="cuda")
    out = torch.zeros(4, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    with pytest.raises(cp.CpbError) as e:
        ocl.query_device(d.data_ptr(), d.data_ptr(), out.data_ptr(), 4)
    assert e.value.code == -2
    ocl.close()


def test_bound_and_objective(ref, fixtures):
    rng = np.random.default_rng(104)
    for A in small_matrices(fixtures):
        for K in [1, 2, 3, 8]:
            spl = np.concatenate(([1], np.sort(rng.integers(1, A.n + 2, K - 1)), [A.n + 1]))
            Phi = cp.SplitPartition(K, spl)
            for mdl in [cp.AffineWorkModel(0, 10, 1), AFF, cp.AffineConnectivityModel(0.0, 1.0, 1.0, 1.0)] + (
                [cp.AffineMonotonizedSymmetricConnectivityModel(10, 10, 10, 100, 8)] if A.m == A.n else []):
                assert cp.bound_stripe(A, K, mdl) == ref.bound_stripe(A, K, mdl)
                assert cp.bottleneck_value(A, Phi, mdl) == ref.bottleneck_value(A, Phi, mdl)
                assert cp.total_value(A, Phi, mdl) == ref.total_value(A, Phi, mdl)


def split_methods(f):
    return [cp.DynamicBottleneckSplitter(f), cp.BisectCostBottleneckSplitter(f, 0.1), cp.BisectCostBottleneckSplitter(f, 0.01),
            cp.LazyBisectCostBottleneckSplitter(f, 0.1), cp.LazyBisectCostBottleneckSplitter(f, 0.01)]


def test_partition_stripe_small(ref, fixtures):
    """The reference's own regime (test_Partitioners.jl:77-113): fixtures + tiny random matrices, K in {1,2,3,4,8}."""
    for A in small_matrices(fixtures):
        models = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), AFF, cp.AffineConnectivityModel(0.0, 3.0, 1.0, 3.5)]
        if A.m == A.n:
            models += [cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5), cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 90)]
        for f in models:
            for K in [1, 2, 3, 4, 8]:
                for mtd in split_methods(f):
                    g = cp.partition_stripe(A, K, mtd)
                    r = ref.partition_stripe(A, K, mtd)
                    assert np.array_equal(g.spl, r.spl), (A, f, K, type(mtd).__name__, g.spl, r.spl)


def test_dynamic_total_splitter(ref, fixtures):
    for A in [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], fixtures["LPnetlib/lp_blend"]]:
        for f in [cp.AffineConnectivityModel(0, 3, 1, 3), AFF, cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0)]:
            for K in [1, 2, 3, 8]:
                mtd = cp.DynamicTotalSplitter(f)
                assert np.array_equal(cp.partition_stripe(A, K, mtd).spl, ref.partition_stripe(A, K, mtd).spl)


def test_config1_downscaled(ref):
    """C1 at 64x64 (n = 4096): DynamicBottleneckSplitter, K = 8, net_model."""
    A = synth.laplacian5(64)
    mtd = cp.DynamicBottleneckSplitter(AFF)
    assert np.array_equal(cp.partition_stripe(A, 8, mtd).spl, ref.partition_stripe(A, 8, mtd).spl)


def test_config2_downscaled(ref):
    """C2 at n = 50,000: BisectCost, K = 64, eps = 0.01."""
    A = synth.erdos_renyi(50000, 10)
    for mtd in [cp.BisectCostBottleneckSplitter(AFF, 0.01), cp.LazyBisectCostBottleneckSplitter(AFF, 0.01)]:
        assert np.array_equal(cp.partition_stripe(A, 64, mtd).spl, ref.partition_stripe(A, 64, mtd).spl)


def test_config3_downscaled(ref):
    """C3 at scale 14: R-MAT, LazyBisect, K = 128, eps = 0.01 (skewed degrees, empty columns)."""
    A = synth.rmat(14, 16 << 14)
    mtd = cp.LazyBisectCostBottleneckSplitter(AFF, 0.01)
    assert np.array_equal(cp.partition_stripe(A, 128, mtd).spl, ref.partition_stripe(A, 128, mtd).spl)


def test_config5_downscaled(ref):
    """C5 at n = 20,000: symmetric plaid partitioning with the monotonized symmetric model."""
    A = synth.random_geometric(20000)
    for dp in (90, 4):
        s = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, dp)
        mtd = cp.LazyBisectCostBottleneckSplitter(s, 0.1)
        Pg, Fg = cp.partition_plaid(A, 32, cp.AlternatingPartitioner(mtd, mtd))
        Pr, Fr = ref.partition_plaid(A, 32, cp.AlternatingPartitioner(mtd, mtd))
        assert np.array_equal(Pg.spl, Pr.spl) and np.array_equal(Fg.spl, Fr.spl)


def test_speculation_depth_does_not_change_result(ref, monkeypatch):
    A = synth.erdos_renyi(20000, 10)
    mtd = cp.BisectCostBottleneckSplitter(AFF, 0.001)
    exp = ref.partition_stripe(A, 16, mtd).spl
    for depth in ("1", "2", "3", "4"):
        monkeypatch.setenv("CPB_BISECT_DEPTH", depth)
        assert np.array_equal(cp.partition_stripe(A, 16, mtd).spl, exp), depth


def test_streaming_probe_tiles(ref):
    """The streaming-probe kernel (k_probe_stream: register tiles, st.async exchanges between the cluster's CTAs) against the
    CPU oracle on inputs whose parts span several super-steps, super-steps that hold many parts, long runs of empty columns
    (more than 4096 boundary candidates per CTA and super-step), the diagonal-augmented stream and Float64 costs."""
    rng = np.random.default_rng(77)
    n_sparse = 300_000
    cols = np.sort(rng.choice(n_sparse, 4000, replace=False))
    deg = np.zeros(n_sparse, dtype=np.int64)
    deg[cols] = rng.integers(1, 12, len(cols))
    colptr = np.concatenate(([1], 1 + np.cumsum(deg)))
    rowval = np.concatenate([np.sort(rng.choice(5000, d, replace=False)) + 1 for d in deg[cols]])
    sparse_cols = cp.SparseMatrixCSC(5000, n_sparse, colptr, rowval)
    sym = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 4)
    cases = [(synth.erdos_renyi(50000, 10), AFF, [7, 64], 0.01), (synth.erdos_renyi(50000, 10), cp.AffineConnectivityModel(0.5, 10.0, 1.0, 100.0), [64], 0.01),
             (synth.rmat(15, 16 << 15), AFF, [128, 1000], 0.01), (sparse_cols, AFF, [3, 16, 200], 0.05),
             (sparse_cols, cp.AffineConnectivityModel(0, 1, 0, 0), [16], 0.01), (synth.random_geometric(30000), sym, [32], 0.1),
             (synth.banded(40000, 40), AFF, [50], 0.01), (synth.laplacian5(150), cp.AffineConnectivityModel(3, 0, 0, 1), [5, 31], 0.001)]
    for A, f, Ks, eps in cases:
        dA = cp.device_matrix(A)
        for K in Ks:
            for mtd in (cp.LazyBisectCostBottleneckSplitter(f, eps), cp.BisectCostBottleneckSplitter(f, eps)):
                exp = ref.partition_stripe(A, K, mtd).spl
                got = cp.partition_stripe(dA, K, mtd).spl
                assert np.array_equal(got, exp), (A.n, K, type(mtd).__name__)
        dA.close()


def test_device_resident_matrix_and_errors():
    A = synth.laplacian5(16)
    dA = cp.device_matrix(A)
    B = dA.to_host()
    assert np.array_equal(B.colptr, A.colptr) and np.array_equal(B.rowval, A.rowval)
    s1 = cp.partition_stripe(dA, 4, cp.DynamicBottleneckSplitter(AFF)).spl
    s2 = cp.partition_stripe(A, 4, cp.DynamicBottleneckSplitter(AFF)).spl
    assert np.array_equal(s1, s2)
    dA.close()
    bad = cp.SparseMatrixCSC(2, 2, [1, 2, 3], [1, 2])
    bad.rowval[1] = 7  # out of range row
    with pytest.raises(cp.CpbError):
        cp.device_matrix(bad)
    with pytest.raises(cp.CpbError):  # no bound_stripe method for this model in the reference
        cp.partition_stripe(A, 4, cp.BisectCostBottleneckSplitter(cp.AffineHyperedgeCutModel(0, 1, 1, 1, 1), 0.1))


def test_full_size_properties_config2():
    """BASELINE config 2 at full size (n = 10^6): size-independent properties of the result."""
    A = synth.erdos_renyi(1_000_000, 10)
    K, eps = 64, 0.01
    dA = cp.device_matrix(A)
    Phi = cp.partition_stripe(dA, K, cp.BisectCostBottleneckSplitter(AFF, eps))
    spl = Phi.spl
    assert spl[0] == 1 and spl[-1] == A.n + 1 and np.all(np.diff(spl) >= 0)
    lo, hi = cp.bound_stripe(dA, K, AFF)
    v = cp.bottleneck_value(dA, Phi, AFF)
    assert lo <= v <= hi
    # greedy maximality (App. B row 4): extending any part but the last by one column must exceed the
    # last feasible threshold, which is at most v * (1 + eps) ... so the extended cost is > v
    ocl = cp.oracle_stripe(AFF, dA)
    ext = ocl.query(spl[:-2], np.minimum(spl[1:-1] + 1, A.n + 1))
    assert np.all(ext[spl[1:-1] <= A.n] > v)
    # Lazy and random-access bisection agree split for split (SURVEY E3)
    Phi2 = cp.partition_stripe(dA, K, cp.LazyBisectCostBottleneckSplitter(AFF, eps))
    assert np.array_equal(Phi2.spl, spl)
    # oracle consistency: nets are sub-additive and monotone under refinement
    j, jp = rand_pairs(np.random.default_rng(5), A.n, 10000)
    mid = (j + jp) // 2
    net = cp.netcount(dA)
    whole, left, right = net.query(j, jp), net.query(j, mid), net.query(mid, jp)
    assert np.all(whole <= left + right) and np.all(whole >= np.maximum(left, right))
    ocl.close()
    dA.close()


def test_large_inputs_independent_engines_agree(monkeypatch):
    """Sizes the CPU oracle does not finish in seconds: the streaming probes (link array, k_probe_stream), the
    dominance-index probes (k_bisect_round) and the exact splitter (k_bisect_index) are three separate device
    implementations -- the first two must return the same split vector, and the eps-bisection's bottleneck must lie
    within (1 + eps) of the exact optimum.  R-MAT takes the radix-sort link construction (heavy rows), the others the
    row-segment form."""
    from chainb200 import synth_torch

    sym = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 4)
    cases = [(synth_torch.rmat(20, 16 << 20), AFF, 256, 0.01), (synth_torch.erdos_renyi(1_000_000, 10), AFF, 64, 0.01),
             (synth_torch.random_geometric(1 << 20), sym, 128, 0.01), (synth.laplacian5(512), AFF, 100, 0.001)]
    for A, f, K, eps in cases:
        dA = cp.device_matrix(A)
        mtd = cp.LazyBisectCostBottleneckSplitter(f, eps)
        monkeypatch.delenv("CPB_PROBE_STREAM", raising=False)
        a = cp.partition_stripe(dA, K, mtd)
        st = cp.bisect_stats()
        monkeypatch.setenv("CPB_PROBE_STREAM", "0")
        b = cp.partition_stripe(dA, K, mtd)
        monkeypatch.delenv("CPB_PROBE_STREAM", raising=False)
        assert np.array_equal(a.spl, b.spl), (A.n, K)
        monkeypatch.setenv("CPB_BISECT_PLAN", "0")  # the complete speculation tree instead of the planned one
        c = cp.partition_stripe(dA, K, mtd)
        monkeypatch.delenv("CPB_BISECT_PLAN", raising=False)
        assert np.array_equal(a.spl, c.spl), (A.n, K)
        exact = cp.partition_stripe(dA, K, cp.BisectIndexBottleneckSplitter(f))
        v, v0 = cp.bottleneck_value(dA, a, f), cp.bottleneck_value(dA, exact, f)
        assert v0 <= v <= v0 * (1 + eps), (A.n, K, v0, v)
        assert st["c_lo_final"] < v0 <= st["c_hi_final"] or v0 <= st["c_lo"]  # the final bracket holds the optimum
        dA.close()


# ------------------------------------------------------------------------------------------ pack_stripe
def chunk_matrices(fixtures):
    rng = np.random.default_rng(200)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], fixtures["LPnetlib/lp_blend"], fixtures["HB/west0132"]]
    mats += [sprand(rng, m, n, p) for (m, n, p) in [(1, 1, 1.0), (3, 1, 0.5), (4, 2, 0.5), (8, 9, 0.4), (30, 41, 0.2), (64, 1500, 0.05), (500, 3000, 0.01)]]
    mats.append(synth.banded(5000, 8))
    return mats


BLOCK_MODELS = [
    cp.BlockComponentCostModel(int, 1, 3, (1, cp.identity), (1, cp.identity)),  # runbenchmarks.jl:22
    cp.BlockComponentCostModel(int, 0, 0, (10, cp.identity), (2, lambda x: 2 * x)),  # test_Partitioners.jl:227
    cp.BlockComponentCostModel(int, cp.identity, lambda x: 3 * x, (10, cp.identity), (2, lambda x: 2 * x)),
]


def test_pack_stripe_dynamic_total_chunker(ref, fixtures):
    """DynamicTotalChunker(ConstrainedCost(f, VertexCount(), w_max)): split vectors identical (leftmost ties)."""
    for A in chunk_matrices(fixtures):
        Pi = ref.pack_stripe(ref.adjointpattern(A), cp.EquiChunker(2))
        models = [cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0, 0, 0, 1), AFF, cp.AffineWorkModel(1, 2, 3),
                  cp.ColumnBlockComponentCostModel(int, 3, lambda w: 1 + w), cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0)] + BLOCK_MODELS
        for f in models:
            for w_max in [1, 2, 4, 8, 13]:
                mtd = cp.DynamicTotalChunker(cp.ConstrainedCost(f, cp.VertexCount(), w_max))
                args = (Pi,) if f.kind == cp.MODEL_BLOCK else ()
                g = cp.pack_stripe(A, mtd, *args)
                r = ref.pack_stripe(A, mtd, *args)
                assert g.K == r.K and np.array_equal(g.spl, r.spl), (A, f, w_max, g.spl[:10], r.spl[:10])


def test_pack_stripe_work_weight(ref, fixtures):
    """ConstrainedCost with an AffineWorkModel weight (test_Partitioners.jl:176-178)."""
    A = fixtures["LPnetlib/lp_blend"]
    for w_max in [2, 4, 8]:
        mtd = cp.DynamicTotalChunker(cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineWorkModel(0, 1, 0), w_max))
        assert np.array_equal(cp.pack_stripe(A, mtd).spl, ref.pack_stripe(A, mtd).spl)
    mtd = cp.DynamicTotalChunker(cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineWorkModel(0, 2, 1), 40))
    assert np.array_equal(cp.pack_stripe(A, mtd).spl, ref.pack_stripe(A, mtd).spl)


def test_pack_stripe_convex(ref, fixtures):
    """ConvexTotalChunker(ConstrainedCost(connectivity, VertexCount(), w_max)) (bin/test_table_constrained_chunks.jl:32-41)."""
    for A in chunk_matrices(fixtures):
        for f in [cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(-0.5, 0.0, 0.0, 1.0)]:
            for w_max in [1, 2, 3, 4, 8]:
                mtd = cp.ConvexTotalChunker(cp.ConstrainedCost(f, cp.VertexCount(), w_max))
                g = cp.pack_stripe(A, mtd)
                r = ref.pack_stripe(A, mtd)
                assert np.array_equal(g.spl, r.spl), (A, f, w_max)


def test_pack_stripe_overlap_strict_equi(ref, fixtures):
    for A in chunk_matrices(fixtures):
        for w_max in [1, 2, 4, 8]:
            for rho in [0.9, 0.8, 0.7, 0.3]:
                bg, br = [None], [None]
                g = cp.pack_stripe(A, cp.OverlapChunker(rho, w_max), n_nets=bg)
                r = ref.pack_stripe(A, cp.OverlapChunker(rho, w_max), n_nets=br)
                assert np.array_equal(g.spl, r.spl), (A, rho, w_max)
                assert np.array_equal(bg[0], br[0])
            assert np.array_equal(cp.pack_stripe(A, cp.StrictChunker(w_max)).spl, ref.pack_stripe(A, cp.StrictChunker(w_max)).spl)
            assert np.array_equal(cp.pack_stripe(A, cp.EquiChunker(w_max)).spl, ref.pack_stripe(A, cp.EquiChunker(w_max)).spl)


def test_strict_chunker_with_repeated_columns(ref):
    rng = np.random.default_rng(201)
    base = sprand(rng, 12, 40, 0.3).to_scipy().tocsc()
    import scipy.sparse as sp

    cols = np.repeat(np.arange(40), rng.integers(1, 6, 40))
    A = cp.SparseMatrixCSC.from_scipy(sp.csc_matrix(base[:, cols]))
    for w_max in [1, 2, 3, 8]:
        assert np.array_equal(cp.pack_stripe(A, cp.StrictChunker(w_max)).spl, ref.pack_stripe(A, cp.StrictChunker(w_max)).spl)


def test_pack_infeasible_and_unsupported():
    A = synth.banded(200, 4)
    with pytest.raises(cp.CpbError) as e:
        cp.pack_stripe(A, cp.DynamicTotalChunker(cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineWorkModel(5, 1, 0), 3)))
    assert e.value.code == -4
    with pytest.raises(cp.CpbError):  # ConcaveTotalChunker.jl:9 has no ConstrainedCost method
        cp.pack_stripe(A, cp.ConcaveTotalChunker(cp.ConstrainedCost(cp.AffineWorkModel(1, 1, 1), cp.VertexCount(), 3)))


def test_config4_downscaled(ref):
    """C4 at n = 2^15: banded, X = adjointpattern(A), Pi = pack_stripe(A, EquiChunker(4)),
    DynamicTotalChunker(block_model, 8) and ConvexTotalChunker(connectivity, 8)."""
    A = synth.banded(1 << 15, 64)
    X = cp.adjointpattern(A)
    Pi = cp.pack_stripe(A, cp.EquiChunker(4))
    g = cp.BlockComponentCostModel(int, 1, 3, (1, cp.identity), (1, cp.identity))
    m1 = cp.DynamicTotalChunker(g, 8)
    assert np.array_equal(cp.pack_stripe(X, m1, Pi).spl, ref.pack_stripe(X, m1, Pi).spl)
    m2 = cp.ConvexTotalChunker(cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.VertexCount(), 8))
    assert np.array_equal(cp.pack_stripe(X, m2).spl, ref.pack_stripe(X, m2).spl)
    Pg, Fg = cp.pack_plaid(A, cp.AlternatingPacker(cp.OverlapChunker(0.9, 8), m1))
    Pr, Fr = ref.pack_plaid(A, cp.AlternatingPacker(cp.OverlapChunker(0.9, 8), m1))
    assert np.array_equal(Pg.spl, Pr.spl) and np.array_equal(Fg.spl, Fr.spl)


def test_chunk_dp_many_blocks(ref):
    """n = 2^19 columns: several staged chunks in the blocked (min,+) combine and in the chain unravel (the kernels
    stage 40 DP blocks / 640 chain blocks at a time in shared memory)."""
    A = synth.banded(1 << 19, 6)
    for mtd in [cp.DynamicTotalChunker(cp.AffineConnectivityModel(0, 3, 1, 3), 8),
                cp.ConvexTotalChunker(cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.VertexCount(), 5)),
                cp.StrictChunker(4)]:
        g, r = cp.pack_stripe(A, mtd), ref.pack_stripe(A, mtd)
        assert g.K == r.K and np.array_equal(g.spl, r.spl), type(mtd).__name__


def test_torch_generators_match_numpy():
    from chainb200 import synth_torch

    for a, b in [(synth.erdos_renyi(3000, 10), synth_torch.erdos_renyi(3000, 10)), (synth.rmat(10, 16 << 10), synth_torch.rmat(10, 16 << 10)),
                 (synth.banded(2000, 16), synth_torch.banded(2000, 16)), (synth.random_geometric(3000), synth_torch.random_geometric(3000))]:
        assert (a.m, a.n) == (b.m, b.n) and np.array_equal(a.colptr, b.colptr) and np.array_equal(a.rowval, b.rowval)


def test_dynamic_total_splitter_divide_and_conquer(ref):
    """DynamicTotalSplitter at sizes where the device uses the monotone divide & conquer layer."""
    for A, Ks in [(synth.laplacian5(40), [2, 3, 5]), (synth.erdos_renyi(1500, 6), [2, 4]), (synth.banded(1000, 5), [3]), (synth.rmat(10, 16 << 10), [4])]:
        models = [cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineWorkModel(2, 3, 1)]
        if A.m == A.n:
            models.append(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 2))
        for f in models:
            for K in Ks:
                mtd = cp.DynamicTotalSplitter(f)
                g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                assert np.array_equal(g.spl, r.spl), (A, f, K, g.spl, r.spl)


def test_constrained_dynamic_splitters(ref, fixtures):
    """AbstractDynamicSplitter{<:ConstrainedCost} (DynamicSplitter.jl:206-247), incl. the degenerate
    partition [1, 1, ..., n+1] returned for infeasible width constraints (:217-222)."""
    rng = np.random.default_rng(300)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 1, 0.5), sprand(rng, 6, 10, 0.3), sprand(rng, 40, 200, 0.1)]
    for A in mats:
        for f in [cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0)]:
            for w, w_max in [(cp.AffineWorkModel(0, 1, 0), 2), (cp.AffineWorkModel(0, 1, 0), 4), (cp.VertexCount(), 8), (cp.AffineWorkModel(1, 2, 0), 9),
                             (cp.AffineWorkModel(5, 1, 0), 3),
                             # weights with a pin term: windows follow the column lengths (binary searches on pos)
                             (cp.AffineWorkModel(0, 1, 1), 12), (cp.AffineWorkModel(0, 0, 1), 9), (cp.AffineWorkModel(2, 1, 2), 40),
                             (cp.AffineWorkModel(0, 0, 1), 2)]:
                for K in [1, 2, 3, 4, 8, 60]:
                    for mk in (cp.DynamicTotalSplitter, cp.DynamicBottleneckSplitter):
                        mtd = mk(cp.ConstrainedCost(f, w, w_max))
                        g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                        assert np.array_equal(g.spl, r.spl), (A, f, w_max, K, mk.__name__, g.spl, r.spl)


def test_constrained_convex_total_splitter(ref, fixtures):
    """partition_stripe(A, K, ConvexTotalSplitter(ConstrainedCost(f, w, w_max))) (ConvexTotalChunker.jl:167-265; the
    reference's own cases test_Partitioners.jl:176-196 and bin/test_table_constrained_splits.jl:26-40): identical split
    vectors for vertex- and pin-weighted windows, incl. the degenerate result for infeasible constraints and wide windows."""
    rng = np.random.default_rng(311)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 1, 0.5), sprand(rng, 6, 10, 0.3), sprand(rng, 40, 200, 0.1),
            synth.laplacian5(20)]
    for A in mats:
        fs = [cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0), cp.AffineWorkModel(0, 0, 0)]
        if A.m == A.n:
            fs.append(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5))
        for f in fs:
            for w, w_max in [(cp.AffineWorkModel(0, 1, 0), 2), (cp.AffineWorkModel(0, 1, 0), 4), (cp.AffineWorkModel(0, 1, 0), 8), (cp.VertexCount(), 8),
                             (cp.AffineWorkModel(1, 2, 0), 9), (cp.AffineWorkModel(5, 1, 0), 3), (cp.AffineWorkModel(0, 1, 1), 12), (cp.AffineWorkModel(0, 0, 1), 9),
                             (cp.AffineWorkModel(2, 1, 2), 40), (cp.VertexCount(), int(np.ceil(A.n / 4 * 1.5)))]:
                for K in [1, 2, 3, 4, 8, 16, 60]:
                    mtd = cp.ConvexTotalSplitter(cp.ConstrainedCost(f, w, w_max))
                    g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                    assert np.array_equal(g.spl, r.spl), (A, f, w_max, K, g.spl, r.spl)
    B = synth.banded(3000, 6, 3)  # wide windows (bin/test_table_constrained_splits.jl: w_max = 1.5 n / K): warp-per-column layers
    for K in (3, 8):
        spec = cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.VertexCount(), int(np.ceil(B.n / K * 1.5)))
        for mk in (cp.ConvexTotalSplitter, cp.DynamicTotalSplitter, cp.DynamicBottleneckSplitter):
            assert np.array_equal(cp.partition_stripe(B, K, mk(spec)).spl, ref.partition_stripe(B, K, mk(spec)).spl), (K, mk.__name__)
        spec = cp.ConstrainedCost(cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineWorkModel(0, 1, 1), int(np.ceil((B.n + B.nnz) / K * 1.5)))
        for mk in (cp.ConvexTotalSplitter, cp.DynamicTotalSplitter):
            assert np.array_equal(cp.partition_stripe(B, K, mk(spec)).spl, ref.partition_stripe(B, K, mk(spec)).spl), (K, mk.__name__, "pin-weighted")


def test_concave_total_chunker_and_splitter(ref, fixtures):
    """a23: pack_stripe(A, ConcaveTotalChunker(f)) (ConcaveTotalChunker.jl:9-24), partition_stripe(A, K, ConcaveTotalSplitter(f))
    (:26-55) and its ConstrainedCost form (:143-181).  The device runs the reference's queue routine (:57-114) step by step, so
    the split vectors equal the restated algorithm's for ANY model -- concave (work model: modular; tabulated column-block
    model with a concave beta(w)), or not (connectivity: the result is then whatever the queue leaves, and still identical)."""
    rng = np.random.default_rng(2300)
    mats = [sprand(rng, 6, 1, 0.5), sprand(rng, 6, 2, 0.5), sprand(rng, 6, 11, 0.3), sprand(rng, 30, 120, 0.1), fixtures["Pajek/GD99_c"], synth.laplacian5(12),
            cp.SparseMatrixCSC(5, 4, [1, 1, 1, 1, 1], np.zeros(0, dtype=np.int64))]
    concave_tab = cp.ColumnBlockComponentCostModel(int, 7, lambda w: int(20 * np.sqrt(w)))  # concave beta_col(w)
    models = [cp.AffineWorkModel(3, 1, 2), cp.AffineWorkModel(0, 0, 0), cp.AffineWorkModel(0.5, 0.25, 1.5), cp.AffineConnectivityModel(0, 10, 1, 100),
              cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0), concave_tab]
    for A in mats:
        for f in models:
            g, r = cp.pack_stripe(A, cp.ConcaveTotalChunker(f)), ref.pack_stripe(A, cp.ConcaveTotalChunker(f))
            assert g.K == r.K and np.array_equal(g.spl, r.spl), (A.n, f, g.spl, r.spl)
            for K in (1, 2, 3, 5, 16):
                mtd = cp.ConcaveTotalSplitter(f)
                g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                assert np.array_equal(g.spl, r.spl), (A.n, f, K, g.spl, r.spl)
        for f in models[:5]:
            for w, w_max in [(cp.VertexCount(), 3), (cp.AffineWorkModel(0, 1, 0), 8), (cp.AffineWorkModel(1, 2, 0), 9), (cp.AffineWorkModel(0, 1, 1), 12),
                             (cp.AffineWorkModel(5, 1, 0), 3)]:
                for K in (1, 2, 4, 9):
                    mtd = cp.ConcaveTotalSplitter(cp.ConstrainedCost(f, w, w_max))
                    g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                    assert np.array_equal(g.spl, r.spl), (A.n, f, w_max, K, g.spl, r.spl)


def test_dynamic_chunker_kform(ref, fixtures):
    """partition_stripe(A, K, DynamicBottleneckChunker(f) / DynamicTotalChunker(f)) (DynamicSplitter.jl:52-87,249-314)."""
    rng = np.random.default_rng(301)
    for A in [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 10, 0.3), sprand(rng, 40, 120, 0.1)]:
        for f in [cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineWorkModel(0, 10, 1)]:
            for K in [1, 2, 3, 8]:
                for mk in (cp.DynamicBottleneckChunker, cp.DynamicTotalChunker):
                    for spec in (f, cp.ConstrainedCost(f, cp.VertexCount(), 8), cp.ConstrainedCost(f, cp.VertexCount(), 2)):
                        g, r = cp.partition_stripe(A, K, mk(spec)), ref.partition_stripe(A, K, mk(spec))
                        assert np.array_equal(g.spl, r.spl), (A, f, K, mk.__name__, g.spl, r.spl)


def test_convex_total_splitter(ref, fixtures):
    """partition_stripe(A, K, ConvexTotalSplitter(f)) (ConvexTotalChunker.jl:26-55): warp-scan layers (n <= 64) and
    monotone divide & conquer layers (larger n) against the reference's stack algorithm."""
    rng = np.random.default_rng(302)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], fixtures["LPnetlib/lp_blend"], sprand(rng, 6, 10, 0.3), sprand(rng, 40, 200, 0.1),
            synth.laplacian5(24), synth.erdos_renyi(1500, 6)]
    for A in mats:
        fs = [cp.AffineConnectivityModel(0, 3, 1, 3), AFF, cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0)]
        if A.m == A.n:
            fs.append(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5))
        for f in fs:
            for K in [1, 2, 3, 8]:
                mtd = cp.ConvexTotalSplitter(f)
                g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                assert np.array_equal(g.spl, r.spl), (A, f, K, g.spl, r.spl)
    with pytest.raises(cp.CpbError):  # not a quadrangle-inequality model: the reference's result is an artefact of its stack
        cp.partition_stripe(mats[0], 3, cp.ConvexTotalSplitter(cp.AffineSymmetricEdgeCutModel(1, 1, 1, 1)))


def test_unconstrained_convex_chunker(ref, fixtures):
    """pack_stripe(A, ConvexTotalChunker(f)) without a constraint (ConvexTotalChunker.jl:9-24)."""
    rng = np.random.default_rng(303)
    for A in [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 10, 0.3), sprand(rng, 5, 1, 0.5), synth.erdos_renyi(2000, 5)]:
        for f in [cp.AffineConnectivityModel(0, 3, 1, 3), AFF, cp.AffineWorkModel(2, 10, 1), cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0)]:
            for mk in (cp.ConvexTotalChunker, cp.DynamicTotalChunker):
                g, r = cp.pack_stripe(A, mk(f)), ref.pack_stripe(A, mk(f))
                assert g.K == r.K and np.array_equal(g.spl, r.spl), (A, f, mk.__name__, g.spl, r.spl)
    with pytest.raises(cp.CpbError):
        cp.pack_stripe(sprand(rng, 6, 10, 0.3), cp.ConvexTotalChunker(cp.AffineConnectivityModel(-1, 3, 1, 3)))


def test_bisect_index_splitter(ref, fixtures):
    """partition_stripe(A, K, BisectIndexBottleneckSplitter(f)) (BisectIndexBottleneckSplitter.jl:5-81): the exact
    bottleneck splitter, one cluster kernel following the reference's control flow; identical split vectors, and the
    bottleneck equals the DynamicBottleneckSplitter optimum."""
    rng = np.random.default_rng(304)
    mats = small_matrices(fixtures)[:10] + [sprand(rng, 40, 200, 0.1), synth.laplacian5(20), synth.erdos_renyi(3000, 6)]
    for A in mats:
        fs = [cp.AffineConnectivityModel(0, 3, 1, 3), AFF, cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0.0, 3.0, 1.0, 3.5)]
        if A.m == A.n:
            fs.append(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5))
        for f in fs:
            for K in [1, 2, 3, 8, 33]:
                mtd = cp.BisectIndexBottleneckSplitter(f)
                g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                assert np.array_equal(g.spl, r.spl), (A, f, K, g.spl, r.spl)
    A = synth.erdos_renyi(3000, 6)
    g = cp.partition_stripe(A, 8, cp.BisectIndexBottleneckSplitter(AFF))
    d = cp.partition_stripe(A, 8, cp.DynamicBottleneckSplitter(AFF))
    assert cp.bottleneck_value(A, g, AFF) == cp.bottleneck_value(A, d, AFF)


def prim_partitions(ref, A, K):
    """Pi = partition_stripe(A', K, EquiSplitter()) as in test_Partitioners.jl:95."""
    return ref.partition_stripe(ref.adjointpattern(A), K, cp.EquiSplitter())


def test_primary_connectivity_model(ref, fixtures):
    """AffinePrimaryConnectivityModel with a row partition (PrimaryConnectivityCosts.jl:5-86, PartwiseCounts.jl:1-101):
    oracle queries with the part index, bound_stripe, and every splitter of test_Partitioners.jl:86-113 on it."""
    rng = np.random.default_rng(305)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 10, 0.3), sprand(rng, 8, 3, 0.5), sprand(rng, 40, 120, 0.1),
            synth.erdos_renyi(2000, 5)]
    for A in mats:
        for K in [1, 2, 3, 8]:
            Pi = prim_partitions(ref, A, K)
            for f in [cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6), cp.AffinePrimaryConnectivityModel(1, 1, 1, 1, 1),
                      cp.AffinePrimaryConnectivityModel(0.0, 0.5, 1.0, 3.0, 6.5)]:
                j, jp = rand_pairs(rng, A.n, 300)
                k = rng.integers(1, K + 1, 300)
                ocl = cp.oracle_stripe(f, A, Pi)
                assert np.array_equal(ocl.query(j, jp, k), ref.oracle_query(f, A, j, jp, k, Pi=Pi))
                ocl.close()
                if A.n > 500 and K > 3:
                    continue
                for mtd in [cp.DynamicBottleneckSplitter(f), cp.DynamicTotalSplitter(f), cp.BisectIndexBottleneckSplitter(f),
                            cp.BisectCostBottleneckSplitter(f, 0.1), cp.BisectCostBottleneckSplitter(f, 0.01), cp.LazyBisectCostBottleneckSplitter(f, 0.01)]:
                    g, r = cp.partition_stripe(A, K, mtd, Pi), ref.partition_stripe(A, K, mtd, Pi)
                    assert np.array_equal(g.spl, r.spl), (A, f, K, type(mtd).__name__, g.spl, r.spl)
                    assert cp.bottleneck_value(A, g, f, Pi) == ref.bottleneck_value(A, g, f, Pi)


def test_secondary_connectivity_model_and_flip_splitters(ref, fixtures):
    """AffineSecondaryConnectivityModel with a row partition (SecondaryConnectivityCosts.jl:5-102) and the Flip family
    (BisectCost...:70-127, LazyBisect...:79-138, BisectIndex...:87-166): queries with the part index, bound_stripe, and
    identical split vectors for every splitter of test_Partitioners.jl:131-148."""
    rng = np.random.default_rng(306)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 10, 0.3), sprand(rng, 8, 3, 0.5), sprand(rng, 40, 120, 0.1),
            synth.erdos_renyi(2000, 5)]
    for A in mats:
        for K in [1, 2, 3, 8]:
            Pi = prim_partitions(ref, A, K)
            for f in [cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6), cp.AffineSecondaryConnectivityModel(1, 1, 1, 1, 1),
                      cp.AffineSecondaryConnectivityModel(0.0, 0.5, 1.0, 3.0, 6.5)]:
                j, jp = rand_pairs(rng, A.n, 300)
                k = rng.integers(1, K + 1, 300)
                ocl = cp.oracle_stripe(f, A, Pi)
                assert np.array_equal(ocl.query(j, jp, k), ref.oracle_query(f, A, j, jp, k, Pi=Pi))
                ocl.close()
                mtds = [cp.FlipBisectIndexBottleneckSplitter(f), cp.FlipBisectCostBottleneckSplitter(f, 0.1), cp.FlipBisectCostBottleneckSplitter(f, 0.001),
                        cp.LazyFlipBisectCostBottleneckSplitter(f, 0.1), cp.LazyFlipBisectCostBottleneckSplitter(f, 0.001)]
                if A.n <= 500:
                    mtds.append(cp.DynamicBottleneckSplitter(f))
                for mtd in mtds:
                    g, r = cp.partition_stripe(A, K, mtd, Pi), ref.partition_stripe(A, K, mtd, Pi)
                    assert np.array_equal(g.spl, r.spl), (A, f, K, type(mtd).__name__, g.spl, r.spl)


def test_edgecut_part_models(ref, fixtures):
    """AffinePrimaryEdgeCutModel / AffineSecondaryEdgeCutModel with a row partition (PrimaryEdgeCutCosts.jl:5-66,
    SecondaryEdgeCutCosts.jl:5-97): queries with the part index, and identical split vectors for the increasing-cost
    splitters (primary) and the Flip family (secondary)."""
    rng = np.random.default_rng(307)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 10, 0.3), sprand(rng, 8, 3, 0.5), sprand(rng, 40, 120, 0.1),
            synth.erdos_renyi(2000, 5)]
    for A in mats:
        for K in [1, 2, 3, 8]:
            Pi = prim_partitions(ref, A, K)
            for co in [(0, 2, 1, 5), (1, 1, 1, 1), (0.0, 0.5, 1.0, 3.5)]:
                for f in (cp.AffinePrimaryEdgeCutModel(*co), cp.AffineSecondaryEdgeCutModel(*co)):
                    j, jp = rand_pairs(rng, A.n, 300)
                    k = rng.integers(1, K + 1, 300)
                    ocl = cp.oracle_stripe(f, A, Pi)
                    assert np.array_equal(ocl.query(j, jp, k), ref.oracle_query(f, A, j, jp, k, Pi=Pi))
                    ocl.close()
                    if isinstance(f, cp.AffinePrimaryEdgeCutModel):
                        mtds = [cp.BisectIndexBottleneckSplitter(f), cp.BisectCostBottleneckSplitter(f, 0.1), cp.BisectCostBottleneckSplitter(f, 0.01),
                                cp.LazyBisectCostBottleneckSplitter(f, 0.01)]
                        if A.n <= 500:
                            mtds += [cp.DynamicBottleneckSplitter(f), cp.DynamicTotalSplitter(f)]
                    else:
                        mtds = [cp.FlipBisectIndexBottleneckSplitter(f), cp.FlipBisectCostBottleneckSplitter(f, 0.1), cp.FlipBisectCostBottleneckSplitter(f, 0.001),
                                cp.LazyFlipBisectCostBottleneckSplitter(f, 0.01)]
                        if A.n <= 500:
                            mtds.append(cp.DynamicBottleneckSplitter(f))
                    for mtd in mtds:
                        g, r = cp.partition_stripe(A, K, mtd, Pi), ref.partition_stripe(A, K, mtd, Pi)
                        assert np.array_equal(g.spl, r.spl), (A, f, K, type(mtd).__name__, g.spl, r.spl)
                        assert cp.bottleneck_value(A, g, f, Pi) == ref.bottleneck_value(A, g, f, Pi)


def test_objective_of_noncontiguous_partitions(ref, fixtures):
    """bottleneck_value / total_value of Map- and DomainPartitions (Costs.jl:26-66, WorkCosts.jl:53-81,
    PrimaryConnectivityCosts.jl:88-163, EnvelopeCosts.jl:75-129): the device gathers the columns part by part
    (cpb_matrix_permute), renames the rows of a non-contiguous row partition, and evaluates contiguous parts.  Also:
    partition_stripe with a MapPartition of the rows, and a SplitPartition seen as a MapPartition has the same value."""
    rng = np.random.default_rng(309)
    models = [cp.AffineWorkModel(1, 2, 3), cp.AffineConnectivityModel(0, 10, 1, 100), cp.AffineConnectivityModel(0.5, 1.0, 0.25, 3.0),
              cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6), cp.AffinePrimaryEdgeCutModel(0, 2, 1, 5), cp.AffineEnvelopeModel(0, 1, 1, 2),
              cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6)]
    mats = [fixtures["LPnetlib/lpi_itest6"], sprand(rng, 6, 10, 0.3), sprand(rng, 8, 3, 0.5), sprand(rng, 40, 120, 0.1), sprand(rng, 5, 7, 0.0),
            synth.erdos_renyi(3000, 6)]
    for A in mats:
        for K in (1, 3, 7):
            Phi = cp.MapPartition(K, rng.integers(1, K + 1, A.n))
            Pi = cp.MapPartition(K, rng.integers(1, K + 1, A.m))
            dom = cp.convert(cp.DomainPartition, Phi)
            for mdl in models:
                pi = Pi if "Primary" in type(mdl).__name__ or "Secondary" in type(mdl).__name__ else None
                for P in (Phi, dom):
                    assert cp.bottleneck_value(A, P, mdl, pi) == ref.bottleneck_value(A, P, mdl, pi), (A, K, mdl)
                    assert cp.total_value(A, P, mdl, pi) == ref.total_value(A, P, mdl, pi), (A, K, mdl)
            f = cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6)
            for mtd in (cp.DynamicBottleneckSplitter(f), cp.BisectCostBottleneckSplitter(f, 0.01)):
                if A.n > 500 and isinstance(mtd, cp.DynamicBottleneckSplitter):
                    continue
                g = cp.partition_stripe(A, K, mtd, Pi)
                Amap, _, Pis = ref._contiguous(A, g, Pi)
                assert np.array_equal(g.spl, ref.partition_stripe(Amap, K, mtd, Pis).spl)
            S = cp.partition_stripe(A, K, cp.EquiSplitter())
            net = cp.AffineConnectivityModel(0, 10, 1, 100)
            assert cp.bottleneck_value(A, cp.convert(cp.MapPartition, S), net) == cp.bottleneck_value(A, S, net)
    B = cp.permute(mats[0], rng.permutation(mats[0].n) + 1, None).to_host()
    assert sorted(np.diff(B.colptr).tolist()) == sorted(np.diff(mats[0].colptr).tolist())
    with pytest.raises(cp.CpbError):
        cp.permute(mats[0], np.ones(mats[0].n, dtype=np.int64), None)


def test_prefix_structures(ref):
    """dominancecount / dominancesum / rookcount! / rooksum! on the device (SparsePrefixMatrices.jl:1-1273; the reference's
    test_SparsePrefixMatrices.jl:26-71 dims and value types, plus sizes that span many rank blocks and scan tiles): every
    entry equals the CPU sweep, single entries through getindex, corners included."""
    rng = np.random.default_rng(308)
    dims = [1, 2, 3, 7, 8, 9, 31, 32, 33, 63, 64, 65]
    cases = [(m, n, 0.5) for m in dims for n in (1, 3, 8, 33)] + [(300, 500, 0.02), (1000, 1000, 0.01), (5000, 40000, 0.002), (70000, 3000, 0.001), (5, 6, 0.0)]
    for m, n, p in cases:
        A = sprand(rng, m, n, p)
        Q = 400 if A.nnz > 1000 else 40
        i = np.concatenate([rng.integers(1, m + 2, Q), [1, 1, m + 1, m + 1]])
        j = np.concatenate([rng.integers(1, n + 2, Q), [1, n + 1, 1, n + 1]])
        for val in (rng.integers(0, 2**64, A.nnz, dtype=np.uint64), rng.integers(-5, 6, A.nnz)):
            C, S = cp.dominancecount(A), cp.dominancesum(A, val)
            assert C.shape == (m + 1, n + 1)
            assert np.array_equal(C.query(i, j), ref.dominancecount(A, i, j))
            got, exp = S.query(i, j), ref.prefix_query(m, n, A.nnz, A.colptr, A.rowval, val, i, j)
            assert got.dtype == exp.dtype and np.array_equal(got, exp), (m, n)
            assert np.array_equal(got, ref.dominancesum(A, val, i, j)), (m, n)  # the restated DominanceSum structure of the reference
            assert S[m + 1, n + 1] == val.sum(dtype=val.dtype) and C[int(i[0]), int(j[0])] == C.query(i[:1], j[:1])[0]
            C.close(); S.close()
    for N in dims + [1000, 100000]:
        idx = rng.permutation(N) + 1
        val = (rng.integers(0, 2**63, N, dtype=np.uint64) << np.uint64(1)) + np.uint64(1)
        i = np.concatenate([rng.integers(1, N + 2, 200), [1, 1, N + 1, N + 1]])
        j = np.concatenate([rng.integers(1, N + 2, 200), [1, N + 1, 1, N + 1]])
        RC, RS = cp.rookcount(N, idx), cp.rooksum(N, idx, val)
        assert np.array_equal(RC.query(i, j), ref.prefix_query(N, N, N, None, idx, None, i, j))
        assert np.array_equal(RS.query(i, j), ref.prefix_query(N, N, N, None, idx, val, i, j))
        assert RC[N + 1, N + 1] == N
    with pytest.raises(TypeError):
        cp.dominancesum(A, np.ones(A.nnz))
    with pytest.raises(cp.CpbError):
        C = cp.dominancecount(A)
        C.query([A.m + 2], [1])


def test_declined_combinations_match_the_reference(ref):
    """Combinations the reference has no method for are declined on both sides (found by tests/fuzz_parity.py): the
    chunker-form K-DP calls f(j, j') without a part index (DynamicSplitter.jl:62-71) -- a MethodError for the
    partition-aware oracles; a weight that does not grow with the part is CPB_ERR_UNSUPPORTED, not an argument error."""
    rng = np.random.default_rng(310)
    A = sprand(rng, 12, 15, 0.3)
    Pi = ref.partition_stripe(ref.adjointpattern(A), 3, cp.EquiSplitter())
    for f in (cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6), cp.AffinePrimaryEdgeCutModel(0, 2, 1, 5)):
        for mtd in (cp.DynamicBottleneckChunker(f), cp.DynamicTotalChunker(f)):
            with pytest.raises(RuntimeError):
                ref.partition_stripe(A, 3, mtd, Pi)
            with pytest.raises(cp.CpbError) as e:
                cp.partition_stripe(A, 3, mtd, Pi)
            assert e.value.code == -2
    with pytest.raises(cp.CpbError) as e:
        cp.partition_stripe(A, 3, cp.DynamicTotalSplitter(cp.ConstrainedCost(AFF, cp.AffineWorkModel(1, 0, 0), 5)))
    assert e.value.code == -2


def test_plaid_with_primary_models(ref):
    """A genuinely 2-D alternation (bin/test_table_bottleneck.jl:47-55 style): columns by connectivity, then rows and
    columns in turn by the primary connectivity cost given the other side's partition."""
    A = synth.erdos_renyi(1500, 5)
    net = cp.AffineConnectivityModel(0, 10, 1, 100)
    comm = cp.AffinePrimaryConnectivityModel(0, 10, 1, 0, 100)
    for K in (4, 7):
        meth = cp.AlternatingPartitioner(cp.LazyBisectCostBottleneckSplitter(net, 0.01), cp.BisectCostBottleneckSplitter(comm, 0.01),
                                         cp.DynamicBottleneckSplitter(comm), cp.BisectIndexBottleneckSplitter(comm))
        (Pg, Fg), (Pr, Fr) = cp.partition_plaid(A, K, meth), ref.partition_plaid(A, K, meth)
        assert np.array_equal(Pg.spl, Pr.spl) and np.array_equal(Fg.spl, Fr.spl), K


def test_two_dimensional_pipeline(ref):
    """bin/test_table_bottleneck.jl:36-37: columns by nets, then rows / columns in turn by the primary (communication) and
    secondary (locality) costs given the other side's partition, with the exact index splitters."""
    A = synth.erdos_renyi(1200, 5)
    net = cp.AffineConnectivityModel(0, 10, 1, 100)
    comm = cp.AffinePrimaryConnectivityModel(0, 10, 1, 0, 100)
    loc = cp.AffineSecondaryConnectivityModel(0, 10, 1, 0, 100)
    for K in (3, 6):
        meth = cp.AlternatingNetPartitioner(cp.SparseHint(), cp.BisectIndexBottleneckSplitter(net), cp.FlipBisectIndexBottleneckSplitter(loc),
                                            cp.BisectIndexBottleneckSplitter(comm), cp.FlipBisectIndexBottleneckSplitter(loc))
        (Pg, Fg), (Pr, Fr) = cp.partition_plaid(A, K, meth), ref.partition_plaid(A, K, meth)
        assert np.array_equal(Pg.spl, Pr.spl) and np.array_equal(Fg.spl, Fr.spl), K


def test_degenerate_inputs(ref):
    """Empty matrices, empty columns/rows, K > n, single column -- the ragged cases."""
    z = np.zeros(0, dtype=np.int64)
    mats = [
        cp.SparseMatrixCSC(5, 4, np.ones(5, dtype=np.int64), z),                      # no nonzeros at all
        cp.SparseMatrixCSC(3, 1, np.array([1, 3]), np.array([1, 3])),                 # one column
        cp.SparseMatrixCSC(1, 6, np.array([1, 1, 2, 2, 2, 3, 3]), np.array([1, 1])),  # one row, mostly empty columns
        cp.SparseMatrixCSC(4, 4, np.array([1, 1, 1, 1, 5]), np.array([1, 2, 3, 4])),  # everything in the last column
    ]
    f = cp.AffineConnectivityModel(0, 3, 1, 3)
    s = cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 1)
    for A in mats:
        j = np.array([1, 1, A.n + 1, max(1, A.n)])
        jp = np.array([1, A.n + 1, A.n + 1, A.n + 1])
        assert np.array_equal(cp.netcount(A).query(j, jp), ref.netcount(A, j, jp))
        assert np.array_equal(cp.selfnetcount(A).query(j, jp), ref.selfnetcount(A, j, jp))
        for K in [1, 2, 7]:
            for mtd in [cp.DynamicBottleneckSplitter(f), cp.DynamicTotalSplitter(f), cp.BisectCostBottleneckSplitter(f, 0.1),
                        cp.LazyBisectCostBottleneckSplitter(f, 0.01), cp.BisectCostBottleneckSplitter(cp.AffineWorkModel(0, 10, 1), 0.1)]:
                g, r = cp.partition_stripe(A, K, mtd), ref.partition_stripe(A, K, mtd)
                assert np.array_equal(g.spl, r.spl), (A, K, type(mtd).__name__, g.spl, r.spl)
            if A.m == A.n:
                mtd = cp.LazyBisectCostBottleneckSplitter(s, 0.1)
                assert np.array_equal(cp.partition_stripe(A, K, mtd).spl, ref.partition_stripe(A, K, mtd).spl)
        for w_max in [1, 3]:
            for mtd in [cp.DynamicTotalChunker(f, w_max), cp.ConvexTotalChunker(cp.ConstrainedCost(f, cp.VertexCount(), w_max)), cp.OverlapChunker(0.5, w_max), cp.StrictChunker(w_max)]:
                g, r = cp.pack_stripe(A, mtd), ref.pack_stripe(A, mtd)
                assert np.array_equal(g.spl, r.spl), (A, w_max, type(mtd).__name__, g.spl, r.spl)
        B = cp.adjointpattern(A)
        Br = ref.adjointpattern(A)
        assert np.array_equal(B.colptr, Br.colptr) and np.array_equal(B.rowval, Br.rowval)


def test_sharded_solve_emulated_ranks_and_single_rank(ref):
    """csrc/sharded.cu on one GPU: the block-wise link construction with the carried "last position" array and rounds of
    world x 15 thresholds, the ranks played one after the other (cpb_partition_stripe_sharded_emulated), and the real entry
    point with a world of one (no communicator)."""
    A = synth.erdos_renyi(30000, 10)
    cases = [(A, 16, 0.01), (synth.rmat(14, 16 << 14), 128, 0.01), (synth.laplacian5(40), 7, 0.001),
             (synth.banded(3000, 20), 5, 0.05), (cp.SparseMatrixCSC(4, 3, [1, 1, 1, 1], np.zeros(0, dtype=np.int64)), 2, 0.1)]
    runs = [(M, K, mtd) for M, K, eps in cases
            for mtd in (cp.LazyBisectCostBottleneckSplitter(AFF, eps), cp.BisectCostBottleneckSplitter(cp.AffineConnectivityModel(0.0, 3.0, 1.0, 7.0), eps))]
    sym = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 4)
    runs += [(A, 16, cp.BisectCostBottleneckSplitter(AFF, 0.01)), (A, 64, cp.LazyBisectCostBottleneckSplitter(AFF, 0.001)),
             (synth.random_geometric(20000), 32, cp.LazyBisectCostBottleneckSplitter(sym, 0.1))]
    for M, K, mtd in runs:
        exp = ref.partition_stripe(M, K, mtd).spl
        for world in (1, 2, 3, 4, 8):
            got = cp.partition_stripe_sharded_emulated(M, K, mtd, world).spl
            assert np.array_equal(got, exp), (M.n, K, type(mtd).__name__, world)
        assert np.array_equal(cp.partition_stripe_sharded(M, K, mtd).spl, exp), (M.n, K, type(mtd).__name__, "world of one")
    # the sharded solve streams links: a work model (bisection on the dominance index) is refused, emulated or not
    for K, work in ((4, cp.LazyBisectCostBottleneckSplitter(cp.AffineWorkModel(0, 1, 1), 0.1)), (8, cp.BisectCostBottleneckSplitter(cp.AffineWorkModel(0, 10, 1), 0.01))):
        with pytest.raises(cp.CpbError):
            cp.partition_stripe_sharded(A, K, work)
        with pytest.raises(cp.CpbError):
            cp.partition_stripe_sharded_emulated(A, K, work, 2)


def test_c_abi_example_binary(ref):
    """The boundary from plain C (examples/c_abi_example.c, built by __graft_entry__.build()): no Python
    in the call path, exactly what a Julia ccall would do."""
    import os
    import subprocess

    exe = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "c_abi_example")
    if not os.path.exists(exe):
        pytest.skip("examples/c_abi_example not built")
    A = synth.erdos_renyi(4000, 8)
    K, eps = 12, 0.01
    text = f"{A.m} {A.n} {A.nnz} {K} {eps}\n" + " ".join(map(str, A.colptr.tolist())) + "\n" + " ".join(map(str, A.rowval.tolist())) + "\n"
    out = subprocess.run([exe], input=text, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    lines = dict(l.split(" ", 1) for l in out.stdout.strip().splitlines())
    mtd = cp.BisectCostBottleneckSplitter(AFF, eps)
    exp = ref.partition_stripe(A, K, mtd)
    assert list(map(int, lines["spl"].split())) == exp.spl.tolist()
    assert tuple(map(float, lines["bound"].split())) == ref.bound_stripe(A, K, AFF)
    assert float(lines["value"]) == ref.bottleneck_value(A, exp, AFF)
    # the other ABI families, each called from plain C
    assert list(map(int, lines["spl_exact"].split())) == ref.partition_stripe(A, K, cp.BisectIndexBottleneckSplitter(AFF)).spl.tolist()
    Q, n = 6, A.n
    qj = np.array([1 + (n * t) // (2 * Q) for t in range(Q)])
    qjp = np.array([n + 1 - (n * t) // (3 * Q) for t in range(Q)])
    assert list(map(float, lines["queries"].split())) == ref.oracle_query(AFF, A, qj, qjp).tolist()
    assert list(map(int, lines["nets"].split())) == ref.netcount(A, qj, qjp).tolist()
    chunker = cp.DynamicTotalChunker(cp.ConstrainedCost(AFF, cp.VertexCount(), 8))
    Pc = ref.pack_stripe(A, chunker)
    tok = lines["chunks"].split()
    assert int(tok[0]) == Pc.K and float(tok[2]) == ref.total_value(A, Pc, AFF) and list(map(int, tok[4:])) == Pc.spl[: min(Pc.K, 8) + 1].tolist()
    nn = []
    Po = ref.pack_stripe(A, cp.OverlapChunker(0.9, 8), n_nets=nn)
    tok = lines["overlap"].split()
    assert int(tok[0]) == Po.K and int(tok[2]) == int(np.sum(nn[0]))
    At = ref.adjointpattern(A)
    tok = lines["adjoint"].split()
    assert (int(tok[0]), int(tok[1]), int(tok[2])) == (At.m, At.n, At.nnz + 1)
    assert int(tok[4]) == int(np.sum((np.arange(At.nnz) % 7 + 1) * At.rowval))
    dom = ref.dominancecount(A, [A.m // 2 + 1, A.m + 1], [A.n // 3 + 1, A.n + 1])
    assert list(map(int, lines["dominance"].split())) == dom.tolist()
    assert list(map(int, lines["spl_sharded"].split())) == ref.partition_stripe(A, K, cp.LazyBisectCostBottleneckSplitter(AFF, eps)).spl.tolist()
