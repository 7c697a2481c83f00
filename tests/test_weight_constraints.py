"""ConstrainedCost(f, w, w_max) with a count weight (Costs.jl:105-147): w an integer AffineConnectivityModel or
AffineMonotonizedSymmetricConnectivityModel (a part's footprint: distinct rows, or bytes of columns, entries and rows).

CPU: the oracle's constrained splitters, run with a count weight by tests/weighted_oracle.py, are optimal against a brute
force over the cost matrix masked where the weight's definition exceeds w_max, the chunker K-form equals the splitter form,
and the witness (tests/weighted_witness.py: a set-based weight and a literal transliteration of DynamicSplitter.jl:144-247)
equals the oracle.  GPU: the device equals the oracle split vector for split vector, cpb_weight_windows equals the
definition, and the refusals return the documented codes."""
import ctypes

import numpy as np
import pytest

import chainb200 as cp
import weighted_oracle as wref
import weighted_witness as wit
from chainb200 import synth
from helpers import brute_optimum, check_split, cost_matrix, objective, ref_cost, sprand

WEIGHTS = [cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 1, 1, 2), cp.AffineConnectivityModel(3, 0, 0, 1)]
SQUARE_WEIGHTS = [cp.AffineMonotonizedSymmetricConnectivityModel(0, 1, 1, 1, 2), cp.AffineMonotonizedSymmetricConnectivityModel(1, 0, 2, 1, 0)]
DYNAMIC = [(True, cp.DynamicTotalSplitter), (False, cp.DynamicBottleneckSplitter)]


def weights_for(A):
    return WEIGHTS + (SQUARE_WEIGHTS if A.m == A.n else [])


def masked(C, Wm, w_max):
    Cw = C.copy()
    Cw[Wm > w_max] = np.inf
    return Cw


def w_max_cases(Wm, n, K):
    """tight (about 1.5 n / K columns' worth), wide (everything fits) and infeasible (below w(j, j))"""
    full = int(Wm[1, n + 1])
    alpha = int(Wm[1, 1])
    return [max(alpha, int(np.ceil(1.5 * full / K))), full, alpha - 1]


def small_inputs(fixtures, seed):
    rng = np.random.default_rng(seed)
    return [fixtures["LPnetlib/lpi_itest6"], sprand(rng, 6, 1, 0.5), sprand(rng, 7, 7, 0.35), sprand(rng, 5, 11, 0.3), sprand(rng, 9, 9, 0.2),
            sprand(rng, 12, 12, 0.25)]


def test_weighted_dynamic_splitters_are_optimal(ref, fixtures):
    """DynamicSplitter.jl:206-247 with a count weight: optimum among the weight-feasible partitions, or the degenerate
    partition when none exists (the pattern of test_dynamic_splitter_constrained_pin_weights)."""
    mats = small_inputs(fixtures, 701) + [fixtures["Pajek/GD99_c"]]
    f = cp.AffineConnectivityModel(0, 1, 0, 2)
    for A in mats:
        n = A.n
        C = cost_matrix(f, A)
        for w in weights_for(A):
            Wm = cost_matrix(w, A)
            for K in [1, 2, 3, 4, 8]:
                for w_max in w_max_cases(Wm, n, K):
                    Cw = masked(C, Wm, w_max)
                    for total, S in DYNAMIC:
                        Phi = wref.partition_stripe(A, K, S(cp.ConstrainedCost(f, w, w_max)))
                        opt = brute_optimum(Cw, n, K, total)
                        if np.isinf(opt):
                            assert Phi.spl.tolist() == [1] * K + [n + 1], (w, w_max, K)
                        else:
                            check_split(Phi.spl, n, K)
                            assert objective(Cw, Phi.spl, total) == opt, (w, w_max, K, Phi.spl)


def test_weighted_convex_and_concave_splitters_are_optimal(ref, fixtures):
    """ConvexTotalSplitter{<:ConstrainedCost} (ConvexTotalChunker.jl:167-265) on the quadrangle-inequality models and
    ConcaveTotalSplitter{<:ConstrainedCost} (ConcaveTotalChunker.jl:143-181) on the work model: optimal total cost among the
    weight-feasible partitions, degenerate when infeasible."""
    cases = [(cp.ConvexTotalSplitter, cp.AffineConnectivityModel(0, 3, 1, 3)), (cp.ConvexTotalSplitter, cp.AffineWorkModel(1, 2, 1)),
             (cp.ConcaveTotalSplitter, cp.AffineWorkModel(1, 2, 1)), (cp.ConcaveTotalSplitter, cp.AffineWorkModel(0, 1, 0))]
    for A in small_inputs(fixtures, 702):
        n = A.n
        for S, f in cases:
            C = cost_matrix(f, A)
            for w in weights_for(A):
                Wm = cost_matrix(w, A)
                for K in [1, 2, 3, 4, 8]:
                    for w_max in w_max_cases(Wm, n, K):
                        Cw = masked(C, Wm, w_max)
                        Phi = wref.partition_stripe(A, K, S(cp.ConstrainedCost(f, w, w_max)))
                        opt = brute_optimum(Cw, n, K, True)
                        if np.isinf(opt):
                            assert Phi.spl.tolist() == [1] * K + [n + 1], (S.__name__, w, w_max, K)
                        else:
                            check_split(Phi.spl, n, K)
                            assert objective(Cw, Phi.spl, True) == opt, (S.__name__, f, w, w_max, K, Phi.spl)


def test_weighted_chunker_kform_equals_splitter_form(ref, fixtures):
    """DynamicSplitter.jl:249-314 (the K-DP with the part index as the inner loop) gives the splitter form's split vectors
    under count weights too -- the device serves both forms with the splitter-form DP."""
    rng = np.random.default_rng(703)
    mats = small_inputs(fixtures, 703) + [fixtures["Pajek/GD99_c"], fixtures["LPnetlib/lp_blend"], sprand(rng, 30, 60, 0.08)]
    for A in mats:
        for f in [cp.AffineConnectivityModel(0, 1, 0, 2), cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0)]:
            for w in weights_for(A):
                Wm = ref.oracle_query(w, A, [1], [A.n + 1])
                for K in [1, 2, 3, 4, 8]:
                    for w_max in [int(np.ceil(1.5 * Wm[0] / K)), int(Wm[0]), int(w.alpha) - 1]:
                        spec = cp.ConstrainedCost(f, w, w_max)
                        for S, Ch in [(cp.DynamicTotalSplitter, cp.DynamicTotalChunker), (cp.DynamicBottleneckSplitter, cp.DynamicBottleneckChunker)]:
                            a = wref.partition_stripe(A, K, S(spec)).spl.tolist()
                            b = wref.partition_stripe(A, K, Ch(spec)).spl.tolist()
                            assert a == b, (S.__name__, f, w, w_max, K)


def test_set_weight_matches_model(fixtures):
    """The witness's set-based weight is the weight model's cost by definition (tests/helpers.ref_cost)."""
    for A in small_inputs(fixtures, 704):
        for w in weights_for(A):
            kind = "conn" if w.kind == cp.MODEL_CONNECTIVITY else "monosym"
            sw = wit.SetWeight(A, kind, w.coef)
            for j in range(1, A.n + 2):
                for jp in range(j, A.n + 2):
                    assert sw(j, jp) == ref_cost(w, A, j, jp), (w, j, jp)


def test_witness_equals_oracle_weighted(ref):
    """The witness (column_constraints + the constrained DynamicSplitter, DynamicSplitter.jl:144-247, with distinct rows
    counted with Python sets) equals the oracle on random tiny matrices with many ties (0/1 costs, small w_max)."""
    rng = np.random.default_rng(705)
    for case in range(300):
        m, n = int(rng.integers(1, 8)), int(rng.integers(1, 12))
        if case % 3 == 0:
            m = n
        A = sprand(rng, m, n, float(rng.choice([0.15, 0.3, 0.5])))
        coef = tuple(int(x) for x in rng.integers(0, 2, 4))
        f = cp.AffineConnectivityModel(*coef)
        if m == n and rng.random() < 0.4:
            wc = (int(rng.integers(0, 2)), int(rng.integers(0, 2)), int(rng.integers(0, 3)), int(rng.integers(0, 3)), int(rng.integers(-1, 3)))
            w, kind = cp.AffineMonotonizedSymmetricConnectivityModel(*wc), "monosym"
        else:
            wc = (int(rng.integers(0, 2)), int(rng.integers(0, 2)), int(rng.integers(0, 2)), int(rng.integers(0, 3)))
            w, kind = cp.AffineConnectivityModel(*wc), "conn"
        w_max = int(rng.integers(0, 8))
        K = int(rng.integers(1, 6))
        for total, S in DYNAMIC:
            got = wit.dynamic_splitter_constrained(wit.Conn(A, coef), K, total, wit.SetWeight(A, kind, wc), w_max)
            exp = wref.partition_stripe(A, K, S(cp.ConstrainedCost(f, w, w_max))).spl.tolist()
            assert got == exp, (case, S.__name__, coef, w, w_max, K)


def test_count_weight_refusals_on_the_host():
    """pack_stripe keeps refusing count weights, the cpb_constraint form cannot hold one, and a monotonized-symmetric weight
    is refused when a non-contiguous row partition renames the rows (no device needed for any of these)."""
    spec = cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 0, 0, 1), 5)
    with pytest.raises(TypeError, match="not built"):
        cp.pack_stripe(cp.SparseMatrixCSC(3, 3, [1, 2, 3, 4], [1, 2, 3]), cp.ConvexTotalChunker(spec))
    with pytest.raises(TypeError):
        spec.constraint()
    assert spec.count_weight() is spec.w
    assert cp.ConstrainedCost(spec.f, cp.AffineWorkModel(0, 1, 1), 5).count_weight() is None
    assert cp.ConstrainedCost(spec.f, cp.VertexCount(), 5).count_weight() is None
    A = cp.SparseMatrixCSC(3, 3, [1, 2, 3, 4], [1, 2, 3])
    mono = cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 0, 1, 0), 5)
    with pytest.raises(TypeError, match="diagonal"):
        cp.oracle_stripe(mono, A, cp.MapPartition(2, np.array([2, 1, 2])))


# ------------------------------------------------------------------------------------------------------------------- GPU

METHODS = [cp.DynamicBottleneckSplitter, cp.DynamicTotalSplitter, cp.DynamicBottleneckChunker, cp.DynamicTotalChunker, cp.ConvexTotalSplitter,
           cp.ConcaveTotalSplitter]
DEVICE_WEIGHTS = [cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 1, 1, 2), cp.AffineConnectivityModel(3, 0, 0, 1),
                  cp.AffineMonotonizedSymmetricConnectivityModel(0, 1, 1, 1, 2)]
FS = [cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0)]


def _full_weight(ref, w, A):
    return int(ref.oracle_query(w, A, [1], [A.n + 1])[0])


@pytest.mark.gpu
@pytest.mark.parametrize("mk", METHODS, ids=lambda m: m.__name__)
@pytest.mark.parametrize("w", DEVICE_WEIGHTS, ids=repr)
def test_weighted_device_equals_oracle(ref, fixtures, mk, w):
    """Every constrained partition_stripe family x count weight x Int64 / Float64 cost x K: identical split vectors."""
    rng = np.random.default_rng(706)
    mats = [fixtures[k] for k in sorted(fixtures)] + [sprand(rng, 6, 1, 0.5), sprand(rng, 12, 12, 0.3), sprand(rng, 40, 200, 0.1), synth.laplacian5(20)]
    if mk is cp.ConcaveTotalSplitter:  # one device thread walks the queue: keep the sequential form on the smaller inputs
        mats = [A for A in mats if A.n <= 400]
    for A in mats:
        if w.kind == cp.MODEL_MONOSYM and A.m != A.n:
            continue
        full = _full_weight(ref, w, A)
        for f in FS:
            for K in [1, 2, 3, 4, 8, 60]:
                for w_max in [max(int(w.alpha), int(np.ceil(1.5 * full / K))), full, int(w.alpha) - 1]:
                    spec = mk(cp.ConstrainedCost(f, w, w_max))
                    g, r = cp.partition_stripe(A, K, spec), wref.partition_stripe(A, K, spec)
                    assert np.array_equal(g.spl, r.spl), (A.m, A.n, f, K, w_max, g.spl, r.spl)
    B = synth.banded(3000, 6, 3)  # windows wider than 64 columns: the warp-per-column layers
    full = _full_weight(ref, w, B)
    Ks = [1, 2, 3, 4, 8, 60] if mk is not cp.ConcaveTotalSplitter else [1, 2, 8]
    for K in Ks:
        w_max = max(int(np.ceil(1.5 * full / K)), 200 * max(1, int(w.coef[3])) + int(w.alpha))
        for f in FS:
            spec = mk(cp.ConstrainedCost(f, w, w_max))
            g, r = cp.partition_stripe(B, K, spec), wref.partition_stripe(B, K, spec)
            assert np.array_equal(g.spl, r.spl), ("banded", f, K, w_max)


@pytest.mark.gpu
def test_weight_windows_definition(ref, fixtures):
    """cpb_weight_windows: first_fit and reach equal their definitions over the weight's brute-force cost matrix."""
    rng = np.random.default_rng(707)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], fixtures["HB/west0132"], sprand(rng, 6, 1, 0.5), sprand(rng, 12, 12, 0.3),
            sprand(rng, 40, 200, 0.1), synth.laplacian5(20), cp.SparseMatrixCSC(5, 4, [1, 1, 1, 1, 1], np.zeros(0, dtype=np.int64))]
    for A in mats:
        n1 = A.n + 1
        jj, jjp = np.triu_indices(n1)
        for w in DEVICE_WEIGHTS + [cp.AffineMonotonizedSymmetricConnectivityModel(2, 0, 3, 1, -1)]:
            if w.kind == cp.MODEL_MONOSYM and A.m != A.n:
                continue
            Wm = np.full((n1 + 1, n1 + 1), np.inf)
            Wm[jj + 1, jjp + 1] = ref.oracle_query(w, A, jj + 1, jjp + 1)
            full = int(Wm[1, n1])
            for w_max in sorted({int(w.alpha) - 1, int(w.alpha), max(1, full // 7), max(1, full // 2), full}):
                ocl = cp.oracle_stripe(cp.ConstrainedCost(cp.AffineWorkModel(0, 1, 0), w, w_max), A)
                try:
                    ff, rc = ocl.weight_windows()
                finally:
                    ocl.close()
                fits = (Wm <= w_max) | np.eye(n1 + 1, dtype=bool)
                for c in range(1, n1 + 1):
                    assert ff[c - 1] == min(j for j in range(1, c + 1) if fits[j, c]), (w, w_max, c)
                    assert rc[c - 1] == max(jp for jp in range(c, n1 + 1) if fits[c, jp]), (w, w_max, c)


def _weighted_abi(f_ocl, code, w_ocl, w_max, K):
    spl = np.empty(K + 1, dtype=np.int64)
    rc = cp.load_library().cpb_partition_stripe_weighted(f_ocl._h, code, w_ocl._h, int(w_max), 0.0, int(K), ctypes.c_void_p(spl.ctypes.data))
    return rc, spl


@pytest.mark.gpu
def test_work_weight_through_weighted_entry(fixtures):
    """An AffineWorkModel weight through cpb_partition_stripe_weighted takes the cpb_constraint path: identical vectors."""
    rng = np.random.default_rng(708)
    for A in [fixtures["Pajek/GD99_c"], sprand(rng, 40, 200, 0.1), synth.laplacian5(20)]:
        dm = cp.device_matrix(A)
        for wm, w_max in [((0, 1, 0), 9), ((0, 1, 1), 30), ((2, 1, 2), 60), ((0, 0, 1), 12)]:
            f = cp.AffineConnectivityModel(0, 3, 1, 3)
            focl, wocl = cp.oracle_stripe(f, dm), cp.oracle_stripe(cp.AffineWorkModel(*wm), dm)
            try:
                for mk, code in [(cp.DynamicTotalSplitter, cp.SPLIT_DYNAMIC_TOTAL), (cp.DynamicBottleneckSplitter, cp.SPLIT_DYNAMIC_BOTTLENECK),
                                 (cp.ConvexTotalSplitter, cp.SPLIT_CONVEX_TOTAL), (cp.ConcaveTotalSplitter, cp.SPLIT_CONCAVE_TOTAL)]:
                    for K in [1, 3, 8]:
                        rc, spl = _weighted_abi(focl, code, wocl, w_max, K)
                        assert rc == 0, cp.load_library().cpb_last_error()
                        exp = cp.partition_stripe(dm, K, mk(cp.ConstrainedCost(f, cp.AffineWorkModel(*wm), w_max)))
                        assert np.array_equal(spl, exp.spl), (wm, w_max, mk.__name__, K)
            finally:
                focl.close()
                wocl.close()
        dm.close()


@pytest.mark.gpu
def test_weighted_query_masks(ref, fixtures):
    """oracle_stripe(ConstrainedCost(f, w, w_max)).query: f's cost where w(j, j') <= w_max, +inf elsewhere."""
    rng = np.random.default_rng(709)
    for A in [fixtures["Pajek/GD99_c"], sprand(rng, 40, 200, 0.1)]:
        j = rng.integers(1, A.n + 2, 3000)
        jp = rng.integers(1, A.n + 2, 3000)
        j, jp = np.minimum(j, jp), np.maximum(j, jp)
        for w in DEVICE_WEIGHTS:
            if w.kind == cp.MODEL_MONOSYM and A.m != A.n:
                continue
            f = cp.AffineConnectivityModel(0, 3, 1, 3)
            wv = ref.oracle_query(w, A, j, jp)
            w_max = int(np.median(wv))
            ocl = cp.oracle_stripe(cp.ConstrainedCost(f, w, w_max), A)
            try:
                got = ocl.query(j, jp)
            finally:
                ocl.close()
            exp = np.where(wv <= w_max, ref.oracle_query(f, A, j, jp), np.inf)
            assert np.array_equal(got, exp), w


@pytest.mark.gpu
def test_weighted_error_codes(fixtures):
    """Float64 weights, negative betas, the non-monotone / part-aware weight models, the Bisect / Flip / Equi methods:
    CPB_ERR_UNSUPPORTED; a weight oracle over another matrix: CPB_ERR_ARG."""
    A = fixtures["Pajek/GD99_c"]
    f = cp.AffineConnectivityModel(0, 3, 1, 3)
    for w in [cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0), cp.AffineConnectivityModel(0, -1, 0, 1), cp.AffineConnectivityModel(0, 0, 0, -1),
              cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, -1, 1, 0), cp.AffineWorkModel(0, -1, 2), cp.AffineSymmetricConnectivityModel(0, 0, 0, 1, 1),
              cp.AffineHyperedgeCutModel(0, 0, 0, 1, 1), cp.AffineSymmetricEdgeCutModel(0, 0, 1, 1), cp.AffineEnvelopeModel(0, 0, 0, 1)]:
        with pytest.raises(cp.CpbError) as e:
            cp.partition_stripe(A, 4, cp.DynamicTotalSplitter(cp.ConstrainedCost(f, w, 50)))
        assert e.value.code == -2, w
    dm = cp.device_matrix(A)
    focl, wocl = cp.oracle_stripe(f, dm), cp.oracle_stripe(cp.AffineConnectivityModel(0, 0, 0, 1), dm)
    other = cp.oracle_stripe(cp.AffineConnectivityModel(0, 0, 0, 1), A)
    try:
        for code in [cp.SPLIT_BISECT_COST, cp.SPLIT_LAZY_BISECT_COST, cp.SPLIT_BISECT_INDEX, cp.SPLIT_FLIP_BISECT_COST, cp.SPLIT_LAZY_FLIP_BISECT_COST,
                     cp.SPLIT_FLIP_BISECT_INDEX, cp.SPLIT_EQUI]:
            assert _weighted_abi(focl, code, wocl, 50, 4)[0] == -2, code
        assert _weighted_abi(focl, cp.SPLIT_DYNAMIC_TOTAL, other, 50, 4)[0] == -1
        assert _weighted_abi(focl, cp.SPLIT_DYNAMIC_TOTAL, wocl, 50, 4)[0] == 0
    finally:
        focl.close()
        wocl.close()
        other.close()
        dm.close()


@pytest.mark.gpu
def test_weighted_random_differential(ref):
    """Seeded random cases: input, count weight, cost type, method, K and w_max drawn at random; device == oracle."""
    rng = np.random.default_rng(710)
    for case in range(300):
        m, n = int(rng.integers(1, 60)), int(rng.integers(1, 160))
        if case % 2 == 0:
            m = n
        A = sprand(rng, m, n, float(rng.choice([0.02, 0.08, 0.2])))
        if m == n and rng.random() < 0.4:
            w = cp.AffineMonotonizedSymmetricConnectivityModel(int(rng.integers(0, 3)), int(rng.integers(0, 3)), int(rng.integers(0, 3)),
                                                               int(rng.integers(0, 3)), int(rng.integers(-1, 4)))
        else:
            w = cp.AffineConnectivityModel(int(rng.integers(0, 3)), int(rng.integers(0, 3)), int(rng.integers(0, 3)), int(rng.integers(0, 4)))
        f = FS[int(rng.integers(0, 2))]
        mk = METHODS[int(rng.integers(0, len(METHODS)))]
        K = int(rng.choice([1, 2, 3, 4, 5, 8, 13, 60]))
        full = _full_weight(ref, w, A)
        w_max = int(rng.integers(int(w.alpha) - 1, max(int(w.alpha), int(2 * full / K)) + 2))
        spec = mk(cp.ConstrainedCost(f, w, w_max))
        g, r = cp.partition_stripe(A, K, spec), wref.partition_stripe(A, K, spec)
        assert np.array_equal(g.spl, r.spl), (case, m, n, w, f, mk.__name__, K, w_max, g.spl, r.spl)


@pytest.mark.gpu
def test_weighted_partition_plaid(ref, fixtures):
    """partition_plaid reaches count weights through partition_stripe (here with a non-contiguous row partition on the
    second solve: the weight is built on the renamed matrix)."""
    A = fixtures["HB/west0132"]
    f = cp.AffineConnectivityModel(0, 3, 1, 3)
    w = cp.AffineConnectivityModel(0, 0, 0, 1)
    spec = cp.ConstrainedCost(f, w, 40)
    for method in [cp.AlternatingPartitioner(cp.DynamicTotalSplitter(spec), cp.DynamicTotalSplitter(spec)),
                   cp.SymmetricPartitioner(cp.DynamicBottleneckSplitter(spec))]:
        g = cp.partition_plaid(A, 6, method)
        r = wref.partition_plaid(A, 6, method)
        assert np.array_equal(g[0].spl, r[0].spl) and np.array_equal(g[1].spl, r[1].spl)
    Pi = cp.MapPartition(3, np.array([1 + (i * 7) % 3 for i in range(A.m)]))
    g = cp.partition_stripe(A, 5, cp.DynamicTotalSplitter(spec), Pi)
    r = cp.partition_stripe(A, 5, cp.DynamicTotalSplitter(spec))
    assert np.array_equal(g.spl, r.spl)  # a connectivity weight and f ignore the row names
