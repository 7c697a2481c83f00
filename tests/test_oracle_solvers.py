"""Pins the CPU oracle's cost models and split-point searches by the properties the reference's own
tests check (test/test_Costs.jl, test/test_Partitioners.jl): model == brute-force definition,
bound sandwich, (eps-)optimality against an independent brute-force DP, chunk constraints -- plus
the per-algorithm tie-breaking rules of SURVEY.md App. B re-derived independently."""
import numpy as np
import pytest

import chainb200 as cp
from helpers import (brute_chunk_optimum, brute_optimum, check_split, col_rows, cost_matrix, objective, ref_cost,
                     ref_netcount, sprand)

HINTS = [cp.NoHint(), cp.SparseHint(), cp.StepHint()]

AFFINE_MODELS = [
    cp.AffineWorkModel(0, 10, 1),
    cp.AffineWorkModel(0, 1, 0),
    cp.AffineConnectivityModel(0, 0, 0, 1),
    cp.AffineConnectivityModel(0, 3, 1, 3),
    cp.AffineConnectivityModel(0, 10, 1, 100),
    cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0),
    cp.AffineConnectivityModel(-0.5, 0.0, 0.0, 1.0),
    cp.AffineEnvelopeModel(1, 2, 3, 4),
]
SQUARE_MODELS = [
    cp.AffineMonotonizedSymmetricConnectivityModel(10, 10, 10, 10, 0),
    cp.AffineMonotonizedSymmetricConnectivityModel(10, 10, 10, 100, 8),
    cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5),
    cp.AffineSymmetricConnectivityModel(1, 1, 1, 1, 1),
    cp.AffineSymmetricConnectivityModel(0, 0, 0, 0, 1),
    cp.AffineHyperedgeCutModel(0, 0, 0, 1, 1),
    cp.AffineHyperedgeCutModel(0, 0, 0, -1, 0),
    cp.AffineSymmetricEdgeCutModel(10, 10, 10, 100),
    cp.AffineSymmetricEdgeCutModel(1, 1, 1, 1),
]


def all_pairs(n):
    return [(j, jp) for j in range(1, n + 2) for jp in range(j, n + 2)]


def test_models_match_definitions(ref):
    """test_Costs.jl:24-30,66-79: oracle value == model evaluated on brute-force counts."""
    rng = np.random.default_rng(10)
    for m in [1, 2, 3, 5, 8, 13, 21]:
        A = sprand(rng, m, m, 0.3)
        pairs = all_pairs(m)
        j = [p[0] for p in pairs]
        jp = [p[1] for p in pairs]
        for mdl in AFFINE_MODELS + SQUARE_MODELS:
            if mdl.kind == cp.MODEL_ENVELOPE:
                continue
            exp = [float(ref_cost(mdl, A, a, b)) for a, b in pairs]
            for hint in HINTS:
                got = ref.oracle_query(mdl, A, j, jp, hint=hint)
                assert got.tolist() == exp, (mdl, hint, m)
        env = cp.AffineEnvelopeModel(1, 2, 3, 4)
        pe = [p for p in pairs if p[0] < p[1]]
        got = ref.oracle_query(env, A, [p[0] for p in pe], [p[1] for p in pe])
        assert got.tolist() == [float(ref_cost(env, A, a, b)) for a, b in pe]


def test_block_oracle_random_access(ref):
    """test_Costs.jl:106-122 + SURVEY E11: BlockComponentCostStepOracle under random access."""
    rng = np.random.default_rng(11)
    models = [
        cp.BlockComponentCostModel(int, 0, 0, (2, cp.identity), (2, lambda x: 2 * x)),
        cp.BlockComponentCostModel(int, cp.identity, lambda x: 3 * x, (2, cp.identity), (2, lambda x: 2 * x)),
        cp.BlockComponentCostModel(int, 1, 3, (1, cp.identity), (1, cp.identity)),
        cp.ColumnBlockComponentCostModel(int, 3, lambda w: 1 + w),
    ]
    for m in [3, 7, 12, 20]:
        for u in [1, 2, 3, 4]:
            A = sprand(rng, m, m + 2, 0.25)
            Pi = ref.pack_stripe(ref.adjointpattern(A), cp.EquiChunker(u))
            pairs = all_pairs(A.n)
            order = rng.permutation(len(pairs))
            pairs = [pairs[t] for t in order]
            for mdl in models:
                got = ref.oracle_query(mdl, A, [p[0] for p in pairs], [p[1] for p in pairs], Pi=Pi, hint=cp.StepHint())
                exp = [float(ref_cost(mdl, A, a, b, Pi)) for a, b in pairs]
                assert got.tolist() == exp


def test_bound_sandwich(ref):
    """test_Costs.jl:26-30: 0 <= c_lo <= bottleneck_value <= c_hi for any K-partition."""
    rng = np.random.default_rng(12)
    for m in range(1, 40, 3):
        A = sprand(rng, m, m, 0.125)
        for K in [1, 2, 3, 4]:
            spl = np.concatenate(([1], np.sort(rng.integers(1, m + 2, K - 1)), [m + 1]))
            Phi = cp.SplitPartition(K, spl)
            for mdl in [cp.AffineWorkModel(0, 1, 1), cp.AffineConnectivityModel(0, 1, 1, 1),
                        cp.AffineMonotonizedSymmetricConnectivityModel(10, 10, 10, 100, 8),
                        cp.AffineConnectivityModel(0.0, 1.0, 1.0, 1.0)]:
                lo, hi = ref.bound_stripe(A, K, mdl)
                v = ref.bottleneck_value(A, Phi, mdl)
                assert 0 <= lo <= v <= hi
                assert v == max(ref_cost(mdl, A, int(spl[k]), int(spl[k + 1])) for k in range(K))


def rightmost_dp(C, n, K, total):
    """Independent statement of App. B: per layer, the LARGEST j among minimisers."""
    g = (lambda a, b: a + b) if total else max
    cst = np.full((K + 1, n + 2), np.inf)
    ptr = np.zeros((K + 1, n + 2), dtype=np.int64)
    for jp in range(1, n + 2):
        cst[1, jp] = C[1, jp]
        ptr[1, jp] = 1
    for k in range(2, K + 1):
        for jp in range(1, n + 2):
            vals = [g(cst[k - 1, j], C[j, jp]) for j in range(1, jp + 1)]
            v = min(vals)
            cst[k, jp] = v
            ptr[k, jp] = max(j for j, x in zip(range(1, jp + 1), vals) if x == v)
    spl = [0] * (K + 1)
    spl[K] = n + 1
    for k in range(K, 0, -1):
        spl[k - 1] = int(ptr[k, spl[k]])
    return spl


def test_dynamic_splitters(ref, fixtures):
    """test_Partitioners.jl:95-113,154-170: Dynamic == Reference optimum; exact rightmost-tie splits."""
    rng = np.random.default_rng(13)
    mats = [fixtures["LPnetlib/lpi_itest6"]] + [sprand(rng, m, n, 0.2) for m in [1, 2, 4, 8] for n in [1, 3, 8, 12]]
    for A in mats:
        models = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(2, 0, 0, 1)]
        if A.m == A.n:
            models.append(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5))
        for mdl in models:
            C = cost_matrix(mdl, A)
            for K in [1, 2, 3, 4, 8]:
                for total, mtd in [(False, cp.DynamicBottleneckSplitter(mdl)), (True, cp.DynamicTotalSplitter(mdl))]:
                    Phi = ref.partition_stripe(A, K, mtd)
                    check_split(Phi.spl, A.n, K)
                    assert objective(C, Phi.spl, total) == brute_optimum(C, A.n, K, total)
                    assert Phi.spl.tolist() == rightmost_dp(C, A.n, K, total)


def test_dynamic_splitter_constrained(ref):
    """DynamicSplitter.jl:206-247: optimum among width-feasible partitions, or the degenerate one."""
    rng = np.random.default_rng(14)
    for n in [1, 3, 6, 10]:
        A = sprand(rng, 6, n, 0.3)
        mdl = cp.AffineConnectivityModel(0, 0, 0, 1)
        C = cost_matrix(mdl, A)
        for w_max in [2, 4]:
            Cw = C.copy()
            for j in range(1, n + 2):
                for jp in range(j, n + 2):
                    if jp - j > w_max:
                        Cw[j, jp] = np.inf
            for K in [1, 2, 3, 4, 8]:
                f = cp.ConstrainedCost(mdl, cp.AffineWorkModel(0, 1, 0), w_max)
                Phi = ref.partition_stripe(A, K, cp.DynamicTotalSplitter(f))
                opt = brute_optimum(Cw, n, K, True)
                if np.isinf(opt):
                    assert Phi.spl.tolist() == [1] * K + [n + 1]
                else:
                    check_split(Phi.spl, n, K)
                    assert objective(Cw, Phi.spl, True) == opt


def test_dynamic_chunker_kform(ref):
    """partition_stripe(A, K, ::AbstractDynamicChunker) (DynamicSplitter.jl:52-87, constrained :249-314): the K-part
    recurrence with the part index as the inner loop -- optimum, and split vectors identical to the splitter form
    (same `<=` rule, same candidate sets), which is what lets the device serve both with one DP."""
    rng = np.random.default_rng(15)
    for trial in range(60):
        A = sprand(rng, int(rng.integers(1, 9)), int(rng.integers(1, 13)), float(rng.choice([0.1, 0.3, 0.5])))
        mdl = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(2, 0, 0, 1)][trial % 3]
        C = cost_matrix(mdl, A)
        for K in [1, 2, 3, 4, 8]:
            for total, S, Ch in [(False, cp.DynamicBottleneckSplitter, cp.DynamicBottleneckChunker), (True, cp.DynamicTotalSplitter, cp.DynamicTotalChunker)]:
                Phi = ref.partition_stripe(A, K, Ch(mdl))
                check_split(Phi.spl, A.n, K)
                assert objective(C, Phi.spl, total) == brute_optimum(C, A.n, K, total)
                assert Phi.spl.tolist() == ref.partition_stripe(A, K, S(mdl)).spl.tolist() == rightmost_dp(C, A.n, K, total)
                for w_max in [2, 4]:
                    f = cp.ConstrainedCost(mdl, cp.VertexCount(), w_max)
                    assert ref.partition_stripe(A, K, Ch(f)).spl.tolist() == ref.partition_stripe(A, K, S(f)).spl.tolist()


def convex_splitter_rule(C, n, K):
    """App. B: each layer keeps the empty last part (ptr = j') only if it is strictly cheaper than the SMALLEST
    minimiser in [1, j' - 1]."""
    prev = [None] + [C[1, jp] for jp in range(1, n + 2)]
    ptrs = [None, [None] + [1] * (n + 1)]
    for k in range(2, K + 1):
        cur, pt = [None] * (n + 2), [None] * (n + 2)
        for jp in range(1, n + 2):
            best, arg = prev[jp] + C[jp, jp], jp
            vals = [prev[j] + C[j, jp] for j in range(1, jp)]
            if vals and min(vals) <= best:
                best, arg = min(vals), 1 + vals.index(min(vals))
            cur[jp], pt[jp] = best, arg
        prev = cur
        ptrs.append(pt)
    spl = [0] * (K + 1)
    spl[K] = n + 1
    for k in range(K, 0, -1):
        spl[k - 1] = ptrs[k][spl[k]]
    return spl


def test_quadrangle_total_splitters(ref, fixtures):
    """ConvexTotalSplitter (ConvexTotalChunker.jl:26-55) on costs obeying the quadrangle inequality: optimal total
    (test_Partitioners.jl:171-199) and the tie rule the device implements; ConcaveTotalSplitter on the additive work
    model (the only affine model that is concave): optimal total."""
    rng = np.random.default_rng(16)
    mats = [fixtures["LPnetlib/lpi_itest6"]] + [sprand(rng, int(rng.integers(1, 10)), int(rng.integers(1, 14)), float(rng.choice([0.1, 0.3, 0.5]))) for _ in range(40)]
    for t, A in enumerate(mats):
        mdl = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(2, 0, 0, 1), cp.AffineConnectivityModel(0, 10, 1, 100)][t % 4]
        C = cost_matrix(mdl, A)
        for K in [1, 2, 3, 4, 8]:
            Phi = ref.partition_stripe(A, K, cp.ConvexTotalSplitter(mdl))
            check_split(Phi.spl, A.n, K)
            assert objective(C, Phi.spl, True) == brute_optimum(C, A.n, K, True)
            assert Phi.spl.tolist() == convex_splitter_rule(C, A.n, K)
            if t % 4 == 0:
                Phi = ref.partition_stripe(A, K, cp.ConcaveTotalSplitter(mdl))
                check_split(Phi.spl, A.n, K)
                assert objective(C, Phi.spl, True) == brute_optimum(C, A.n, K, True)


def test_unconstrained_convex_chunker_is_one_chunk(ref):
    """pack_stripe(A, ConvexTotalChunker(f)) without a width constraint on the affine quadrangle-inequality models
    (alpha, beta >= 0): subadditive costs make j = 1 the smallest minimiser of every prefix, so the restated stack
    algorithm (ConvexTotalChunker.jl:9-24,57-112) returns the single chunk -- the closed form the device returns."""
    rng = np.random.default_rng(17)
    for trial in range(150):
        m, n = int(rng.integers(1, 10)), int(rng.integers(1, 14))
        A = sprand(rng, m, n, float(rng.choice([0.0, 0.1, 0.3, 0.5])))
        mdls = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(2, 0, 0, 1),
                cp.AffineConnectivityModel(0.0, 0.0, 0.0, 1.0), cp.AffineWorkModel(0, 0, 0)]
        if m == n:
            mdls.append(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5))
        for mdl in mdls:
            assert ref.pack_stripe(A, cp.ConvexTotalChunker(mdl)).spl.tolist() == [1, n + 1]
            assert ref.pack_stripe(A, cp.DynamicTotalChunker(mdl)).spl.tolist() == [1, n + 1]  # `<` keeps the smallest j too


def test_dynamic_splitter_constrained_pin_weights(ref):
    """DynamicSplitter.jl:206-247 with a weight that counts pins (AffineWorkModel(a, b_v, b_p) as the weight oracle):
    optimum among weight-feasible partitions, or the degenerate partition."""
    rng = np.random.default_rng(18)
    for n in [1, 4, 7, 11]:
        A = sprand(rng, 6, n, 0.4)
        mdl = cp.AffineConnectivityModel(0, 1, 0, 2)
        C = cost_matrix(mdl, A)
        for (a, bv, bp), w_max in [((0, 1, 1), 6), ((0, 0, 1), 4), ((1, 1, 2), 12)]:
            Cw = C.copy()
            for j in range(1, n + 2):
                for jp in range(j, n + 2):
                    if a + bv * (jp - j) + bp * int(A.colptr[jp - 1] - A.colptr[j - 1]) > w_max:
                        Cw[j, jp] = np.inf
            for K in [1, 2, 3, 5]:
                for total, S in [(True, cp.DynamicTotalSplitter), (False, cp.DynamicBottleneckSplitter)]:
                    Phi = ref.partition_stripe(A, K, S(cp.ConstrainedCost(mdl, cp.AffineWorkModel(a, bv, bp), w_max)))
                    opt = brute_optimum(Cw, n, K, total)
                    if np.isinf(opt):
                        assert Phi.spl.tolist() == [1] * K + [n + 1]
                    else:
                        check_split(Phi.spl, n, K)
                        assert objective(Cw, Phi.spl, total) == opt


def greedy_probe(C, n, K, c):
    """every part as long as feasible at threshold c; None if infeasible"""
    spl = [1]
    j = 1
    for k in range(1, K):
        jp = j
        while jp + 1 <= n + 1 and C[j, jp + 1] <= c:
            jp += 1
        if C[j, jp] > c:
            return None
        spl.append(jp)
        j = jp
    if C[j, n + 1] > c:
        return None
    return spl + [n + 1]


def bisect_reference(C, n, K, eps, lo, hi):
    """Independent statement of App. A "Bisection loop" + App. B row 4 (no windows, no streaming)."""
    best = [1] + [n + 1] * K
    while lo * (1 + eps) < hi:
        c = (lo + hi) / 2
        s = greedy_probe(C, n, K, c)
        if s is not None:
            hi, best = c, s
        else:
            lo = c
    return best


@pytest.mark.parametrize("eps", [0.1, 0.01])
def test_bisect_and_lazy(ref, fixtures, eps):
    """test_Partitioners.jl:95-113 eps-optimality; SURVEY E3/E4: BisectCost == LazyBisect == greedy definition."""
    rng = np.random.default_rng(15)
    mats = [fixtures["LPnetlib/lpi_itest6"]] + [sprand(rng, m, n, 0.2) for m in [1, 3, 8] for n in [1, 2, 4, 8, 16]] + [sprand(rng, 14, 14, 0.3)]
    for A in mats:
        models = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0, 10, 1, 100),
                  cp.AffineConnectivityModel(0.0, 3.0, 1.0, 3.5)]
        if A.m == A.n:
            models += [cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5), cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 2)]
        for mdl in models:
            C = cost_matrix(mdl, A)
            for K in [1, 2, 3, 4, 8]:
                opt = brute_optimum(C, A.n, K, False)
                lo, hi = ref.bound_stripe(A, K, mdl)
                lo = max(lo, float(mdl.coef[0]))
                exp = bisect_reference(C, A.n, K, eps, lo, hi)
                got = {}
                for name, mtd in [("bisect", cp.BisectCostBottleneckSplitter(mdl, eps)), ("lazy", cp.LazyBisectCostBottleneckSplitter(mdl, eps))]:
                    Phi = ref.partition_stripe(A, K, mtd)
                    check_split(Phi.spl, A.n, K)
                    assert objective(C, Phi.spl, False) <= opt * (1 + eps) + 1e-9
                    got[name] = Phi.spl.tolist()
                assert got["lazy"] == exp, (mdl, K)
                if mdl.kind != cp.MODEL_WORK or True:
                    # BisectCost has no c_lo = max(c_lo, alpha) step; identical whenever alpha <= c_lo
                    assert got["bisect"] == got["lazy"], (mdl, K, A)


def test_bisect_index_is_exact(ref, fixtures):
    """BisectIndexBottleneckSplitter (BisectIndexBottleneckSplitter.jl:5-81): the reference tests it with tolerance 0
    against the brute-force optimum (test_Partitioners.jl:101,109-111)."""
    rng = np.random.default_rng(19)
    mats = [fixtures["LPnetlib/lpi_itest6"]] + [sprand(rng, int(rng.integers(1, 10)), int(rng.integers(1, 14)), float(rng.choice([0.1, 0.3, 0.5]))) for _ in range(60)]
    for A in mats:
        mdls = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(2, 0, 0, 1), cp.AffineConnectivityModel(0.0, 0.5, 1.0, 3.0)]
        if A.m == A.n:
            mdls.append(cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5))
        for mdl in mdls:
            C = cost_matrix(mdl, A)
            for K in [1, 2, 3, 4, 8]:
                Phi = ref.partition_stripe(A, K, cp.BisectIndexBottleneckSplitter(mdl))
                check_split(Phi.spl, A.n, K)
                assert objective(C, Phi.spl, False) == brute_optimum(C, A.n, K, False)


def primary_cost(mdl, A, Pi, j, jp, k):
    """PrimaryConnectivityCosts.jl:19,66-73 from the set definition: nets of columns [j, j') owned by row part k are local."""
    c = mdl.coef
    rows = set()
    for col in range(j, jp):
        rows |= set(col_rows(A, col).tolist())
    l = sum(1 for r in rows if Pi.spl[k - 1] <= r < Pi.spl[k])
    return c[0] + (jp - j) * c[1] + int(A.colptr[jp - 1] - A.colptr[j - 1]) * c[2] + l * c[3] + (len(rows) - l) * c[4]


def test_primary_connectivity_oracle_and_solvers(ref, fixtures):
    """AffinePrimaryConnectivityModel with Pi = partition_stripe(A', K, EquiSplitter()) (test_Partitioners.jl:86-113;
    test_Costs.jl:51-79): the oracle equals the set definition for every (j, j', k) and every hint (the partwise
    "stacked" matrix of PartwiseCounts.jl restated), bound sandwich, Dynamic / BisectIndex optimal, Bisect within eps."""
    rng = np.random.default_rng(20)
    for trial in range(40):
        m, n = int(rng.integers(1, 9)), int(rng.integers(1, 10))
        A = sprand(rng, m, n, float(rng.choice([0.1, 0.3, 0.6])))
        for K in [1, 2, 3, 4]:
            Pi = ref.partition_stripe(ref.adjointpattern(A), K, cp.EquiSplitter())
            mdl = [cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6), cp.AffinePrimaryConnectivityModel(1, 1, 1, 1, 1),
                   cp.AffinePrimaryConnectivityModel(0.0, 0.5, 1.0, 3.0, 6.5)][trial % 3]
            Ck = {(k, j, jp): primary_cost(mdl, A, Pi, j, jp, k) for k in range(1, K + 1) for j in range(1, n + 2) for jp in range(j, n + 2)}
            keys = list(Ck)
            for hint in HINTS:
                got = ref.oracle_query(mdl, A, [t[1] for t in keys], [t[2] for t in keys], [t[0] for t in keys], hint=hint, Pi=Pi)
                assert got.tolist() == [float(Ck[t]) for t in keys]

            def dp(total):
                prev = {jp: Ck[(1, 1, jp)] for jp in range(1, n + 2)}
                for k in range(2, K + 1):
                    prev = {jp: min((prev[j] + Ck[(k, j, jp)]) if total else max(prev[j], Ck[(k, j, jp)]) for j in range(1, jp + 1)) for jp in range(1, n + 2)}
                return prev[n + 1]

            def value(spl, total):
                v = [Ck[(k + 1, int(spl[k]), int(spl[k + 1]))] for k in range(K)]
                return sum(v) if total else max(v)

            for mtd, total, eps in [(cp.DynamicBottleneckSplitter(mdl), False, 0), (cp.DynamicTotalSplitter(mdl), True, 0),
                                    (cp.BisectIndexBottleneckSplitter(mdl), False, 0), (cp.BisectCostBottleneckSplitter(mdl, 0.1), False, 0.1),
                                    (cp.LazyBisectCostBottleneckSplitter(mdl, 0.01), False, 0.01)]:
                Phi = ref.partition_stripe(A, K, mtd, Pi)
                check_split(Phi.spl, n, K)
                opt = dp(total)
                assert opt <= value(Phi.spl, total) <= opt * (1 + eps), type(mtd).__name__
                assert ref.bottleneck_value(A, Phi, mdl, Pi) == value(Phi.spl, False)


def secondary_cost(mdl, M, Pi, i, ip, k):
    """SecondaryConnectivityCosts.jl:19,83-90 from the set definition: rows, pins and touched columns of row part k are
    fixed; the touched columns inside [i, i') are local."""
    c = mdl.coef
    cols, pins = set(), 0
    for j in range(1, M.n + 1):
        hit = [r for r in col_rows(M, j) if Pi.spl[k - 1] <= r < Pi.spl[k]]
        pins += len(hit)
        if hit:
            cols.add(j)
    l = sum(1 for j in cols if i <= j < ip)
    return c[0] + int(Pi.spl[k] - Pi.spl[k - 1]) * c[1] + pins * c[2] + l * c[3] + (len(cols) - l) * c[4]


def test_secondary_connectivity_oracle_and_flip_solvers(ref):
    """AffineSecondaryConnectivityModel + the Flip family (test_Partitioners.jl:115-148, test_Costs.jl:51-79): oracle equals
    the set definition, bounds bracket the optimum, DynamicBottleneck / FlipBisectIndex optimal, FlipBisectCost and
    LazyFlipBisectCost within eps."""
    rng = np.random.default_rng(22)
    for trial in range(40):
        m, n = int(rng.integers(1, 9)), int(rng.integers(1, 10))
        A = sprand(rng, m, n, float(rng.choice([0.1, 0.3, 0.6])))
        for K in [1, 2, 3, 4]:
            Pi = ref.partition_stripe(ref.adjointpattern(A), K, cp.EquiSplitter())
            mdl = [cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6), cp.AffineSecondaryConnectivityModel(1, 1, 1, 1, 1),
                   cp.AffineSecondaryConnectivityModel(0.0, 0.5, 1.0, 3.0, 6.5)][trial % 3]
            Ck = {(k, i, ip): secondary_cost(mdl, A, Pi, i, ip, k) for k in range(1, K + 1) for i in range(1, n + 2) for ip in range(i, n + 2)}
            keys = list(Ck)
            got = ref.oracle_query(mdl, A, [t[1] for t in keys], [t[2] for t in keys], [t[0] for t in keys], Pi=Pi)
            assert got.tolist() == [float(Ck[t]) for t in keys]
            prev = {jp: Ck[(1, 1, jp)] for jp in range(1, n + 2)}
            for k in range(2, K + 1):
                prev = {jp: min(max(prev[j], Ck[(k, j, jp)]) for j in range(1, jp + 1)) for jp in range(1, n + 2)}
            opt = prev[n + 1]
            for mtd, eps in [(cp.DynamicBottleneckSplitter(mdl), 0), (cp.FlipBisectIndexBottleneckSplitter(mdl), 0),
                             (cp.FlipBisectCostBottleneckSplitter(mdl, 0.01), 0.01), (cp.LazyFlipBisectCostBottleneckSplitter(mdl, 0.01), 0.01),
                             (cp.FlipBisectCostBottleneckSplitter(mdl, 0.1), 0.1), (cp.LazyFlipBisectCostBottleneckSplitter(mdl, 0.1), 0.1)]:
                Phi = ref.partition_stripe(A, K, mtd, Pi)
                check_split(Phi.spl, n, K)
                v = max(Ck[(k + 1, int(Phi.spl[k]), int(Phi.spl[k + 1]))] for k in range(K))
                assert opt <= v <= opt * (1 + eps), type(mtd).__name__


def edgecut_part_cost(mdl, M, Pi, j, jp, k):
    """PrimaryEdgeCutCosts.jl:18,50-56 / SecondaryEdgeCutCosts.jl:18,78-85 from the set definition: a pin (r, c) is a
    self pin of part k when row part k of Pi owns r and c lies in [j, j')."""
    c = mdl.coef
    own = lambda r: Pi.spl[k - 1] <= r < Pi.spl[k]
    self_pins = sum(1 for q in range(j, jp) for r in col_rows(M, q) if own(r))
    if mdl.kind == cp.types.MODEL_PRIMEDGE:
        pins = sum(len(col_rows(M, q)) for q in range(j, jp))
        return c[0] + (jp - j) * c[1] + self_pins * c[2] + (pins - self_pins) * c[3]
    pins = sum(1 for q in range(1, M.n + 1) for r in col_rows(M, q) if own(r))
    return c[0] + int(Pi.spl[k] - Pi.spl[k - 1]) * c[1] + self_pins * c[2] + (pins - self_pins) * c[3]


def test_edgecut_part_oracles_and_solvers(ref):
    """AffinePrimaryEdgeCutModel / AffineSecondaryEdgeCutModel with a row partition (PrimaryEdgeCutCosts.jl:5-66,
    SecondaryEdgeCutCosts.jl:5-97): the oracle equals the set definition for every (j, j', k); the primary cost grows with
    the part (Dynamic, BisectIndex, BisectCost, LazyBisectCost), the secondary one shrinks when beta_self <= beta_cut
    (Dynamic, the Flip family); exact solvers optimal, bisections within eps."""
    rng = np.random.default_rng(23)
    for trial in range(40):
        m, n = int(rng.integers(1, 9)), int(rng.integers(1, 10))
        A = sprand(rng, m, n, float(rng.choice([0.1, 0.3, 0.6])))
        for K in [1, 2, 3, 4]:
            Pi = ref.partition_stripe(ref.adjointpattern(A), K, cp.EquiSplitter())
            co = [(0, 2, 1, 5), (1, 1, 1, 1), (0.0, 0.5, 1.0, 3.5)][trial % 3]
            for mdl in (cp.AffinePrimaryEdgeCutModel(*co), cp.AffineSecondaryEdgeCutModel(*co)):
                prim = mdl.kind == cp.types.MODEL_PRIMEDGE
                Ck = {(k, j, jp): edgecut_part_cost(mdl, A, Pi, j, jp, k) for k in range(1, K + 1) for j in range(1, n + 2) for jp in range(j, n + 2)}
                keys = list(Ck)
                got = ref.oracle_query(mdl, A, [t[1] for t in keys], [t[2] for t in keys], [t[0] for t in keys], Pi=Pi)
                assert got.tolist() == [float(Ck[t]) for t in keys]
                prev = {jp: Ck[(1, 1, jp)] for jp in range(1, n + 2)}
                for k in range(2, K + 1):
                    prev = {jp: min(max(prev[j], Ck[(k, j, jp)]) for j in range(1, jp + 1)) for jp in range(1, n + 2)}
                opt = prev[n + 1]
                if prim:
                    mtds = [(cp.DynamicBottleneckSplitter(mdl), 0), (cp.BisectIndexBottleneckSplitter(mdl), 0),
                            (cp.BisectCostBottleneckSplitter(mdl, 0.1), 0.1), (cp.LazyBisectCostBottleneckSplitter(mdl, 0.01), 0.01)]
                else:
                    mtds = [(cp.DynamicBottleneckSplitter(mdl), 0), (cp.FlipBisectIndexBottleneckSplitter(mdl), 0),
                            (cp.FlipBisectCostBottleneckSplitter(mdl, 0.01), 0.01), (cp.LazyFlipBisectCostBottleneckSplitter(mdl, 0.1), 0.1)]
                for mtd, eps in mtds:
                    Phi = ref.partition_stripe(A, K, mtd, Pi)
                    check_split(Phi.spl, n, K)
                    v = max(Ck[(k + 1, int(Phi.spl[k]), int(Phi.spl[k + 1]))] for k in range(K))
                    assert opt <= v <= opt * (1 + eps), type(mtd).__name__


def part_cost_by_definition(mdl, A, cols, row_asg, k):
    """compute_objective's per-part numbers from the set definition (WorkCosts.jl:63-77, Costs.jl:52-66 on A[:, prm],
    PrimaryConnectivityCosts.jl:127-159, EnvelopeCosts.jl:100-125): ``cols`` = the columns of part k in domain order."""
    c = mdl.coef
    rows = [r for j in cols for r in col_rows(A, j).tolist()]
    nv, pins, nets = len(cols), len(rows), len(set(rows))
    kind = mdl.kind
    if kind == cp.types.MODEL_WORK:
        return c[0] + nv * c[1] + pins * c[2]
    if kind == cp.types.MODEL_CONNECTIVITY:
        return c[0] + nv * c[1] + pins * c[2] + nets * c[3]
    if kind == cp.types.MODEL_PRIMCONN:
        l = sum(1 for r in set(rows) if row_asg[r - 1] == k)
        return c[0] + nv * c[1] + pins * c[2] + l * c[3] + (nets - l) * c[4]
    if kind == cp.types.MODEL_PRIMEDGE:
        l = sum(1 for r in rows if row_asg[r - 1] == k)
        return c[0] + nv * c[1] + l * c[2] + (pins - l) * c[3]
    if kind == cp.types.MODEL_ENVELOPE:
        lo, hi = A.m + 1, 0
        for j in cols:
            r = col_rows(A, j)
            if len(r):
                lo, hi = min(lo, int(r[0])), max(hi, int(r[-1]))
        return c[0] + nv * c[1] + pins * c[2] + max(hi - lo, 0) * c[3]
    raise AssertionError(kind)


OBJECTIVE_MODELS = [cp.AffineWorkModel(1, 2, 3), cp.AffineConnectivityModel(0, 10, 1, 100), cp.AffineConnectivityModel(0.5, 1.0, 0.25, 3.0),
                    cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6), cp.AffinePrimaryEdgeCutModel(0, 2, 1, 5), cp.AffineEnvelopeModel(0, 1, 1, 2)]


def test_objective_of_noncontiguous_partitions(ref):
    """bottleneck_value / total_value for Map- and DomainPartitions of the columns and MapPartitions of the rows
    (Costs.jl:26-66, WorkCosts.jl:53-81, PrimaryConnectivityCosts.jl:88-163, EnvelopeCosts.jl:75-129) equal the set definition."""
    rng = np.random.default_rng(24)
    for trial in range(60):
        m, n = int(rng.integers(1, 10)), int(rng.integers(1, 12))
        A = sprand(rng, m, n, float(rng.choice([0.1, 0.3, 0.6])))
        K = int(rng.integers(1, 5))
        Phi = cp.MapPartition(K, rng.integers(1, K + 1, n))
        Pi = cp.MapPartition(K, rng.integers(1, K + 1, m))
        dom = cp.convert(cp.DomainPartition, Phi)
        for mdl in OBJECTIVE_MODELS:
            needs_pi = mdl.kind in (cp.types.MODEL_PRIMCONN, cp.types.MODEL_PRIMEDGE)
            costs = [part_cost_by_definition(mdl, A, dom.prm[dom.spl[k] - 1 : dom.spl[k + 1] - 1].tolist(), Pi.asg, k + 1) for k in range(K)]
            for P in (Phi, dom):
                assert ref.bottleneck_value(A, P, mdl, Pi if needs_pi else None) == max(costs)
                assert ref.total_value(A, P, mdl, Pi if needs_pi else None) == sum(costs)


def test_constrained_convex_total_splitter_is_optimal(ref):
    """ConvexTotalSplitter{<:ConstrainedCost} (ConvexTotalChunker.jl:167-265) restated with Extended costs and window-
    constrained columns: the reference's own check (test_Partitioners.jl:176-196) -- the total cost equals the constrained
    DynamicTotalSplitter's, and both are feasible or both degenerate."""
    rng = np.random.default_rng(25)
    for trial in range(300):
        m, n = int(rng.integers(1, 12)), int(rng.integers(1, 16))
        A = sprand(rng, m, n, float(rng.choice([0.1, 0.3, 0.6])))
        K = int(rng.integers(1, 7))
        f = [cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineWorkModel(0, 0, 0), cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0)][trial % 4]
        w, w_max = [(cp.AffineWorkModel(0, 1, 0), 2), (cp.AffineWorkModel(0, 1, 0), 4), (cp.VertexCount(), 8), (cp.AffineWorkModel(0, 1, 1), 12), (cp.AffineWorkModel(2, 1, 2), 30)][trial % 5]
        spec = cp.ConstrainedCost(f, w, w_max)
        r = ref.partition_stripe(A, K, cp.ConvexTotalSplitter(spec))
        d = ref.partition_stripe(A, K, cp.DynamicTotalSplitter(spec))
        check_split(r.spl, n, K)
        assert ref.total_value(A, r, f) == ref.total_value(A, d, f), (A, K, r.spl, d.spl)
        pos = A.colptr
        wgt = lambda P: [w.coef[0] + (P.spl[k + 1] - P.spl[k]) * w.coef[1] + (pos[P.spl[k + 1] - 1] - pos[P.spl[k] - 1]) * w.coef[2] if not isinstance(w, cp.VertexCount)
                         else P.spl[k + 1] - P.spl[k] for k in range(K)]
        assert (max(wgt(r)) <= w_max) == (max(wgt(d)) <= w_max)
        if trial % 4 == 2:  # the additive work model is also (weakly) concave: ConcaveTotalSplitter{<:ConstrainedCost} (ConcaveTotalChunker.jl:143-181)
            c = ref.partition_stripe(A, K, cp.ConcaveTotalSplitter(spec))
            check_split(c.spl, n, K)
            assert (max(wgt(c)) <= w_max) == (max(wgt(d)) <= w_max)
            assert ref.total_value(A, c, f) == ref.total_value(A, d, f)


def leftmost_chunk_dp(C, n, w_max):
    cst = np.full(n + 2, np.inf)
    cst[1] = 0
    ptr = np.zeros(n + 2, dtype=np.int64)
    for jp in range(2, n + 2):
        lo = 1 if w_max is None else max(1, jp - w_max)
        vals = [cst[j] + C[j, jp] for j in range(lo, jp)]
        v = min(vals)
        cst[jp] = v
        ptr[jp] = lo + vals.index(v)
    spl = [n + 1]
    while spl[-1] != 1:
        spl.append(int(ptr[spl[-1]]))
    return spl[::-1], cst


def test_dynamic_total_chunker(ref, fixtures):
    """test_Partitioners.jl:225-248: width <= w_max, optimal total; App. B: leftmost argmin."""
    rng = np.random.default_rng(16)
    mats = [fixtures["LPnetlib/lpi_itest6"]] + [sprand(rng, m, n, 0.3) for m in [2, 5, 9] for n in [1, 2, 5, 11, 17]]
    mats += [sprand(rng, m, n, p) for m, n, p in [(6, 90, 0.15), (20, 130, 0.05)]]  # the device's wide window templates
    for A in mats:
        Pi = ref.pack_stripe(ref.adjointpattern(A), cp.EquiChunker(2))
        for mdl in [cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0, 0, 0, 1),
                    cp.BlockComponentCostModel(int, 0, 0, (10, cp.identity), (2, lambda x: 2 * x)),
                    cp.BlockComponentCostModel(int, 1, 3, (1, cp.identity), (1, cp.identity)),
                    cp.ColumnBlockComponentCostModel(int, 3, lambda w: 1 + w)]:
            C = cost_matrix(mdl, A, Pi)
            for w_max in [1, 2, 4, 8, 16, 17, 32, 33, 64]:
                Phi = ref.pack_stripe(A, cp.DynamicTotalChunker(cp.ConstrainedCost(mdl, cp.VertexCount(), w_max)), Pi)
                check_split(Phi.spl, A.n)
                assert np.all(np.diff(Phi.spl) <= w_max)
                exp, cst = leftmost_chunk_dp(C, A.n, w_max)
                assert objective(C, Phi.spl, True) == brute_chunk_optimum(C, A.n, w_max)
                assert Phi.spl.tolist() == exp
            if mdl.kind == cp.MODEL_CONNECTIVITY:
                Phi = ref.pack_stripe(A, cp.DynamicTotalChunker(mdl))  # unconstrained == ReferenceTotalChunker
                assert Phi.spl.tolist() == leftmost_chunk_dp(C, A.n, None)[0]


def convex_constrained_rule(C, n, w_max):
    """SURVEY App. B: windows B_t = (1+t w, 1+(t+1) w]; in-window leftmost unless prev strictly better (then rightmost)."""
    cst = np.full(n + 2, np.inf)
    cst[1] = 0
    ptr = np.zeros(n + 2, dtype=np.int64)
    for jp in range(2, n + 2):
        t = (jp - 2) // w_max
        j0 = 1 + t * w_max
        in_ = list(range(max(jp - w_max, j0), jp))
        prev = list(range(max(jp - w_max, 1), j0))
        vin = [cst[j] + C[j, jp] for j in in_]
        vpr = [cst[j] + C[j, jp] for j in prev]
        if not vpr or min(vin) <= min(vpr):
            v = min(vin)
            ptr[jp] = in_[vin.index(v)]
        else:
            v = min(vpr)
            ptr[jp] = max(j for j, x in zip(prev, vpr) if x == v)
        cst[jp] = v
    spl = [n + 1]
    while spl[-1] != 1:
        spl.append(int(ptr[spl[-1]]))
    return spl[::-1]


def test_convex_chunkers(ref, fixtures):
    """test_Partitioners.jl:250-275 (optimal value); SURVEY E5/E6 tie rules for convex costs."""
    rng = np.random.default_rng(17)
    mats = [fixtures["LPnetlib/lpi_itest6"]] + [sprand(rng, m, n, 0.3) for m in [2, 5, 9] for n in [1, 2, 5, 11, 17, 30]]
    mats += [sprand(rng, m, n, p) for m, n, p in [(6, 90, 0.15), (20, 130, 0.05)]]  # the device's wide window templates
    for A in mats:
        for mdl in [cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(1, 0, 0, 1),
                    cp.AffineConnectivityModel(-0.5, 0.0, 0.0, 1.0)]:
            C = cost_matrix(mdl, A)
            Phi = ref.pack_stripe(A, cp.ConvexTotalChunker(mdl))
            check_split(Phi.spl, A.n)
            assert objective(C, Phi.spl, True) == brute_chunk_optimum(C, A.n, None)
            assert Phi.spl.tolist() == leftmost_chunk_dp(C, A.n, None)[0]
            for w_max in [1, 2, 3, 4, 8, 16, 17, 32, 33, 64]:
                Phi = ref.pack_stripe(A, cp.ConvexTotalChunker(cp.ConstrainedCost(mdl, cp.VertexCount(), w_max)))
                check_split(Phi.spl, A.n)
                assert np.all(np.diff(Phi.spl) <= w_max)
                assert objective(C, Phi.spl, True) == brute_chunk_optimum(C, A.n, w_max)
                assert Phi.spl.tolist() == convex_constrained_rule(C, A.n, w_max), (mdl, w_max, A.n)


def test_concave_chunker(ref):
    """test_Partitioners.jl:277-299: concave chunker reaches the optimum on a concave cost (work model
    with alpha > 0 is both convex and concave: modular)."""
    rng = np.random.default_rng(18)
    for n in [1, 2, 5, 11, 17]:
        A = sprand(rng, 6, n, 0.3)
        for mdl in [cp.AffineWorkModel(3, 1, 2), cp.AffineWorkModel(0, 0, 0)]:
            C = cost_matrix(mdl, A)
            Phi = ref.pack_stripe(A, cp.ConcaveTotalChunker(mdl))
            check_split(Phi.spl, A.n)
            assert objective(C, Phi.spl, True) == brute_chunk_optimum(C, A.n, None)


def overlap_definition(A, rho, w_max):
    """SURVEY App. C / E10: greedy from set definitions, `c` frozen at deg(column 1)."""
    n = A.n
    c0 = len(col_rows(A, 1))
    spl, nets = [1], []
    j = 1
    for jp in range(2, n + 1):
        cc = len(set(col_rows(A, j).tolist()) & set(col_rows(A, jp).tolist()))
        if jp - j == w_max or cc < rho * min(c0, len(col_rows(A, jp))):
            nets.append(ref_netcount(A, j, jp))
            spl.append(jp)
            j = jp
    nets.append(ref_netcount(A, j, n + 1))
    spl.append(n + 1)
    return spl, nets


def strict_definition(A, w_max):
    n = A.n
    spl = [1]
    j = 1
    for jp in range(2, n + 1):
        same = col_rows(A, j).tolist() == col_rows(A, jp).tolist()
        if not (same and jp - j != w_max):
            spl.append(jp)
            j = jp
    return spl + [n + 1]


def test_overlap_and_strict(ref, fixtures):
    rng = np.random.default_rng(19)
    mats = [fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"]] + [sprand(rng, m, n, p) for m in [3, 6] for n in [1, 2, 9, 25] for p in [0.3, 0.8]]
    mats += [sprand(rng, m, n, p) for m, n, p in [(2, 100, 0.9), (3, 120, 0.8), (6, 70, 0.5)]]  # runs of identical / overlapping columns
    for A in mats:
        for w_max in [1, 2, 4, 8, 16, 17, 32, 33, 64]:
            for rho in [0.9, 0.8, 0.7, 0.3]:
                box = [None]
                Phi = ref.pack_stripe(A, cp.OverlapChunker(rho, w_max), n_nets=box)
                exp_spl, exp_nets = overlap_definition(A, rho, w_max)
                assert Phi.spl.tolist() == exp_spl
                assert box[0].tolist() == exp_nets
                assert np.all(np.diff(Phi.spl) <= w_max)
            Phi = ref.pack_stripe(A, cp.StrictChunker(w_max))
            assert Phi.spl.tolist() == strict_definition(A, w_max)


def test_equi(ref):
    for n in [1, 5, 17]:
        A = cp.SparseMatrixCSC(1, n, np.ones(n + 1, dtype=np.int64), np.zeros(0, dtype=np.int64))
        for K in [1, 2, 3, 8]:
            spl = ref.partition_stripe(A, K, cp.EquiSplitter()).spl
            assert spl.tolist() == [(k - 1) * (n // K) + min(n % K, k - 1) + 1 for k in range(1, K + 2)]
        for w in [1, 2, 4]:
            assert ref.pack_stripe(A, cp.EquiChunker(w)).spl.tolist() == list(range(1, n + 1, w)) + [n + 1]


def test_plaid(ref, fixtures):
    """AlternatingPartitioner.jl:18-32 on the symmetric fixture (config 5 in miniature)."""
    A = fixtures["HB/can_292"]
    s = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 90)
    mtd = cp.LazyBisectCostBottleneckSplitter(s, 0.1)
    Pi, Phi = ref.partition_plaid(A, 8, cp.AlternatingPartitioner(mtd, mtd))
    check_split(Pi.spl, A.m, 8)
    check_split(Phi.spl, A.n, 8)
    assert Pi == Phi  # symmetric pattern: both stripe solves see the same matrix


def test_envelope_bound_forms(ref, fixtures):
    """bound_stripe(A, K, ocl) vs bound_stripe(A, K, mdl) for the envelope model (EnvelopeCosts.jl:30-42, 44-54): equal for Int64
    coefficients, equal up to roundings for Float64 ones; only the oracle form accepts an empty pattern."""
    import chainb200 as cp

    A = fixtures["LPnetlib/lp_blend"]
    fi = cp.AffineEnvelopeModel(2, 3, 1, 5)
    ff = cp.AffineEnvelopeModel(0.1, 0.7, 0.3, 1.9)
    for K in (1, 4, 9):
        assert ref.bound_stripe(A, K, fi, via_oracle=True) == ref.bound_stripe(A, K, fi, via_oracle=False)
        a, b = ref.bound_stripe(A, K, ff, via_oracle=True), ref.bound_stripe(A, K, ff, via_oracle=False)
        assert abs(a[0] - b[0]) <= 1e-9 * abs(b[0]) + 1.0 and abs(a[1] - b[1]) <= 1e-9 * abs(b[1])
    E = cp.SparseMatrixCSC(5, 4, [1, 1, 1, 1, 1], np.zeros(0, dtype=np.int64))
    assert ref.bound_stripe(E, 2, fi, via_oracle=True) == (2 + (3 * 4) // 2, 2 + 3 * 4)
    with pytest.raises(RuntimeError):
        ref.bound_stripe(E, 2, fi, via_oracle=False)
