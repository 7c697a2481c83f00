"""partition_stripe_batch / cpb_partition_stripe_batch: many BisectIndex and Flip problems in one launch, one cluster each.
Every batch result is compared with the single partition_stripe call and with the CPU oracle; refusals fail the whole call
before anything is written."""
import ctypes

import numpy as np
import pytest

import chainb200 as cp
from chainb200 import synth
from helpers import sprand

SPLIT_BISECT_COST, SPLIT_BISECT_INDEX = 2, 12
SPLIT_FLIP_BISECT_COST, SPLIT_LAZY_FLIP_BISECT_COST, SPLIT_FLIP_BISECT_INDEX = 6, 7, 13


def row_partition(ref, A, K):
    """Pi = partition_stripe(A', K, EquiSplitter()) as in test_Partitioners.jl:95."""
    return ref.partition_stripe(ref.adjointpattern(A), K, cp.EquiSplitter())


def check_batch(ref, problems):
    got = cp.partition_stripe_batch(problems)
    assert len(got) == len(problems)
    for p, g in zip(problems, got):
        A, K, mtd = p[:3]
        Pi = p[3] if len(p) == 4 else None
        single = cp.partition_stripe(A, K, mtd, Pi) if Pi is not None else cp.partition_stripe(A, K, mtd)
        r = ref.partition_stripe(A, K, mtd, Pi) if Pi is not None else ref.partition_stripe(A, K, mtd)
        assert g.K == K
        assert np.array_equal(g.spl, single.spl), (A.n, K, type(mtd).__name__, g.spl, single.spl)
        assert np.array_equal(g.spl, r.spl), (A.n, K, type(mtd).__name__, g.spl, r.spl)
    return got


def raw_batch(ocls, methods, Ks, eps=None, fill=-7):
    """cpb_partition_stripe_batch on prebuilt oracles -> (return code, outputs)."""
    B = len(ocls)
    outs = [np.full(int(K) + 1, fill, dtype=np.int64) for K in Ks]
    f = (ctypes.c_void_p * B)(*[o._h.value for o in ocls])
    m = np.array(methods, dtype=np.int32)
    k = np.array(Ks, dtype=np.int64)
    e = np.array(eps, dtype=np.float64) if eps is not None else None
    spl = (ctypes.c_void_p * B)(*[o.ctypes.data for o in outs])
    rc = cp.load_library().cpb_partition_stripe_batch(B, f, m.ctypes.data, e.ctypes.data if e is not None else None, k.ctypes.data, spl)
    return rc, outs


# ------------------------------------------------------------------------------------------------ no GPU


def test_unsupported_methods_raise_type_error_before_any_device_call():
    A = cp.SparseMatrixCSC(2, 2, [1, 2, 3], [1, 2])
    f = cp.AffineConnectivityModel(0, 1, 1, 1)
    for mtd in (cp.DynamicBottleneckSplitter(f), cp.BisectCostBottleneckSplitter(f, 0.1), cp.LazyBisectCostBottleneckSplitter(f, 0.1),
                cp.EquiSplitter(), cp.ConvexTotalSplitter(f)):
        with pytest.raises(TypeError):
            cp.partition_stripe_batch([(A, 2, cp.BisectIndexBottleneckSplitter(f)), (A, 2, mtd)])
    assert cp.partition_stripe_batch([]) == []


def test_batch_without_device_is_a_cuda_error():
    lib = cp.load_library()
    if lib.cpb_device_count() > 0:
        pytest.skip("a GPU is visible")
    assert lib.cpb_partition_stripe_batch(0, None, None, None, None, None) == 0  # B = 0: nothing to do
    assert lib.cpb_partition_stripe_batch(1, None, None, None, None, None) == -3
    assert "no CPU fallback" in lib.cpb_last_error().decode()
    A = cp.SparseMatrixCSC(2, 2, [1, 2, 3], [1, 2])
    with pytest.raises(cp.CpbError) as e:
        cp.partition_stripe_batch([(A, 2, cp.BisectIndexBottleneckSplitter(cp.AffineWorkModel(0, 1, 1)))])
    assert e.value.code == -3


# ------------------------------------------------------------------------------------------------ GPU


@pytest.mark.gpu
def test_bisect_index_models(ref, fixtures):
    rng = np.random.default_rng(900)
    mats = [fixtures["LPnetlib/lp_blend"], fixtures["Pajek/GD99_c"], sprand(rng, 40, 200, 0.1), synth.laplacian5(20), synth.erdos_renyi(3000, 6)]
    problems = []
    for A in mats:
        fs = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 10, 1, 100), cp.AffineConnectivityModel(0.0, 3.0, 1.0, 3.5),
              cp.AffineEnvelopeModel(0, 1, 1, 2), cp.AffineEnvelopeModel(0.5, 1.0, 0.0, 2.0)]
        if A.m == A.n:
            fs += [cp.AffineMonotonizedSymmetricConnectivityModel(0, 3, 1, 3, 5), cp.AffineMonotonizedSymmetricConnectivityModel(0.0, 3.0, 1.0, 3.5, 5)]
        for f in fs:
            for K in (1, 3, 8, 33):
                problems.append((A, K, cp.BisectIndexBottleneckSplitter(f)))
    check_batch(ref, problems)


@pytest.mark.gpu
def test_bisect_index_primary_models(ref, fixtures):
    rng = np.random.default_rng(901)
    problems = []
    for A in (fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 40, 120, 0.1), synth.erdos_renyi(2000, 5)):
        for K in (1, 2, 3, 8):
            Pi = row_partition(ref, A, K)
            for f in (cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6), cp.AffinePrimaryConnectivityModel(0.0, 0.5, 1.0, 3.0, 6.5),
                      cp.AffinePrimaryEdgeCutModel(0, 2, 1, 5), cp.AffinePrimaryEdgeCutModel(0.0, 0.5, 1.0, 3.5)):
                problems.append((A, K, cp.BisectIndexBottleneckSplitter(f), Pi))
    check_batch(ref, problems)


@pytest.mark.gpu
def test_flip_methods_secondary_models(ref, fixtures):
    rng = np.random.default_rng(902)
    problems = []
    for A in (fixtures["LPnetlib/lpi_itest6"], fixtures["Pajek/GD99_c"], sprand(rng, 6, 10, 0.3), sprand(rng, 40, 120, 0.1), synth.erdos_renyi(2000, 5)):
        for K in (1, 2, 3, 8):
            Pi = row_partition(ref, A, K)
            for f in (cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6), cp.AffineSecondaryConnectivityModel(0.0, 0.5, 1.0, 3.0, 6.5),
                      cp.AffineSecondaryEdgeCutModel(0, 2, 1, 5), cp.AffineSecondaryEdgeCutModel(0.0, 0.5, 1.0, 3.5)):
                for mtd in (cp.FlipBisectIndexBottleneckSplitter(f), cp.FlipBisectCostBottleneckSplitter(f, 0.1), cp.FlipBisectCostBottleneckSplitter(f, 0.001),
                            cp.LazyFlipBisectCostBottleneckSplitter(f, 0.1), cp.LazyFlipBisectCostBottleneckSplitter(f, 0.001)):
                    problems.append((A, K, mtd, Pi))
    check_batch(ref, problems)


@pytest.mark.gpu
def test_mixed_batch_larger_than_the_resident_clusters(ref, fixtures):
    """Different matrices, models, methods and cost types in random order; K = 1, K >= n and K = 4097; more problems than
    the device keeps resident."""
    rng = np.random.default_rng(903)
    cap = cp.partition_stripe_batch_capacity()
    assert cap >= 1
    mats = [fixtures["LPnetlib/lp_blend"], fixtures["Pajek/GD99_c"], sprand(rng, 30, 40, 0.2), sprand(rng, 8, 8, 0.5), synth.laplacian5(12)]
    big = synth.erdos_renyi(6000, 4)
    pis = {}
    problems = [(big, 4097, cp.BisectIndexBottleneckSplitter(cp.AffineConnectivityModel(0, 10, 1, 100))),
                (big, 4097, cp.BisectIndexBottleneckSplitter(cp.AffineWorkModel(0.0, 1.0, 0.5)))]
    while len(problems) < max(300, cap + 20):
        A = mats[rng.integers(len(mats))]
        K = int(rng.choice([1, 2, 5, A.n, A.n + 3]))
        kind = rng.integers(4)
        if kind == 0:
            f = [cp.AffineWorkModel(0, 10, 1), cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0.0, 3.0, 1.0, 3.5)][rng.integers(3)]
            problems.append((A, K, cp.BisectIndexBottleneckSplitter(f)))
            continue
        if (id(A), K) not in pis:
            pis[(id(A), K)] = row_partition(ref, A, K)
        Pi = pis[(id(A), K)]
        if kind == 1:
            problems.append((A, K, cp.BisectIndexBottleneckSplitter(cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6)), Pi))
        else:
            f = cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6) if kind == 2 else cp.AffineSecondaryEdgeCutModel(0.0, 0.5, 1.0, 3.5)
            mtd = [cp.FlipBisectIndexBottleneckSplitter(f), cp.FlipBisectCostBottleneckSplitter(f, 0.01), cp.LazyFlipBisectCostBottleneckSplitter(f, 0.01)][rng.integers(3)]
            problems.append((A, K, mtd, Pi))
    order = rng.permutation(len(problems))
    check_batch(ref, [problems[i] for i in order])


@pytest.mark.gpu
def test_shared_oracle_k_sweep(ref):
    A = synth.erdos_renyi(4000, 6)
    dA = cp.device_matrix(A)
    mtd = cp.BisectIndexBottleneckSplitter(cp.AffineConnectivityModel(0, 10, 1, 100))
    got = cp.partition_stripe_batch([(dA, K, mtd) for K in range(1, 65)])
    for K, g in zip(range(1, 65), got):
        assert np.array_equal(g.spl, cp.partition_stripe(dA, K, mtd).spl), K
        assert np.array_equal(g.spl, ref.partition_stripe(A, K, mtd).spl), K
    dA.close()


@pytest.mark.gpu
def test_refusals_fail_the_whole_call(ref, fixtures):
    A = fixtures["Pajek/GD99_c"]
    Pi = row_partition(ref, A, 4)
    conn = cp.oracle_stripe(cp.AffineConnectivityModel(0, 3, 1, 3), A)
    dec = cp.oracle_stripe(cp.AffineWorkModel(100, -1, 0), A)
    sec = cp.oracle_stripe(cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6), A, Pi)
    try:
        good = ([conn, sec], [SPLIT_BISECT_INDEX, SPLIT_FLIP_BISECT_COST], [4, 4], [0.0, 0.01])
        rc, outs = raw_batch(*good)
        assert rc == 0
        assert np.array_equal(outs[0], cp.partition_stripe(A, 4, cp.BisectIndexBottleneckSplitter(cp.AffineConnectivityModel(0, 3, 1, 3))).spl)
        assert np.array_equal(outs[1], cp.partition_stripe(A, 4, cp.FlipBisectCostBottleneckSplitter(cp.AffineSecondaryConnectivityModel(0, 2, 1, 3, 6), 0.01), Pi).spl)
        for ocls, methods, Ks, code, bad in (
                ([conn, conn, sec], [SPLIT_BISECT_INDEX, SPLIT_BISECT_COST, SPLIT_FLIP_BISECT_INDEX], [4, 4, 4], -2, 1),  # BisectCost is not batched
                ([conn, sec, conn], [SPLIT_BISECT_INDEX, SPLIT_LAZY_FLIP_BISECT_COST, SPLIT_BISECT_INDEX], [4, 5, 4], -1, 1),  # K != pi_K
                ([conn, sec, dec], [SPLIT_BISECT_INDEX, SPLIT_FLIP_BISECT_INDEX, SPLIT_BISECT_INDEX], [4, 4, 4], -2, 2)):  # a shrinking cost
            rc, outs = raw_batch(ocls, methods, Ks, [0.01] * len(Ks))
            assert rc == code, (rc, cp.load_library().cpb_last_error())
            assert f"problem {bad}" in cp.load_library().cpb_last_error().decode()
            for o in outs:
                assert (o == -7).all()
        # eps may be NULL only without a FlipBisectCost problem
        rc, outs = raw_batch([conn, sec], [SPLIT_BISECT_INDEX, SPLIT_FLIP_BISECT_INDEX], [4, 4], None)
        assert rc == 0
        rc, outs = raw_batch([conn, sec], [SPLIT_BISECT_INDEX, SPLIT_FLIP_BISECT_COST], [4, 4], None)
        assert rc == -1 and all((o == -7).all() for o in outs)
        lib = cp.load_library()
        assert lib.cpb_partition_stripe_batch(0, None, None, None, None, None) == 0
        assert lib.cpb_partition_stripe_batch(2, None, None, None, None, None) == -1
        assert lib.cpb_partition_stripe_batch(-1, None, None, None, None, None) == -1
    finally:
        for o in (conn, dec, sec):
            o.close()


@pytest.mark.gpu
def test_launch_count_of_a_batch(ref, fixtures):
    """Once the oracles exist, a batch is at most two launches (one per cost type), whatever B."""
    A = synth.erdos_renyi(3000, 6)
    Pi = row_partition(ref, A, 8)
    ocls = [cp.oracle_stripe(cp.AffineConnectivityModel(0, 10, 1, 100), A), cp.oracle_stripe(cp.AffineWorkModel(0.0, 1.0, 0.5), A),
            cp.oracle_stripe(cp.AffineSecondaryEdgeCutModel(0, 2, 1, 5), A, Pi), cp.oracle_stripe(cp.AffinePrimaryConnectivityModel(0, 2, 1, 3, 6), A, Pi),
            cp.oracle_stripe(cp.AffineEnvelopeModel(0, 1, 1, 2), A)]
    try:
        args = ([ocls[0]] * 20 + ocls[1:], [SPLIT_BISECT_INDEX] * 21 + [SPLIT_FLIP_BISECT_COST, SPLIT_BISECT_INDEX, SPLIT_BISECT_INDEX],
                list(range(1, 21)) + [8, 8, 8, 8], [0.0] * 21 + [0.01, 0.0, 0.0])
        rc, first = raw_batch(*args)  # builds the oracles' indices
        assert rc == 0, cp.load_library().cpb_last_error()
        n0 = cp.launch_count()
        rc, second = raw_batch(*args)
        assert rc == 0
        assert cp.launch_count() - n0 <= 2
        for a, b in zip(first, second):
            assert np.array_equal(a, b)
    finally:
        for o in ocls:
            o.close()
