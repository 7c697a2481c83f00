"""Multi-GPU partition_plaid pieces of csrc/sharded.cu on one GPU (-m gpu): the A + I link blocks of the monotonized
symmetric model and the sharded adjointpattern with the ranks played one after the other, the real entry points with a
world of one, and partition_plaid_sharded -- every result equal to the single-GPU one and the CPU oracle's."""
import numpy as np
import pytest

import chainb200 as cp
from chainb200 import synth
from helpers import sprand

pytestmark = pytest.mark.gpu

AFF = cp.AffineConnectivityModel(0, 10, 1, 100)


def sym_cases():
    z = np.zeros(0, dtype=np.int64)
    return [(synth.random_geometric(5000), 16, 0.1, 90), (synth.random_geometric(20000), 32, 0.1, 4), (synth.laplacian5(40), 7, 0.001, 2),
            (synth.banded(3000, 20), 5, 0.05, 3), (synth.erdos_renyi(3000, 6), 9, 0.01, 4), (synth.rmat(12, 16 << 12), 64, 0.01, 8),
            (cp.SparseMatrixCSC(3, 3, np.ones(4, dtype=np.int64), z), 2, 0.1, 1),
            (cp.SparseMatrixCSC(6, 6, np.array([1, 1, 1, 1, 3, 3, 3]), np.array([1, 4])), 3, 0.1, 0),  # fewer nonzeros than ranks
            (cp.SparseMatrixCSC(6, 6, np.array([0, 0, 2, 4, 6, 6, 8]) + 1, np.array([0, 3, 0, 4, 0, 5, 2, 5]) + 1), 3, 0.1, 1)]


def test_sharded_sym_solve_emulated_and_single_rank(ref):
    """partition_stripe_sharded(_emulated) with the monotonized symmetric model: the links of A + I by blocks (virtual
    diagonals placed by the A + I block rule, both carry forms) equal the single-GPU and CPU-oracle split vectors."""
    for A, K, eps, dp in sym_cases():
        s = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, dp)
        for mtd in (cp.LazyBisectCostBottleneckSplitter(s, eps), cp.BisectCostBottleneckSplitter(cp.AffineMonotonizedSymmetricConnectivityModel(0.0, 3.0, 1.0, 7.0, dp), eps)):
            exp = ref.partition_stripe(A, K, mtd).spl
            assert np.array_equal(cp.partition_stripe(A, K, mtd).spl, exp), (A.n, K)
            for world in (1, 2, 3, 4, 8):
                got = cp.partition_stripe_sharded_emulated(A, K, mtd, world).spl
                assert np.array_equal(got, exp), (A.n, K, world)
            assert np.array_equal(cp.partition_stripe_sharded(A, K, mtd).spl, exp), (A.n, K, "world of one")


def test_sharded_sym_chain_carry_form(ref, monkeypatch):
    """The chain carry form (CPB_SHARD_CHAIN) with more than two emulated ranks gives the same A + I links."""
    monkeypatch.setenv("CPB_SHARD_CHAIN", "1")
    A = synth.random_geometric(8000)
    mtd = cp.LazyBisectCostBottleneckSplitter(cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 6), 0.1)
    exp = ref.partition_stripe(A, 16, mtd).spl
    for world in (3, 8):
        assert np.array_equal(cp.partition_stripe_sharded_emulated(A, 16, mtd, world).spl, exp), world


def test_sharded_sym_refuses_non_square():
    mtd = cp.LazyBisectCostBottleneckSplitter(cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 1), 0.1)
    A = cp.SparseMatrixCSC(4, 3, [1, 1, 1, 1], np.zeros(0, dtype=np.int64))
    with pytest.raises(cp.CpbError):
        cp.partition_stripe_sharded_emulated(A, 2, mtd, 2)
    with pytest.raises(cp.CpbError):
        cp.partition_stripe_sharded(A, 2, mtd)


def transpose_cases(fixtures):
    rng = np.random.default_rng(5)
    z = np.zeros(0, dtype=np.int64)
    return list(fixtures.values()) + [synth.erdos_renyi(20000, 10), synth.rmat(12, 16 << 12), sprand(rng, 300, 170, 0.05), sprand(rng, 90, 410, 0.03),
                                      cp.SparseMatrixCSC(4, 3, np.ones(4, dtype=np.int64), z)]


def test_sharded_adjointpattern_emulated_and_single_rank(ref, fixtures):
    """cpb_adjointpattern_sharded_emulated equals adjointpattern for 1..8 ranks (rectangular and empty patterns too); the
    real entry point with a world of one returns the transpose as a ShardedMatrix."""
    for A in transpose_cases(fixtures):
        B = cp.adjointpattern(A)
        R = ref.adjointpattern(A)
        assert np.array_equal(B.colptr, R.colptr) and np.array_equal(B.rowval, R.rowval)
        for world in (1, 2, 3, 4, 8):
            E = cp.adjointpattern_sharded_emulated(A, world)
            assert (E.m, E.n, E.nnz) == (A.n, A.m, A.nnz)
            assert np.array_equal(E.colptr, B.colptr) and np.array_equal(E.rowval, B.rowval), (A.m, A.n, world)
        S = cp.ShardedMatrix(A)
        T = S.adjointpattern()
        colptr, rowval, lo, hi = T.to_host_block()
        assert (T.m, T.n, T.nnz) == (A.n, A.m, A.nnz) and (lo, hi) == (0, A.nnz)
        assert np.array_equal(colptr, B.colptr) and np.array_equal(rowval, B.rowval)
        c2, r2, _, _ = S.to_host_block()
        assert np.array_equal(c2, A.colptr) and np.array_equal(r2, A.rowval)
        T.close()
        S.close()


def plaid_cases():
    A = synth.random_geometric(20000)
    sym = cp.LazyBisectCostBottleneckSplitter(cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 90), 0.1)
    net = cp.LazyBisectCostBottleneckSplitter(AFF, 0.01)
    E = synth.erdos_renyi(3000, 6)
    return [(A, 32, cp.AlternatingPartitioner(sym, sym)),  # C5 shape
            (E, 12, cp.AlternatingPartitioner(net, cp.BisectCostBottleneckSplitter(AFF, 0.01), net)),
            (E, 7, cp.SymmetricPartitioner(sym, sym, sym)), (E, 5, cp.DisjointPartitioner(net, sym)), (E, 6, cp.SymmetricPartitioner(net))]


def test_partition_plaid_sharded(ref):
    """partition_plaid_sharded_emulated (1..8 ranks) and partition_plaid_sharded (a world of one) equal partition_plaid on
    the GPU and the CPU oracle's."""
    for A, K, meth in plaid_cases():
        Pg, Fg = cp.partition_plaid(A, K, meth)
        Pr, Fr = ref.partition_plaid(A, K, meth)
        assert np.array_equal(Pg.spl, Pr.spl) and np.array_equal(Fg.spl, Fr.spl)
        for world in (1, 2, 3, 8):
            Pe, Fe = cp.partition_plaid_sharded_emulated(A, K, meth, world)
            assert np.array_equal(Pe.spl, Pr.spl) and np.array_equal(Fe.spl, Fr.spl), (K, world)
        Ps, Fs = cp.partition_plaid_sharded(A, K, meth)
        assert np.array_equal(Ps.spl, Pr.spl) and np.array_equal(Fs.spl, Fr.spl), (K, "world of one")
        S = cp.ShardedMatrix(A)
        Ps, Fs = cp.partition_plaid_sharded(S, K, meth, adj_A=cp.adjointpattern(A))
        S.close()
        assert np.array_equal(Ps.spl, Pr.spl) and np.array_equal(Fs.spl, Fr.spl), (K, "resident, given transpose")


def test_partition_plaid_sharded_refusals():
    A = synth.erdos_renyi(500, 4)
    prim = cp.AffinePrimaryConnectivityModel(0, 10, 1, 0, 100)
    for meth in (cp.AlternatingPartitioner(cp.LazyBisectCostBottleneckSplitter(cp.AffineWorkModel(0, 1, 1), 0.1), cp.LazyBisectCostBottleneckSplitter(AFF, 0.1)),
                 cp.AlternatingPartitioner(cp.DynamicBottleneckSplitter(AFF), cp.LazyBisectCostBottleneckSplitter(AFF, 0.1)),
                 cp.AlternatingPartitioner(cp.LazyBisectCostBottleneckSplitter(AFF, 0.1), cp.BisectCostBottleneckSplitter(prim, 0.1)),
                 cp.LazyBisectCostBottleneckSplitter(AFF, 0.1)):
        with pytest.raises(TypeError):
            cp.partition_plaid_sharded(A, 4, meth)
        with pytest.raises(TypeError):
            cp.partition_plaid_sharded_emulated(A, 4, meth, 2)
    with pytest.raises(cp.CpbError):
        cp.partition_stripe_sharded(A, 4, cp.LazyBisectCostBottleneckSplitter(cp.AffinePrimaryConnectivityModel(0, 10, 1, 0, 100), 0.1))
