"""No-GPU checks of the drop-in boundary: the C-ABI library loads, exports every symbol
include/chainb200.h declares, and fails loudly (no CPU fallback) when no device is usable."""
import os
import re

import numpy as np
import pytest

import chainb200 as cp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "chainb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cpb_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = cp.load_library()
    syms = declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"libchainb200.so does not export {s}"
    assert sorted(cp.api.ABI_SYMBOLS) == syms
    assert lib.cpb_version() == 101


def test_model_struct_layout_matches_header():
    # cpb_model: 2 x int32, 8 x double, 4 x int32, 3 pointers
    assert cp.types.CModel.coef.offset == 8
    assert cp.types.CModel.R.offset == 72
    assert cp.types.CModel.alpha_col.offset == 88
    assert ctypes_sizeof(cp.types.CModel) == 112
    assert ctypes_sizeof(cp.types.CConstraint) == 40


def ctypes_sizeof(t):
    import ctypes

    return ctypes.sizeof(t)


def test_no_cpu_fallback_without_device():
    lib = cp.load_library()
    if lib.cpb_device_count() > 0:
        pytest.skip("a GPU is visible")
    A = cp.SparseMatrixCSC(2, 2, [1, 2, 3], [1, 2])
    with pytest.raises(cp.CpbError) as e:
        cp.partition_stripe(A, 2, cp.DynamicBottleneckSplitter(cp.AffineWorkModel(0, 1, 1)))
    assert e.value.code == -3 and "no CPU fallback" in str(e.value)


def test_host_types_mirror_reference():
    f = cp.AffineConnectivityModel(0, 10, 1, 100)
    assert not f.is_float and f.coef == (0, 10, 1, 100)
    g = cp.AffineConnectivityModel(beta_net=1.0)
    assert g.is_float and g.coef == (0.0, 0.0, 0.0, 1.0)
    P = cp.SplitPartition(3, [1, 3, 3, 6])
    M = cp.convert(cp.MapPartition, P)
    assert M.asg.tolist() == [1, 1, 3, 3, 3]
    D = cp.convert(cp.DomainPartition, M)
    assert D.spl.tolist() == [1, 3, 3, 6] and D.prm.tolist() == [1, 2, 3, 4, 5]
    assert cp.convert(cp.MapPartition, D) == M
    c = cp.DynamicTotalChunker(f, 8)  # deprecated two-argument form, ChainPartitioners.jl:221
    assert isinstance(c.f, cp.ConstrainedCost) and c.f.w_max == 8


def test_synthetic_generators_are_deterministic():
    from chainb200 import synth

    A = synth.laplacian5(8)
    assert (A.m, A.n, A.nnz) == (64, 64, 5 * 64 - 4 * 8)
    B = synth.erdos_renyi(1000, 10)
    C = synth.erdos_renyi(1000, 10)
    assert np.array_equal(B.rowval, C.rowval) and 9000 < B.nnz <= 10000
    assert int(synth.splitmix64(np.uint64(0))) == 0xE220A8397B1DCDAF
    R = synth.rmat(8, 2048)
    assert R.n == 256 and 0 < R.nnz <= 2048
    G = synth.random_geometric(2000)
    S = G.to_scipy()
    assert (S != S.T).nnz == 0 and S.diagonal().sum() == 0
    Bd = synth.banded(300, 8)
    d = Bd.to_scipy().tocoo()
    assert np.all(np.abs(d.row - d.col) <= 8) and np.all(Bd.to_scipy().diagonal() == 1)
