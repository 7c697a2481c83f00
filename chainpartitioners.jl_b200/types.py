"""Host-side vocabulary mirroring ChainPartitioners.jl's public types.

Same names, argument order and meaning as the reference so that call sites read
like the Julia ones:

  * matrices / partitions : SparseMatrixCSC, SplitPartition, MapPartition,
    DomainPartition                       (src/Partitions.jl:3-81)
  * hints                 : NoHint, RandomHint, SparseHint, StepHint
                                          (src/ChainPartitioners.jl:172-176)
  * cost models           : Affine*Model, ColumnBlockComponentCostModel,
    BlockComponentCostModel, ConstrainedCost, VertexCount
                                          (src/*Costs.jl, src/Costs.jl:105-147)
  * methods               : Dynamic*/Bisect*/LazyBisect* splitters, chunkers,
    Alternating*/Symmetric* drivers       (src/*Splitter.jl, src/*Chunker.jl,
                                           src/AlternatingPartitioner.jl)

Everything here is plain data; the arithmetic lives in the CUDA library behind
the C ABI (include/chainb200.h).  Indices are 1-based Int64 exactly as Julia
stores them.
"""
from __future__ import annotations

import ctypes
import numbers
from dataclasses import dataclass, field
from typing import Any, Callable, Optional, Sequence, Tuple, Union

import numpy as np

I64 = np.int64

# --------------------------------------------------------------------------- matrices


class SparseMatrixCSC:
    """Pattern of a Julia ``SparseMatrixCSC{Tv,Int64}``: ``colptr`` (n+1) and ``rowval`` (nnz),
    both 1-based.  Values are irrelevant to every oracle on the path (util.jl:33 ``pattern``)."""

    __slots__ = ("m", "n", "colptr", "rowval")

    def __init__(self, m: int, n: int, colptr, rowval):
        self.m = int(m)
        self.n = int(n)
        self.colptr = np.ascontiguousarray(colptr, dtype=I64)
        self.rowval = np.ascontiguousarray(rowval, dtype=I64)
        if self.colptr.shape != (self.n + 1,):
            raise ValueError("colptr must have n+1 entries")
        if self.n >= 0 and (self.colptr[0] != 1 or self.colptr[-1] != self.rowval.shape[0] + 1):
            raise ValueError("colptr must be 1-based with colptr[n+1] == nnz+1")

    @property
    def nnz(self) -> int:
        return int(self.rowval.shape[0])

    @property
    def shape(self) -> Tuple[int, int]:
        return (self.m, self.n)

    @classmethod
    def from_scipy(cls, S) -> "SparseMatrixCSC":
        S = S.tocsc()
        S.sort_indices()
        S.sum_duplicates()
        return cls(S.shape[0], S.shape[1], S.indptr.astype(I64) + 1, S.indices.astype(I64) + 1)

    @classmethod
    def from_coo(cls, m, n, I, J) -> "SparseMatrixCSC":
        """``sparse(I, J, V, m, n)`` with 1-based I, J (duplicates merged, rows sorted)."""
        import scipy.sparse as sp

        I = np.asarray(I, dtype=I64) - 1
        J = np.asarray(J, dtype=I64) - 1
        S = sp.coo_matrix((np.ones(len(I), dtype=np.int8), (I, J)), shape=(m, n)).tocsc()
        return cls.from_scipy(S)

    def to_scipy(self):
        import scipy.sparse as sp

        return sp.csc_matrix(
            (np.ones(self.nnz, dtype=np.int8), self.rowval - 1, self.colptr - 1), shape=(self.m, self.n)
        )

    def __repr__(self):
        return f"SparseMatrixCSC({self.m}x{self.n}, nnz={self.nnz})"


# --------------------------------------------------------------------------- partitions


@dataclass
class SplitPartition:
    """Partitions.jl:3-6 -- contiguous parts ``spl[k] .. spl[k+1]-1`` (1-based, K+1 entries)."""

    K: int
    spl: np.ndarray

    def __post_init__(self):
        self.K = int(self.K)
        self.spl = np.ascontiguousarray(self.spl, dtype=I64)

    def __len__(self):
        return self.K

    def __eq__(self, other):
        return isinstance(other, SplitPartition) and np.array_equal(self.spl, other.spl)


@dataclass
class MapPartition:
    """Partitions.jl:19-22 -- ``asg[j]`` = part of element j."""

    K: int
    asg: np.ndarray

    def __post_init__(self):
        self.K = int(self.K)
        self.asg = np.ascontiguousarray(self.asg, dtype=I64)

    def __len__(self):
        return self.K

    def __eq__(self, other):
        return isinstance(other, MapPartition) and self.K == other.K and np.array_equal(self.asg, other.asg)


@dataclass
class DomainPartition:
    """Partitions.jl:10-15 -- permutation ``prm`` grouped by part with offsets ``spl``."""

    K: int
    prm: np.ndarray
    spl: np.ndarray

    def __post_init__(self):
        self.K = int(self.K)
        self.prm = np.ascontiguousarray(self.prm, dtype=I64)
        self.spl = np.ascontiguousarray(self.spl, dtype=I64)

    def __len__(self):
        return self.K

    def __eq__(self, other):
        return (
            isinstance(other, DomainPartition)
            and np.array_equal(self.prm, other.prm)
            and np.array_equal(self.spl, other.spl)
        )


def convert(T, P):
    """``Base.convert`` between partition types (Partitions.jl:37-81)."""
    if isinstance(P, T):
        return P
    if T is DomainPartition and isinstance(P, SplitPartition):
        return DomainPartition(P.K, np.arange(1, int(P.spl[-1]), dtype=I64), P.spl.copy())
    if T is DomainPartition and isinstance(P, MapPartition):
        order = np.argsort(P.asg, kind="stable")
        counts = np.bincount(P.asg - 1, minlength=P.K)
        spl = np.concatenate(([1], 1 + np.cumsum(counts))).astype(I64)
        return DomainPartition(P.K, order.astype(I64) + 1, spl)
    if T is MapPartition and isinstance(P, SplitPartition):
        widths = np.diff(P.spl)
        return MapPartition(P.K, np.repeat(np.arange(1, P.K + 1, dtype=I64), widths))
    if T is MapPartition and isinstance(P, DomainPartition):
        asg = np.empty(int(P.spl[-1]) - 1, dtype=I64)
        widths = np.diff(P.spl)
        asg[P.prm - 1] = np.repeat(np.arange(1, P.K + 1, dtype=I64), widths)
        return MapPartition(P.K, asg)
    raise TypeError(f"no conversion {type(P).__name__} -> {T.__name__} (none in the reference either)")


# --------------------------------------------------------------------------- hints


class AbstractHint:
    code = 0


class NoHint(AbstractHint):
    code = 0


class RandomHint(AbstractHint):
    code = 1


class SparseHint(AbstractHint):
    code = 2


class StepHint(AbstractHint):
    code = 3


# --------------------------------------------------------------------------- cost models

MODEL_WORK, MODEL_CONNECTIVITY, MODEL_MONOSYM, MODEL_SYMCONN = 0, 1, 2, 3
MODEL_HYPEREDGE, MODEL_SYMEDGECUT, MODEL_ENVELOPE, MODEL_COLBLOCK, MODEL_BLOCK, MODEL_PRIMCONN, MODEL_SECCONN = 4, 5, 6, 7, 8, 9, 10
MODEL_PRIMEDGE, MODEL_SECEDGE = 11, 12


def _is_int(x) -> bool:
    return isinstance(x, (bool, numbers.Integral, np.integer))


class CModel(ctypes.Structure):
    """Binary layout of ``cpb_model`` (include/chainb200.h); the CPU oracle's ``cpo_model`` is
    declared with the same layout on purpose so one packer serves both."""

    _fields_ = [
        ("kind", ctypes.c_int32),
        ("is_float", ctypes.c_int32),
        ("coef", ctypes.c_double * 8),
        ("R", ctypes.c_int32),
        ("w_tab", ctypes.c_int32),
        ("u_tab", ctypes.c_int32),
        ("_pad", ctypes.c_int32),
        ("alpha_col", ctypes.POINTER(ctypes.c_double)),
        ("beta_col", ctypes.POINTER(ctypes.c_double)),
        ("beta_row", ctypes.POINTER(ctypes.c_double)),
    ]


class CConstraint(ctypes.Structure):
    """Binary layout of ``cpb_constraint``."""

    _fields_ = [
        ("enabled", ctypes.c_int32),
        ("_pad", ctypes.c_int32),
        ("w_coef", ctypes.c_int64 * 3),
        ("w_max", ctypes.c_int64),
    ]


class _AffineModel:
    kind = -1
    names: Tuple[str, ...] = ()

    def __init__(self, *args, **kwargs):
        vals = list(args)
        if len(vals) > len(self.names):
            raise TypeError(f"{type(self).__name__} takes {len(self.names)} coefficients")
        for name in self.names[len(vals):]:
            vals.append(kwargs.pop(name, False))  # Julia keyword constructors default to `false`
        if kwargs:
            raise TypeError(f"unknown coefficients {sorted(kwargs)}")
        # promote(...) : Int64 if every coefficient is an integer, else Float64
        self.is_float = not all(_is_int(v) for v in vals)
        self.coef = tuple(float(v) if self.is_float else int(v) for v in vals)
        for name, v in zip(self.names, self.coef):
            setattr(self, name, v)

    def to_c(self, **_) -> Tuple[CModel, list]:
        c = CModel()
        c.kind = self.kind
        c.is_float = int(self.is_float)
        for t, v in enumerate(self.coef):
            c.coef[t] = float(v)
        return c, []

    def __repr__(self):
        body = ", ".join(f"{n}={v}" for n, v in zip(self.names, self.coef))
        return f"{type(self).__name__}({body})"


class AffineWorkModel(_AffineModel):
    """WorkCosts.jl:5-17: ``alpha + n_vertices*beta_vertex + n_pins*beta_pin``."""

    kind = MODEL_WORK
    names = ("alpha", "beta_vertex", "beta_pin")


class AffineConnectivityModel(_AffineModel):
    """ConnectivityCosts.jl:7-20: ``... + n_nets*beta_net``."""

    kind = MODEL_CONNECTIVITY
    names = ("alpha", "beta_vertex", "beta_pin", "beta_net")


class AffineMonotonizedSymmetricConnectivityModel(_AffineModel):
    """MonotonizedSymmetricConnectivityCosts.jl:5-33."""

    kind = MODEL_MONOSYM
    names = ("alpha", "beta_vertex", "beta_over_pin", "beta_dia_net", "delta_pins")


class AffineSymmetricConnectivityModel(_AffineModel):
    """SymmetricConnectivityCosts.jl:5-19."""

    kind = MODEL_SYMCONN
    names = ("alpha", "beta_vertex", "beta_pin", "beta_local_net", "beta_remote_net")


class AffineHyperedgeCutModel(_AffineModel):
    """HyperedgeCutCosts.jl:7-21."""

    kind = MODEL_HYPEREDGE
    names = ("alpha", "beta_vertex", "beta_pin", "beta_self_net", "beta_cut_net")


class AffineSymmetricEdgeCutModel(_AffineModel):
    """SymmetricEdgeCutCosts.jl:5-18."""

    kind = MODEL_SYMEDGECUT
    names = ("alpha", "beta_vertex", "beta_self_pin", "beta_cut_pin")


class AffinePrimaryConnectivityModel(_AffineModel):
    """PrimaryConnectivityCosts.jl:5-19: ``alpha + n_vertices*beta_vertex + n_pins*beta_pin + n_local_nets*beta_local_net +
    n_remote_nets*beta_remote_net`` where a net of part k's columns is local if row part k of Pi owns it; always used
    with a row partition (``oracle_stripe(mdl, A, Pi)``, ``partition_stripe(A, K, method, Pi)``)."""

    kind = MODEL_PRIMCONN
    names = ("alpha", "beta_vertex", "beta_pin", "beta_local_net", "beta_remote_net")


class AffineSecondaryConnectivityModel(_AffineModel):
    """SecondaryConnectivityCosts.jl:5-19: the cost of part k seen from the other side -- vertex, pin and net totals of
    row part k of Pi are fixed, only the number of its nets (columns) that fall inside the column range [i, i') -- the
    local ones -- depends on the split; used as ``partition_stripe(adj_A, K, method, Phi)``."""

    kind = MODEL_SECCONN
    names = ("alpha", "beta_vertex", "beta_pin", "beta_local_net", "beta_remote_net")


class AffinePrimaryEdgeCutModel(_AffineModel):
    """PrimaryEdgeCutCosts.jl:5-18: ``alpha + n_vertices*beta_vertex + n_self_pins*beta_self_pin + n_cut_pins*beta_cut_pin``;
    a pin of part k's columns is a self pin if row part k of Pi owns its row."""

    kind = MODEL_PRIMEDGE
    names = ("alpha", "beta_vertex", "beta_self_pin", "beta_cut_pin")


class AffineSecondaryEdgeCutModel(_AffineModel):
    """SecondaryEdgeCutCosts.jl:5-18: the same seen from the other side (vertices and pins of row part k fixed, its pins
    inside the column range [i, i') are the self pins)."""

    kind = MODEL_SECEDGE
    names = ("alpha", "beta_vertex", "beta_self_pin", "beta_cut_pin")


class AffineEnvelopeModel(_AffineModel):
    """EnvelopeCosts.jl:5-20."""

    kind = MODEL_ENVELOPE
    names = ("alpha", "beta_vertex", "beta_pin", "beta_net")


def identity(x):
    return x


def block_component(f, w: int):
    """BlockCosts.jl:41-44: number -> itself, tuple/array -> f[w] (1-based), callable -> f(w)."""
    if callable(f):
        return f(w)
    if isinstance(f, (tuple, list, np.ndarray)):
        return f[w - 1] if 1 <= w <= len(f) else 0
    return f


def _tabulate(f, hi: int) -> np.ndarray:
    return np.array([float(block_component(f, w)) for w in range(hi + 1)], dtype=np.float64)


class ColumnBlockComponentCostModel:
    """BlockCosts.jl:1-17 (1-D VBR): ``alpha_col(w) + n_nets * beta_col(w)``.  Functors cannot
    cross the C ABI, so components are tabulated for widths ``0..w_tab`` on the host."""

    kind = MODEL_COLBLOCK

    def __init__(self, Tv=int, alpha_col=False, beta_col=False):
        self.is_float = Tv is float
        self.alpha_col = alpha_col
        self.beta_col = beta_col

    def to_c(self, w_tab: int = 0, **_):
        c = CModel()
        c.kind = self.kind
        c.is_float = int(self.is_float)
        c.R = 1
        c.w_tab = int(w_tab)
        a = _tabulate(self.alpha_col, w_tab)
        b = _tabulate(self.beta_col, w_tab)
        c.alpha_col = a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        c.beta_col = b.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        return c, [a, b]


class BlockComponentCostModel:
    """BlockCosts.jl:19-44 (2-D VBR): ``alpha_col(w) + sum_r d_r * beta_col[r](w)`` with
    ``d_r = sum over row parts k touched by the columns of beta_row[r](u_k)``."""

    kind = MODEL_BLOCK

    def __init__(self, Tv=int, alpha_row=False, alpha_col=False, beta_row=(), beta_col=()):
        if len(beta_row) != len(beta_col):
            raise ValueError("beta_row and beta_col must have the same length R")
        self.is_float = Tv is float
        self.alpha_row, self.alpha_col = alpha_row, alpha_col
        self.beta_row, self.beta_col = tuple(beta_row), tuple(beta_col)

    def permutedims(self):
        return BlockComponentCostModel(float if self.is_float else int, self.alpha_col, self.alpha_row, self.beta_col, self.beta_row)

    def to_c(self, w_tab: int = 0, u_tab: int = 0, **_):
        c = CModel()
        c.kind = self.kind
        c.is_float = int(self.is_float)
        R = len(self.beta_row)
        c.R, c.w_tab, c.u_tab = R, int(w_tab), int(u_tab)
        a = _tabulate(self.alpha_col, w_tab)
        bc = np.concatenate([_tabulate(f, w_tab) for f in self.beta_col]) if R else np.zeros(1)
        br = np.concatenate([_tabulate(f, u_tab) for f in self.beta_row]) if R else np.zeros(1)
        c.alpha_col = a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        c.beta_col = bc.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        c.beta_row = br.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        return c, [a, bc, br]


class VertexCount:
    """SparseColorArrays.jl:1-6: ``w(j, j') = j' - j``."""

    w_coef = (0, 1, 0)


class FeasibleCost:
    """Costs.jl:164-171: the "no constraint" weight."""


@dataclass
class ConstrainedCost:
    """Costs.jl:105-147: cost ``f`` if ``w(j,j') <= w_max`` else +inf, ``w(j, j')`` being the weight model's own cost of
    the columns ``j..j'-1``.  ``w`` is ``VertexCount()`` or an integer ``AffineWorkModel`` (an affine work weight, the form
    every solver takes), or -- for ``partition_stripe`` with the Dynamic, Convex and Concave splitters -- an integer
    ``AffineConnectivityModel`` or ``AffineMonotonizedSymmetricConnectivityModel`` with non-negative betas (a count
    weight: distinct rows, i.e. a part's footprint).  The count weight gets an oracle of its own on the same matrix."""

    f: Any
    w: Any
    w_max: Any

    def count_weight(self):
        """The weight model if it is evaluated through an oracle of its own (anything but an affine work weight), else None."""
        if isinstance(self.w, (FeasibleCost, VertexCount)) or (isinstance(self.w, AffineWorkModel) and not self.w.is_float):
            return None
        return self.w if isinstance(self.w, _AffineModel) else None

    def constraint(self) -> CConstraint:
        c = CConstraint()
        if isinstance(self.w, FeasibleCost):
            c.enabled = 0
            return c
        if isinstance(self.w, VertexCount):
            coef = VertexCount.w_coef
        elif isinstance(self.w, AffineWorkModel) and not self.w.is_float:
            coef = self.w.coef
        elif self.count_weight() is not None:
            raise TypeError("a count weight (AffineConnectivityModel / AffineMonotonizedSymmetricConnectivityModel) is taken by "
                            "partition_stripe's Dynamic, Convex and Concave splitters only; here the weight must be VertexCount() "
                            "or an integer AffineWorkModel")
        else:
            raise TypeError("ConstrainedCost weight must be VertexCount() or an integer AffineWorkModel")
        c.enabled = 1
        for t in range(3):
            c.w_coef[t] = int(coef[t])
        c.w_max = int(self.w_max)
        return c


def split_constrained(f) -> Tuple[Any, CConstraint]:
    if isinstance(f, ConstrainedCost):
        return f.f, f.constraint()
    return f, CConstraint()


# --------------------------------------------------------------------------- methods


@dataclass
class DynamicBottleneckSplitter:
    """DynamicSplitter.jl:3-7."""
    f: Any


@dataclass
class DynamicTotalSplitter:
    """DynamicSplitter.jl:9-13."""
    f: Any


ReferenceBottleneckSplitter = DynamicBottleneckSplitter  # ReferenceSplitter.jl:8-13 (same generic method)
ReferenceTotalSplitter = DynamicTotalSplitter            # ReferenceSplitter.jl:1-6


@dataclass
class BisectCostBottleneckSplitter:
    """BisectCostBottleneckSplitter.jl:1-4."""
    f: Any
    eps: float


@dataclass
class FlipBisectCostBottleneckSplitter:
    """BisectCostBottleneckSplitter.jl:65-68."""
    f: Any
    eps: float


@dataclass
class BisectIndexBottleneckSplitter:
    """BisectIndexBottleneckSplitter.jl:1-3 (exact bottleneck, :5-81)."""
    f: Any


@dataclass
class FlipBisectIndexBottleneckSplitter:
    """BisectIndexBottleneckSplitter.jl:83-85 (exact bottleneck for decreasing costs, :87-166)."""
    f: Any


@dataclass
class LazyBisectCostBottleneckSplitter:
    """LazyBisectCostBottleneckSplitter.jl:1-4."""
    f: Any
    eps: float


@dataclass
class LazyFlipBisectCostBottleneckSplitter:
    """LazyBisectCostBottleneckSplitter.jl:72-75."""
    f: Any
    eps: float


class EquiSplitter:
    """EquiPartitioner.jl:1."""


@dataclass
class EquiChunker:
    """EquiPartitioner.jl:11-13."""
    w: int


@dataclass
class DynamicBottleneckChunker:
    """DynamicChunker.jl:3-5 (only usable through partition_stripe: DynamicSplitter.jl:52-87)."""
    f: Any


class DynamicTotalChunker:
    """DynamicChunker.jl:9-11; the deprecated two-argument form ``DynamicTotalChunker(f, w_max)``
    means ``ConstrainedCost(f, VertexCount(), w_max)`` (ChainPartitioners.jl:221)."""

    def __init__(self, f, w_max=None):
        self.f = ConstrainedCost(f, VertexCount(), w_max) if w_max is not None else f


ReferenceTotalChunker = DynamicTotalChunker  # ReferenceSplitter.jl:16-20


@dataclass
class ConvexTotalChunker:
    """ConvexTotalChunker.jl:1-3."""
    f: Any


@dataclass
class ConcaveTotalChunker:
    """ConcaveTotalChunker.jl:1-3."""
    f: Any


@dataclass
class ConvexTotalSplitter:
    """ConvexTotalChunker.jl:5-7 (partition_stripe, :26-55)."""
    f: Any


@dataclass
class ConcaveTotalSplitter:
    """ConcaveTotalChunker.jl:5-7 (partition_stripe, :26-55)."""
    f: Any


@dataclass
class OverlapChunker:
    """OverlapChunker.jl:1-4."""
    rho: float
    w_max: int


@dataclass
class StrictChunker:
    """StrictChunker.jl:1-3."""
    w_max: int


class AlternatingPartitioner:
    """AlternatingPartitioner.jl:11-16."""

    def __init__(self, *mtds):
        self.mtds = mtds


class AlternatingNetPartitioner(AlternatingPartitioner):
    """AlternatingPartitioner.jl:34-57: AlternatingPartitioner that shares one net count of ``A`` between the solves
    (``net=`` keyword).  The hint only chooses a CPU data structure in the reference; the result is the alternation's."""

    def __init__(self, *mtds):
        if mtds and isinstance(mtds[0], (NoHint, SparseHint, StepHint, RandomHint)):
            mtds = mtds[1:]
        super().__init__(*mtds)


class SymmetricPartitioner:
    """AlternatingPartitioner.jl:59-69."""

    def __init__(self, *mtds):
        self.mtds = mtds


@dataclass
class DisjointPartitioner:
    """AlternatingPartitioner.jl:1-4."""
    mtd: Any
    mtd2: Any


class AlternatingPacker:
    """AlternatingPacker.jl:12-16."""

    def __init__(self, *mtds):
        self.mtds = mtds


class SymmetricPacker:
    """AlternatingPacker.jl:33-37."""

    def __init__(self, *mtds):
        self.mtds = mtds


@dataclass
class DisjointPacker:
    """AlternatingPacker.jl:1-4."""
    mtd: Any
    mtd2: Any


# method codes shared by the C ABI (include/chainb200.h) and the CPU oracle (oracle/cpo.h)
SPLIT_DYNAMIC_BOTTLENECK, SPLIT_DYNAMIC_TOTAL, SPLIT_BISECT_COST, SPLIT_LAZY_BISECT_COST = 0, 1, 2, 3
SPLIT_LAZY_BISECT_GENERIC, SPLIT_EQUI, SPLIT_FLIP_BISECT_COST, SPLIT_LAZY_FLIP_BISECT_COST = 4, 5, 6, 7
SPLIT_CONVEX_TOTAL, SPLIT_CONCAVE_TOTAL = 8, 9
SPLIT_DYNAMIC_BOTTLENECK_CHUNKER, SPLIT_DYNAMIC_TOTAL_CHUNKER, SPLIT_BISECT_INDEX, SPLIT_FLIP_BISECT_INDEX = 10, 11, 12, 13
PACK_DYNAMIC_TOTAL, PACK_CONVEX_TOTAL, PACK_CONCAVE_TOTAL, PACK_OVERLAP, PACK_STRICT, PACK_EQUI = 0, 1, 2, 3, 4, 5


def split_method_code(method) -> Tuple[int, Any, float]:
    """-> (method code, cost spec or None, eps)."""
    if isinstance(method, DynamicBottleneckSplitter):
        return SPLIT_DYNAMIC_BOTTLENECK, method.f, 0.0
    if isinstance(method, DynamicTotalSplitter):
        return SPLIT_DYNAMIC_TOTAL, method.f, 0.0
    if isinstance(method, BisectCostBottleneckSplitter):
        return SPLIT_BISECT_COST, method.f, float(method.eps)
    if isinstance(method, BisectIndexBottleneckSplitter):
        return SPLIT_BISECT_INDEX, method.f, 0.0
    if isinstance(method, FlipBisectIndexBottleneckSplitter):
        return SPLIT_FLIP_BISECT_INDEX, method.f, 0.0
    if isinstance(method, FlipBisectCostBottleneckSplitter):
        return SPLIT_FLIP_BISECT_COST, method.f, float(method.eps)
    if isinstance(method, LazyBisectCostBottleneckSplitter):
        return SPLIT_LAZY_BISECT_COST, method.f, float(method.eps)
    if isinstance(method, LazyFlipBisectCostBottleneckSplitter):
        return SPLIT_LAZY_FLIP_BISECT_COST, method.f, float(method.eps)
    if isinstance(method, EquiSplitter):
        return SPLIT_EQUI, None, 0.0
    if isinstance(method, ConvexTotalSplitter):
        return SPLIT_CONVEX_TOTAL, method.f, 0.0
    if isinstance(method, ConcaveTotalSplitter):
        return SPLIT_CONCAVE_TOTAL, method.f, 0.0
    # partition_stripe(A, K, ::AbstractDynamicChunker) (DynamicSplitter.jl:52-87): the K-part DP with the part
    # index as the inner loop
    if isinstance(method, DynamicBottleneckChunker):
        return SPLIT_DYNAMIC_BOTTLENECK_CHUNKER, method.f, 0.0
    if isinstance(method, DynamicTotalChunker):
        return SPLIT_DYNAMIC_TOTAL_CHUNKER, method.f, 0.0
    raise TypeError(f"partition_stripe: unsupported method {type(method).__name__}")


def pack_method_code(method) -> Tuple[int, Any, float, int]:
    """-> (method code, cost spec or None, rho, w_max)."""
    if isinstance(method, DynamicTotalChunker):
        return PACK_DYNAMIC_TOTAL, method.f, 0.0, 0
    if isinstance(method, ConvexTotalChunker):
        return PACK_CONVEX_TOTAL, method.f, 0.0, 0
    if isinstance(method, ConcaveTotalChunker):
        return PACK_CONCAVE_TOTAL, method.f, 0.0, 0
    if isinstance(method, OverlapChunker):
        return PACK_OVERLAP, None, float(method.rho), int(method.w_max)
    if isinstance(method, StrictChunker):
        return PACK_STRICT, None, 0.0, int(method.w_max)
    if isinstance(method, EquiChunker):
        return PACK_EQUI, None, 0.0, int(method.w)
    raise TypeError(f"pack_stripe: unsupported method {type(method).__name__}")


def model_tables(mdl, A: SparseMatrixCSC, con: CConstraint, Pi: Optional[SplitPartition]) -> dict:
    """Table extents for tabulated (block) models: widths up to the window (or n), part sizes up to
    the largest row part."""
    w_tab = A.n
    if con.enabled and con.w_coef[1] > 0 and con.w_coef[2] >= 0 and con.w_coef[0] >= 0:
        w_tab = min(A.n, int(con.w_max) // int(con.w_coef[1]) + 1)
    u_tab = 0
    if Pi is not None and len(Pi.spl) > 1:
        u_tab = int(np.max(np.diff(Pi.spl)))
    return dict(w_tab=int(w_tab), u_tab=int(u_tab))
