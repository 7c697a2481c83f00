"""Host-side mirror of ChainPartitioners.jl's functions over the C ABI of libchainb200.so.

``partition_stripe`` / ``pack_stripe`` / ``partition_plaid`` / ``pack_plaid`` / ``oracle_stripe`` /
``bound_stripe`` / ``bottleneck_value`` / ``total_value`` / ``netcount`` ... take the same arguments, in
the same order, with the same meaning as the Julia methods they stand for (file:line in
include/chainb200.h).  All arithmetic runs on the GPU; there is no CPU fallback -- if the CUDA library
is missing or no device is visible every call raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import numpy as np

from . import types as T

__all__ = [
    "DeviceMatrix", "device_matrix", "device_matrix_i32", "adjointpattern", "permute", "oracle_stripe", "bound_stripe", "partition_stripe",
    "pack_stripe", "partition_plaid", "pack_plaid", "bottleneck_value", "total_value", "pincount", "netcount",
    "dianetcount", "selfnetcount", "selfpincount", "PrefixMatrix", "dominancecount", "dominancesum", "rookcount", "rooksum", "profile_enable", "profile_reset", "profile_get",
    "Communicator", "ShardedMatrix", "partition_stripe_sharded", "partition_stripe_sharded_emulated", "sharded_stats", "shard_range",
    "partition_plaid_sharded", "partition_plaid_sharded_emulated", "adjointpattern_sharded_emulated",
    "weight_windows", "launch_count", "bisect_stats", "bisect_plan", "bisect_prewalk", "timer_start", "timer_stop", "StripeOracle", "init", "synchronize", "trim_memory", "library_path", "load_library", "CpbError",
]

I64 = np.int64
_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("CHAINB200_LIB") or os.path.join(_HERE, "libchainb200.so")  # override: instrumented builds only
_lib = None

ABI_SYMBOLS = [
    "cpb_last_error", "cpb_version", "cpb_init", "cpb_device_count", "cpb_synchronize", "cpb_matrix_create",
    "cpb_matrix_create_device", "cpb_matrix_dims", "cpb_matrix_get", "cpb_matrix_destroy", "cpb_adjointpattern",
    "cpb_oracle_create", "cpb_oracle_destroy", "cpb_oracle_query", "cpb_oracle_query_device", "cpb_count_query",
    "cpb_bound_stripe", "cpb_objective", "cpb_partition_stripe", "cpb_pack_stripe", "cpb_profile_enable",
    "cpb_profile_reset", "cpb_profile_get", "cpb_launch_count", "cpb_timer_start", "cpb_timer_stop",
    "cpb_bisect_stats", "cpb_bisect_plan", "cpb_bisect_prewalk",
    "cpb_comm_unique_id", "cpb_comm_init", "cpb_comm_destroy", "cpb_comm_info", "cpb_shard_range", "cpb_sharded_matrix_create", "cpb_sharded_matrix_destroy",
    "cpb_partition_stripe_sharded", "cpb_partition_stripe_sharded_emulated", "cpb_sharded_stats",
    "cpb_sharded_adjointpattern", "cpb_adjointpattern_sharded_emulated", "cpb_sharded_matrix_get",
    "cpb_prefix_create", "cpb_prefix_query", "cpb_prefix_destroy", "cpb_matrix_permute", "cpb_trim_memory", "cpb_matrix_create_i32",
    "cpb_partition_stripe_weighted", "cpb_weight_windows",
]


class CpbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libchainb200 error {code}: {msg}")
        self.code = code


def library_path() -> str:
    return _LIB_PATH


def load_library():
    """Loads libchainb200.so (built in-tree by ``__graft_entry__.build()``); raises if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise RuntimeError(
                f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(this package has no CPU fallback)"
            )
        lib = ctypes.CDLL(_LIB_PATH)
        lib.cpb_last_error.restype = ctypes.c_char_p
        lib.cpb_launch_count.restype = ctypes.c_int64
        vp, i64, dbl, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_double, ctypes.c_int
        lib.cpb_matrix_create.argtypes = [i64, i64, i64, vp, vp, ctypes.POINTER(vp)]
        lib.cpb_matrix_create_device.argtypes = [i64, i64, i64, vp, vp, ctypes.POINTER(vp)]
        lib.cpb_matrix_dims.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(i64), ctypes.POINTER(i64)]
        lib.cpb_matrix_get.argtypes = [vp, vp, vp]
        lib.cpb_matrix_destroy.argtypes = [vp]
        lib.cpb_matrix_destroy.restype = None
        lib.cpb_adjointpattern.argtypes = [vp, ctypes.POINTER(vp)]
        lib.cpb_oracle_create.argtypes = [vp, ctypes.POINTER(T.CModel), vp, i64, ctypes.POINTER(vp)]
        lib.cpb_oracle_destroy.argtypes = [vp]
        lib.cpb_oracle_destroy.restype = None
        lib.cpb_oracle_query.argtypes = [vp, i64, vp, vp, vp, vp]
        lib.cpb_oracle_query_device.argtypes = [vp, i64, vp, vp, vp]
        lib.cpb_count_query.argtypes = [vp, i32, i64, vp, vp, vp]
        lib.cpb_bound_stripe.argtypes = [vp, i64, ctypes.POINTER(dbl)]
        lib.cpb_objective.argtypes = [vp, i32, i64, vp, ctypes.POINTER(dbl)]
        lib.cpb_partition_stripe.argtypes = [vp, i32, ctypes.POINTER(T.CConstraint), dbl, i64, vp]
        lib.cpb_partition_stripe_weighted.argtypes = [vp, i32, vp, i64, dbl, i64, vp]
        lib.cpb_weight_windows.argtypes = [vp, i64, vp, vp]
        lib.cpb_pack_stripe.argtypes = [vp, vp, i32, ctypes.POINTER(T.CConstraint), dbl, i64, vp, ctypes.POINTER(i64), vp]
        lib.cpb_profile_get.argtypes = [i32, vp, vp, vp, vp]
        lib.cpb_comm_unique_id.argtypes = [vp]
        lib.cpb_comm_init.argtypes = [vp, i32, i32]
        lib.cpb_comm_info.argtypes = [ctypes.POINTER(i32), ctypes.POINTER(i32)]
        lib.cpb_shard_range.argtypes = [i64, i32, i32, ctypes.POINTER(i64), ctypes.POINTER(i64)]
        lib.cpb_sharded_matrix_create.argtypes = [i64, i64, i64, vp, vp, i32, ctypes.POINTER(vp)]
        lib.cpb_sharded_matrix_destroy.argtypes = [vp]
        lib.cpb_sharded_matrix_destroy.restype = None
        lib.cpb_partition_stripe_sharded.argtypes = [vp, ctypes.POINTER(T.CModel), i32, dbl, i64, vp]
        lib.cpb_partition_stripe_sharded_emulated.argtypes = [vp, ctypes.POINTER(T.CModel), i32, dbl, i64, i32, vp]
        lib.cpb_sharded_stats.argtypes = [vp]
        lib.cpb_sharded_adjointpattern.argtypes = [vp, ctypes.POINTER(vp)]
        lib.cpb_adjointpattern_sharded_emulated.argtypes = [vp, i32, ctypes.POINTER(vp)]
        lib.cpb_sharded_matrix_get.argtypes = [vp, vp, vp, ctypes.POINTER(i64), ctypes.POINTER(i64)]
        _lib = lib
    return _lib


def _check(rc):
    if rc != 0:
        raise CpbError(rc, load_library().cpb_last_error().decode())


def init(device: int = 0):
    """One process per GPU: selects the CUDA device of this process."""
    _check(load_library().cpb_init(int(device)))


def synchronize():
    _check(load_library().cpb_synchronize())


def _arr(x) -> np.ndarray:
    return np.ascontiguousarray(x, dtype=I64)


def _p(a: Optional[np.ndarray]):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else ctypes.c_void_p(0)


# ------------------------------------------------------------------------------- matrices


class DeviceMatrix:
    """A SparseMatrixCSC pattern resident in HBM (``cpb_matrix``)."""

    def __init__(self, handle, m, n, nnz):
        self._h = handle
        self.m, self.n, self._nnz = int(m), int(n), int(nnz)

    @property
    def nnz(self):
        return self._nnz

    @property
    def shape(self):
        return (self.m, self.n)

    def to_host(self) -> T.SparseMatrixCSC:
        colptr = np.empty(self.n + 1, dtype=I64)
        rowval = np.empty(self.nnz, dtype=I64)
        _check(load_library().cpb_matrix_get(self._h, _p(colptr), _p(rowval)))
        return T.SparseMatrixCSC(self.m, self.n, colptr, rowval)

    def close(self):
        if self._h is not None and _lib is not None:
            _lib.cpb_matrix_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def device_matrix(A) -> DeviceMatrix:
    """Uploads ``A`` (host SparseMatrixCSC) once; pass the result wherever a matrix is expected."""
    if isinstance(A, DeviceMatrix):
        return A
    h = ctypes.c_void_p()
    _check(load_library().cpb_matrix_create(A.m, A.n, A.nnz, _p(A.colptr), _p(A.rowval), ctypes.byref(h)))
    return DeviceMatrix(h, A.m, A.n, A.nnz)


# ------------------------------------------------------------------------------- 2-D prefix structures


def _as_i64_values(val):
    """Integer values as the 64-bit words the device sums (Julia's Int64 / UInt64 wrap-around arithmetic)."""
    val = np.asarray(val)
    if val.dtype.kind not in "iub":
        raise TypeError("dominance / rook sums on the device take integer values (Float64 sums depend on the summation order)")
    dtype = np.uint64 if val.dtype == np.uint64 else I64
    return np.ascontiguousarray(val.astype(dtype, copy=False)).view(I64), dtype


class PrefixMatrix:
    """``C = dominancecount(A)`` / ``S = dominancesum(A, val)`` / ``rookcount!(N, idx)`` / ``rooksum!(N, idx, val)``
    (SparsePrefixMatrices.jl:1-1273) resident in HBM: an ``(m+1) x (n+1)`` matrix, ``P[i, j]`` = number (or sum of the values)
    of the points ``(r, c)`` with ``r <= i-1`` and ``c <= j-1``.  ``P[i, j]`` answers one entry, ``P.query(i, j)`` a batch."""

    def __init__(self, handle, m, n, summed, dtype):
        self._h, self.m, self.n, self.summed, self.dtype = handle, int(m), int(n), bool(summed), dtype

    @property
    def shape(self):
        return (self.m + 1, self.n + 1)

    def query(self, i, j) -> np.ndarray:
        i, j = np.ascontiguousarray(i, dtype=I64), np.ascontiguousarray(j, dtype=I64)
        if i.shape != j.shape or i.ndim != 1:
            raise ValueError("i and j must be 1-d arrays of equal length")
        out = np.empty(len(i), dtype=I64)
        none = ctypes.c_void_p(0)
        _check(load_library().cpb_prefix_query(self._h, ctypes.c_longlong(len(i)), _p(i), _p(j), none if self.summed else _p(out), _p(out) if self.summed else none))
        return out.view(self.dtype)

    def __getitem__(self, ij):
        i, j = ij
        return self.query([int(i)], [int(j)])[0]

    def close(self):
        if self._h is not None and _lib is not None:
            _lib.cpb_prefix_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _prefix_create(m, n, N, pos, idx, val):
    idx = np.ascontiguousarray(idx, dtype=I64)
    pos = None if pos is None else np.ascontiguousarray(pos, dtype=I64)
    dtype = I64
    if val is not None:
        val, dtype = _as_i64_values(val)
        if val.shape != (N,):
            raise ValueError("one value per point expected")
    if idx.shape != (N,):
        raise ValueError("one row index per point expected")
    h = ctypes.c_void_p()
    _check(load_library().cpb_prefix_create(ctypes.c_longlong(m), ctypes.c_longlong(n), ctypes.c_longlong(N), _p(pos), _p(idx), _p(val), ctypes.byref(h)))
    return PrefixMatrix(h, m, n, val is not None, dtype)


def dominancecount(A, hint=None, **layout) -> PrefixMatrix:
    """``dominancecount([hint,] A; b, H, b')`` (SparsePrefixMatrices.jl:440-460).  The hint and the layout keywords select
    among the reference's CPU structures; the device has one index, so they are accepted and ignored."""
    return _prefix_create(A.m, A.n, A.nnz, A.colptr, A.rowval, None)


def dominancesum(A, val, hint=None, **layout) -> PrefixMatrix:
    """``dominancesum([hint,] A; ...)`` (SparsePrefixMatrices.jl:31-58); ``val`` = ``A.nzval`` (the host matrix type here
    holds the pattern only)."""
    return _prefix_create(A.m, A.n, A.nnz, A.colptr, A.rowval, val)


def rookcount(N, idx, hint=None, **layout) -> PrefixMatrix:
    """``rookcount!([hint,] N, idx)`` (SparsePrefixMatrices.jl:1056-1063): the points ``(idx[q], q)``."""
    return _prefix_create(N, N, N, None, idx, None)


def rooksum(N, idx, val, hint=None, **layout) -> PrefixMatrix:
    """``rooksum!([hint,] N, idx, val)`` (SparsePrefixMatrices.jl:840-851)."""
    return _prefix_create(N, N, N, None, idx, val)


def permute(A, col_prm=None, row_new=None) -> DeviceMatrix:
    """``A[:, col_prm]`` with row ``r`` renamed ``row_new[r]`` (1-based permutations, ``None`` = identity), built on the
    device -- the first step of ``compute_objective`` for non-contiguous partitions (Costs.jl:34-39, 52-57)."""
    with _Scoped(A) as dm:
        c = None if col_prm is None else _arr(col_prm)
        r = None if row_new is None else _arr(row_new)
        if (c is not None and c.shape != (dm.n,)) or (r is not None and r.shape != (dm.m,)):
            raise ValueError("col_prm needs n entries, row_new needs m entries")
        h = ctypes.c_void_p()
        _check(load_library().cpb_matrix_permute(dm._h, _p(c), _p(r), ctypes.byref(h)))
        return DeviceMatrix(h, dm.m, dm.n, dm.nnz)


def _rows_by_part(Pi, m):
    """A Map/DomainPartition of the rows as (row_new, SplitPartition): rows renumbered part by part (stable)."""
    dom = T.convert(T.DomainPartition, Pi)
    if dom.prm.shape != (m,):
        raise ValueError("row partition must cover the m rows")
    row_new = np.empty(m, dtype=I64)
    row_new[dom.prm - 1] = np.arange(1, m + 1, dtype=I64)
    return row_new, T.SplitPartition(dom.K, dom.spl)


def device_matrix_i32(m, n, colptr, rowval) -> DeviceMatrix:
    """Uploads the pattern of a ``SparseMatrixCSC{Tv, Int32}`` (1-based int32 ``colptr`` / ``rowval``): half the bytes of the
    Int64 form over PCIe."""
    colptr = np.ascontiguousarray(colptr, dtype=np.int32)
    rowval = np.ascontiguousarray(rowval, dtype=np.int32)
    if colptr.shape != (int(n) + 1,):
        raise ValueError("colptr must have n+1 entries")
    h = ctypes.c_void_p()
    _check(load_library().cpb_matrix_create_i32(int(m), int(n), int(rowval.shape[0]), _p(colptr), _p(rowval), ctypes.byref(h)))
    return DeviceMatrix(h, m, n, rowval.shape[0])


class _Scoped:
    """device view of a matrix argument; frees the upload on exit if we made it"""

    def __init__(self, A):
        self.owned = not isinstance(A, DeviceMatrix)
        self.dm = device_matrix(A)

    def __enter__(self):
        return self.dm

    def __exit__(self, *exc):
        if self.owned:
            self.dm.close()


def adjointpattern(A):
    """util.jl:67-95.  Host matrix in -> host matrix out; DeviceMatrix in -> DeviceMatrix out."""
    with _Scoped(A) as dm:
        h = ctypes.c_void_p()
        _check(load_library().cpb_adjointpattern(dm._h, ctypes.byref(h)))
        out = DeviceMatrix(h, dm.n, dm.m, dm.nnz)
        if isinstance(A, DeviceMatrix):
            return out
        res = out.to_host()
        out.close()
        return res


# ------------------------------------------------------------------------------- oracles


def _pi(Pi):
    if Pi is None:
        return None, 0
    if not isinstance(Pi, T.SplitPartition):
        raise TypeError("the row partition must be a SplitPartition (the reference has no MapPartition -> SplitPartition conversion either)")
    return _arr(Pi.spl), Pi.K


class StripeOracle:
    """``oracle_stripe(hint, mdl, A[, Pi])``: callable ``ocl(j, j'[, k])``; arrays are batched on the GPU.  For
    ``ConstrainedCost(f, w, w_max)`` with a count weight ``w`` (``ConstrainedCost.count_weight``), ``weight`` is a second
    oracle: ``w``'s own, on the same device matrix (its own wavelet index)."""

    def __init__(self, mdl, A, Pi=None, hint=None, w_tab=None):
        self.weight, self.w_max = None, None
        wmdl = mdl.count_weight() if isinstance(mdl, T.ConstrainedCost) else None
        if wmdl is not None:
            f, con = mdl.f, T.CConstraint()
            self.w_max = int(mdl.w_max)
        else:
            f, con = T.split_constrained(mdl)
        self.model, self.constraint = f, con
        self._h = None
        if Pi is not None and not isinstance(Pi, T.SplitPartition):
            if wmdl is not None and wmdl.kind == T.MODEL_MONOSYM:
                # the rows are renamed part by part below: the diagonal the weight counts would move
                raise TypeError("a monotonized-symmetric weight needs a SplitPartition of the rows (renaming the rows moves the diagonal)")
            # oracle_stripe converts any row partition to a MapPartition (PrimaryConnectivityCosts.jl:56-67); the device
            # structures want contiguous row parts, and the counts depend on a row only through its part: rename the rows
            row_new, Pi = _rows_by_part(Pi, A.m)
            A = permute(A, None, row_new)
            self._own = _Scoped(A)
            self._own.owned = True
        else:
            self._own = _Scoped(A)
        self.dm = self._own.dm
        self.Pi = Pi
        tabs = T.model_tables(f, self.dm, con, Pi) if hasattr(f, "to_c") else {}
        if w_tab is not None:
            tabs["w_tab"] = int(w_tab)
        cm, self._keep = f.to_c(**tabs)
        spl, pK = _pi(Pi)
        self._h = ctypes.c_void_p()
        _check(load_library().cpb_oracle_create(self.dm._h, ctypes.byref(cm), _p(spl), pK, ctypes.byref(self._h)))
        if wmdl is not None:
            self.weight = StripeOracle(wmdl, self.dm)

    def query(self, j, jp, k=None) -> np.ndarray:
        j, jp = _arr(np.atleast_1d(j)), _arr(np.atleast_1d(jp))
        out = np.empty(len(j), dtype=np.float64)
        kk = None
        if k is not None:  # the part index: only the row-partition-aware (primary) models read it
            kk = _arr(np.broadcast_to(np.atleast_1d(k), j.shape))
        _check(load_library().cpb_oracle_query(self._h, len(j), _p(j), _p(jp), _p(kk) if kk is not None else None, ctypes.c_void_p(out.ctypes.data)))
        if self.constraint.enabled:  # ConstrainedCostOracle (Costs.jl:141-147)
            w = self.constraint.w_coef
            dm_pos = None
            width = w[0] + (jp - j) * w[1]
            if w[2]:
                dm_pos = self.dm.to_host().colptr
                width = width + (dm_pos[jp - 1] - dm_pos[j - 1]) * w[2]
            out = np.where(width <= self.constraint.w_max, out, np.inf)
        if self.weight is not None:  # the same with the weight model's own oracle
            out = np.where(self.weight.query(j, jp) <= self.w_max, out, np.inf)
        return out

    def weight_windows(self):
        """``(first_fit, reach)`` of the count weight, 1-based, ``n + 1`` entries each (index ``c - 1`` is column ``c``):
        ``first_fit[j'-1]`` = smallest ``j <= j'`` with ``j == j'`` or ``w(j, j') <= w_max``, ``reach[j-1]`` = largest
        ``j' >= j`` with ``j' == j`` or ``w(j, j') <= w_max``."""
        if self.weight is None:
            raise TypeError("weight_windows needs a ConstrainedCost with a count weight")
        return weight_windows(self.weight, self.w_max)

    def query_device(self, d_j: int, d_jp: int, d_out: int, Q: int):
        """Batched queries on device-resident Int64 arrays (raw device pointers), result Float64 on the device."""
        _check(load_library().cpb_oracle_query_device(self._h, int(Q), ctypes.c_void_p(d_j), ctypes.c_void_p(d_jp), ctypes.c_void_p(d_out)))

    def __call__(self, j, jp, k=None):
        r = self.query(j, jp, k)
        if np.ndim(j) == 0:
            v = r[0]
            return v if (self.model.is_float or np.isinf(v)) else int(v)
        return r

    def close(self):
        if getattr(self, "weight", None) is not None:
            self.weight.close()
            self.weight = None
        if getattr(self, "_h", None) is not None and _lib is not None:
            _lib.cpb_oracle_destroy(self._h)
        self._h = None
        if getattr(self, "_own", None) is not None:
            self._own.__exit__()
            self._own = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def weight_windows(w: StripeOracle, w_max: int):
    """``cpb_weight_windows``: the windows of the weight oracle ``w`` under ``w_max`` (see ``StripeOracle.weight_windows``)."""
    n1 = w.dm.n + 1
    first_fit, reach = np.empty(n1, dtype=I64), np.empty(n1, dtype=I64)
    _check(load_library().cpb_weight_windows(w._h, int(w_max), _p(first_fit), _p(reach)))
    return first_fit, reach


def oracle_stripe(*args, **kwargs) -> StripeOracle:
    """``oracle_stripe([hint,] mdl, A[, Pi]; ...)`` (Costs.jl:3-7).  The hint only selects a CPU data
    structure in the reference; on the device one index serves all of them, so it is ignored."""
    args = list(args)
    hint = args.pop(0) if args and isinstance(args[0], T.AbstractHint) else None
    mdl, A = args[0], args[1]
    Pi = args[2] if len(args) > 2 else kwargs.get("Pi")
    return StripeOracle(mdl, A, Pi, hint, w_tab=kwargs.get("w_tab"))


def _as_oracle(A, mdl_or_ocl, Pi=None):
    if isinstance(mdl_or_ocl, StripeOracle):
        return mdl_or_ocl, False
    return StripeOracle(mdl_or_ocl, A, Pi), True


def bound_stripe(A, K, mdl_or_ocl, Pi=None):
    """``bound_stripe(A, K[, Pi], mdl-or-ocl) -> (c_lo, c_hi)`` (Costs.jl:9-19 and the per-model methods)."""
    ocl, own = _as_oracle(A, mdl_or_ocl, Pi)
    try:
        out = (ctypes.c_double * 2)()
        _check(load_library().cpb_bound_stripe(ocl._h, int(K), out))
        lo, hi = out[0], out[1]
        return (lo, hi) if ocl.model.is_float else (int(lo), int(hi))
    finally:
        if own:
            ocl.close()


def _objective(total, A, Phi, mdl_or_ocl, Pi):
    tmp = None
    if not isinstance(Phi, T.SplitPartition):
        # compute_objective for Map / DomainPartitions (Costs.jl:34-39, 52-57; WorkCosts.jl:63-81; PrimaryConnectivityCosts.jl:
        # 127-163; EnvelopeCosts.jl:100-129): gather the columns part by part, then evaluate the contiguous parts
        if isinstance(mdl_or_ocl, StripeOracle):
            raise TypeError("a non-contiguous partition needs the model, not an oracle of the unpermuted matrix")
        dom = T.convert(T.DomainPartition, Phi)
        if dom.prm.shape != (A.n,):
            raise ValueError("the partition must cover the n columns")
        tmp = A = permute(A, dom.prm, None)
        Phi = T.SplitPartition(dom.K, dom.spl)
    ocl, own = _as_oracle(A, mdl_or_ocl, Pi)
    try:
        out = ctypes.c_double()
        spl = _arr(Phi.spl)
        _check(load_library().cpb_objective(ocl._h, int(total), Phi.K, _p(spl), ctypes.byref(out)))
        return out.value if ocl.model.is_float else int(out.value)
    finally:
        if own:
            ocl.close()
        if tmp is not None:
            tmp.close()


def bottleneck_value(A, Phi, mdl, Pi=None):
    """Costs.jl:26-27: ``Phi`` a Split-, Domain- or MapPartition of the columns, ``Pi`` (for the partition-aware models) any
    partition of the rows."""
    return _objective(False, A, Phi, mdl, Pi)


def total_value(A, Phi, mdl, Pi=None):
    """Costs.jl:28-29 (same argument forms as ``bottleneck_value``)."""
    return _objective(True, A, Phi, mdl, Pi)


class _ColorArray:
    """netcount(A)[j, j'] and friends (SparseColorArrays.jl); ``.query(j, j')`` batches on the GPU."""

    def __init__(self, which, A):
        self.which = which
        self._own = _Scoped(A)
        self.dm = self._own.dm

    def query(self, j, jp) -> np.ndarray:
        j, jp = _arr(np.atleast_1d(j)), _arr(np.atleast_1d(jp))
        out = np.empty(len(j), dtype=I64)
        _check(load_library().cpb_count_query(self.dm._h, self.which, len(j), _p(j), _p(jp), _p(out)))
        return out

    def __getitem__(self, idx):
        j, jp = idx
        r = self.query(j, jp)
        return int(r[0]) if np.ndim(j) == 0 else r

    __call__ = lambda self, j, jp: self[j, jp]


def pincount(A, hint=None):
    return _ColorArray(0, A)


def netcount(A, hint=None):
    return _ColorArray(1, A)


def dianetcount(A, hint=None):
    return _ColorArray(2, A)


def selfnetcount(A, hint=None):
    return _ColorArray(3, A)


def selfpincount(A, hint=None):
    return _ColorArray(4, A)


# ------------------------------------------------------------------------------- solvers


def partition_stripe(A, K, method, Pi=None, **kwargs) -> T.SplitPartition:
    """``partition_stripe(A, K, method[, Pi]; kwargs...)`` -> ``SplitPartition(K, spl)``."""
    K = int(K)
    code, spec, eps = T.split_method_code(method)
    spl = np.empty(K + 1, dtype=I64)
    with _Scoped(A) as dm:
        if spec is None:  # EquiSplitter
            spec = T.AffineWorkModel(0, 0, 0)
        ocl = StripeOracle(spec, dm, Pi)
        try:
            if ocl.weight is not None:  # ConstrainedCost with a count weight
                _check(load_library().cpb_partition_stripe_weighted(ocl._h, code, ocl.weight._h, ocl.w_max, eps, K, _p(spl)))
            else:
                _check(load_library().cpb_partition_stripe(ocl._h, code, ctypes.byref(ocl.constraint), eps, K, _p(spl)))
        finally:
            ocl.close()
    return T.SplitPartition(K, spl)


_SCRATCH = {}


def _scratch(name: str, count: int) -> np.ndarray:
    buf = _SCRATCH.get(name)
    if buf is None or buf.size < count:
        buf = np.empty(max(count, 1024), dtype=I64)
        _SCRATCH[name] = buf
    return buf[:count]


def pack_stripe(A, method, Pi=None, n_nets=None, **kwargs) -> T.SplitPartition:
    """``pack_stripe(A, method[, Pi]; kwargs...)`` -> ``SplitPartition(K, spl)`` with a free number of chunks."""
    code, spec, rho, w_max = T.pack_method_code(method)
    if isinstance(spec, T.ConstrainedCost) and spec.count_weight() is not None:
        raise TypeError("pack_stripe takes VertexCount() or an integer AffineWorkModel as the weight: count weights "
                        "(AffineConnectivityModel / AffineMonotonizedSymmetricConnectivityModel) are not built for the chunkers")
    with _Scoped(A) as dm:
        # the ABI wants room for the worst case (n + 1 boundaries): reuse one scratch array across calls instead of
        # faulting in tens of megabytes per call
        spl = _scratch("spl", dm.n + 1)
        nn = _scratch("nn", max(dm.n, 1)) if n_nets is not None else None
        Kout = ctypes.c_int64()
        ocl = None
        con = T.CConstraint()
        if spec is not None:
            ocl = StripeOracle(spec, dm, Pi)
            con = ocl.constraint
        try:
            _check(load_library().cpb_pack_stripe(dm._h, ocl._h if ocl else None, code, ctypes.byref(con), rho, w_max, _p(spl),
                                                   ctypes.byref(Kout), _p(nn) if nn is not None else None))
        finally:
            if ocl:
                ocl.close()
    K = Kout.value
    if n_nets is not None:
        n_nets[:] = [nn[:K].copy()]
    return T.SplitPartition(K, spl[: K + 1].copy())


def partition_plaid(A, K, method, adj_A=None, **kwargs):
    """AlternatingPartitioner.jl:6-88: alternating stripe solves on ``A`` and ``adjointpattern(A)``; both
    stay resident in HBM for the whole call."""
    with _Scoped(A) as dA:
        if isinstance(method, T.SymmetricPartitioner) and len(method.mtds) == 1:
            Pi = partition_stripe(dA, K, method.mtds[0])
            return Pi, Pi
        own_adj = adj_A is None
        dT = adjointpattern(dA) if own_adj else device_matrix(adj_A)
        try:
            if isinstance(method, T.DisjointPartitioner):
                Phi = partition_stripe(dA, K, method.mtd)
                Pi = partition_stripe(dT, K, method.mtd2, Phi)
                return Pi, Phi
            if isinstance(method, T.AlternatingPartitioner):
                Phi = partition_stripe(dA, K, method.mtds[0])
                Pi = partition_stripe(dT, K, method.mtds[1], Phi)
                for i, mtd in enumerate(method.mtds[2:], start=1):
                    if i % 2 == 1:
                        Phi = partition_stripe(dA, K, mtd, Pi)
                    else:
                        Pi = partition_stripe(dT, K, mtd, Phi)
                return Pi, Phi
            if isinstance(method, T.SymmetricPartitioner):
                Pi = partition_stripe(dA, K, method.mtds[0])
                for i, mtd in enumerate(method.mtds[1:], start=1):
                    Pi = partition_stripe(dA if i % 2 == 1 else dT, K, mtd, Pi)
                return Pi, Pi
            raise TypeError(f"partition_plaid: unsupported method {type(method).__name__}")
        finally:
            if own_adj or not isinstance(adj_A, DeviceMatrix):
                dT.close()


def pack_plaid(A, method, adj_A=None, **kwargs):
    """AlternatingPacker.jl:6-53."""
    with _Scoped(A) as dA:
        own_adj = adj_A is None
        dT = adjointpattern(dA) if own_adj else device_matrix(adj_A)
        try:
            if isinstance(method, T.DisjointPacker):
                Phi = pack_stripe(dA, method.mtd)
                Pi = pack_stripe(dT, method.mtd2, Phi)
                return Pi, Phi
            if isinstance(method, T.AlternatingPacker):
                Phi = pack_stripe(dA, method.mtds[0])
                Pi = pack_stripe(dT, method.mtds[1], Phi)
                for i, mtd in enumerate(method.mtds[2:], start=1):
                    if i % 2 == 1:
                        Phi = pack_stripe(dA, mtd, Pi)
                    else:
                        Pi = pack_stripe(dT, mtd, Phi)
                return Pi, Phi
            if isinstance(method, T.SymmetricPacker):
                Pi = pack_stripe(dA, method.mtds[0])
                for i, mtd in enumerate(method.mtds[1:], start=1):
                    Pi = pack_stripe(dA if i % 2 == 1 else dT, mtd, Pi)
                return Pi, Pi
            raise TypeError(f"pack_plaid: unsupported method {type(method).__name__}")
        finally:
            if own_adj or not isinstance(adj_A, DeviceMatrix):
                dT.close()


# ------------------------------------------------------------------------------- one solve over several GPUs


class Communicator:
    """The library-owned NCCL communicator (``cpb_comm_*``): one process per GPU.  Rank 0 makes the 128-byte id with
    ``Communicator.unique_id()``, the host ships it to the other ranks (MPI bcast, a file, torch.distributed -- see
    ``parallel.library_communicator``), every rank constructs ``Communicator(id, rank, world)`` after ``init(device)``."""

    def __init__(self, uid: bytes, rank: int, world: int):
        if len(uid) != 128:
            raise ValueError("the NCCL unique id is 128 bytes")
        self.rank, self.world = int(rank), int(world)
        buf = ctypes.create_string_buffer(bytes(uid), 128)
        _check(load_library().cpb_comm_init(buf, self.rank, self.world))
        self._open = True

    @staticmethod
    def unique_id() -> bytes:
        buf = ctypes.create_string_buffer(128)
        _check(load_library().cpb_comm_unique_id(buf))
        return buf.raw

    def close(self):
        if getattr(self, "_open", False) and _lib is not None:
            _lib.cpb_comm_destroy()
        self._open = False

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def shard_range(nnz: int, rank: int, world: int):
    """0-based half-open block of CSC positions owned by ``rank`` (``cpb_shard_range``; host arithmetic only)."""
    lo, hi = ctypes.c_int64(), ctypes.c_int64()
    _check(load_library().cpb_shard_range(int(nnz), int(rank), int(world), ctypes.byref(lo), ctypes.byref(hi)))
    return lo.value, hi.value


class ShardedMatrix:
    """A pattern spread over the ranks of the communicator (``cpb_sharded``): every rank holds the column offsets and its own
    block of ``rowval``.  Collective: every rank constructs it from the same host matrix."""

    def __init__(self, A, comm: Optional[Communicator] = None):
        self.m, self.n, self.nnz = int(A.m), int(A.n), int(A.nnz)
        self.comm = comm
        self._h = ctypes.c_void_p()
        _check(load_library().cpb_sharded_matrix_create(self.m, self.n, self.nnz, _p(A.colptr), _p(A.rowval), 0, ctypes.byref(self._h)))

    @classmethod
    def _adopt(cls, h, m, n, nnz, comm):
        S = cls.__new__(cls)
        S.m, S.n, S.nnz, S.comm, S._h = int(m), int(n), int(nnz), comm, h
        return S

    def adjointpattern(self) -> "ShardedMatrix":
        """``adjointpattern`` of the sharded pattern (``cpb_sharded_adjointpattern``; collective): a ``ShardedMatrix`` of the
        transpose with the same blocks of CSC positions."""
        h = ctypes.c_void_p()
        _check(load_library().cpb_sharded_adjointpattern(self._h, ctypes.byref(h)))
        return ShardedMatrix._adopt(h, self.n, self.m, self.nnz, self.comm)

    def to_host_block(self):
        """-> ``(colptr, rowval_block, q_lo, q_hi)``: the complete 1-based column offsets, the 1-based row indices of this
        rank's CSC positions ``[q_lo, q_hi)`` (0-based, half-open, as ``shard_range``)."""
        lib = load_library()
        lo, hi = ctypes.c_int64(), ctypes.c_int64()
        _check(lib.cpb_sharded_matrix_get(self._h, None, None, ctypes.byref(lo), ctypes.byref(hi)))
        colptr = np.empty(self.n + 1, dtype=I64)
        rowval = np.empty(hi.value - lo.value, dtype=I64)
        _check(lib.cpb_sharded_matrix_get(self._h, _p(colptr), _p(rowval) if rowval.size else None, None, None))
        return colptr, rowval, lo.value, hi.value

    def close(self):
        if self._h is not None and _lib is not None:
            _lib.cpb_sharded_matrix_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _sharded_args(method):
    code, spec, eps = T.split_method_code(method)
    f, con = T.split_constrained(spec)
    if con.enabled:
        raise TypeError("sharded solves take an unconstrained AffineConnectivityModel or AffineMonotonizedSymmetricConnectivityModel")
    cm, keep = f.to_c()
    return code, cm, keep, eps


def partition_stripe_sharded(A, K, method, comm: Optional[Communicator] = None) -> T.SplitPartition:
    """``partition_stripe(A, K, BisectCost/LazyBisectCost(f, eps))`` as ONE solve over all ranks of the communicator
    (collective; every rank gets the same ``SplitPartition``), ``f`` an ``AffineConnectivityModel`` or an
    ``AffineMonotonizedSymmetricConnectivityModel`` (square ``A``).  ``A``: a ``ShardedMatrix`` (resident) or a host matrix
    (every rank uploads its block inside the call)."""
    K = int(K)
    code, cm, keep, eps = _sharded_args(method)
    own = not isinstance(A, ShardedMatrix)
    sh = ShardedMatrix(A, comm) if own else A
    try:
        spl = np.empty(K + 1, dtype=I64)
        _check(load_library().cpb_partition_stripe_sharded(sh._h, ctypes.byref(cm), code, eps, K, _p(spl)))
    finally:
        if own:
            sh.close()
    return T.SplitPartition(K, spl)


def partition_stripe_sharded_emulated(A, K, method, world: int) -> T.SplitPartition:
    """The sharded solve with ``world`` ranks played one after the other on this GPU (tests: block construction + carry
    rule + world x 15 thresholds per round, no NCCL)."""
    K = int(K)
    code, cm, keep, eps = _sharded_args(method)
    spl = np.empty(K + 1, dtype=I64)
    with _Scoped(A) as dm:
        _check(load_library().cpb_partition_stripe_sharded_emulated(dm._h, ctypes.byref(cm), code, eps, K, int(world), _p(spl)))
    return T.SplitPartition(K, spl)


def sharded_stats() -> dict:
    out = (ctypes.c_double * 16)()
    _check(load_library().cpb_sharded_stats(out))
    return {"world": int(out[0]), "host_ms_until_links_queued": out[1], "bisection_ms_incl_links_wait": out[2], "rounds": int(out[3]),
            "link_allgather_bytes": out[4], "carry_bytes_per_hop": out[5], "threshold_allgather_bytes": out[6], "thresholds_per_round": int(out[7]),
            "transpose_pair_bytes_received": out[8], "transpose_histogram_allgather_bytes": out[9],
            "limiting_collective": "in-place gather of the link array (nnz x 4 bytes on every rank; nnz of A + I for the monotonized symmetric model)"}


def adjointpattern_sharded_emulated(A, world: int):
    """``adjointpattern`` built as ``ShardedMatrix.adjointpattern`` would build it over ``world`` ranks, the ranks played one
    after the other on this GPU (tests).  Host matrix in -> host matrix out; DeviceMatrix in -> DeviceMatrix out."""
    with _Scoped(A) as dm:
        h = ctypes.c_void_p()
        _check(load_library().cpb_adjointpattern_sharded_emulated(dm._h, int(world), ctypes.byref(h)))
        out = DeviceMatrix(h, dm.n, dm.m, dm.nnz)
        if isinstance(A, DeviceMatrix):
            return out
        res = out.to_host()
        out.close()
        return res


def _plaid_sharded_methods(method):
    """The stripe methods of a plaid partitioner, each checked for the sharded solve (before any collective starts)."""
    if isinstance(method, T.DisjointPartitioner):
        mtds = [method.mtd, method.mtd2]
    elif isinstance(method, (T.AlternatingPartitioner, T.SymmetricPartitioner)):
        mtds = list(method.mtds)
    else:
        raise TypeError(f"partition_plaid_sharded: unsupported method {type(method).__name__}")
    if not mtds:
        raise TypeError("partition_plaid_sharded: no stripe methods")
    for mtd in mtds:
        code, spec, _ = T.split_method_code(mtd)
        if code not in (T.SPLIT_BISECT_COST, T.SPLIT_LAZY_BISECT_COST):
            raise TypeError(f"partition_plaid_sharded: {type(mtd).__name__} has no sharded form (BisectCost / LazyBisectCost splitters only)")
        f, con = T.split_constrained(spec)
        if con.enabled or getattr(f, "kind", None) not in (T.MODEL_CONNECTIVITY, T.MODEL_MONOSYM):
            raise TypeError("partition_plaid_sharded: the stripe methods must use an unconstrained AffineConnectivityModel or "
                            f"AffineMonotonizedSymmetricConnectivityModel, not {type(f).__name__}")
    return mtds


def _plaid_walk(method, mtds, solve, on_A, on_T):
    """partition_plaid's alternation (AlternatingPartitioner.jl:6-88) over a stripe solve ``solve(side, K, mtd)``."""
    if isinstance(method, T.DisjointPartitioner):
        Phi = solve(on_A(), mtds[0])
        return solve(on_T(), mtds[1]), Phi
    if isinstance(method, T.AlternatingPartitioner):
        Phi = solve(on_A(), mtds[0])
        Pi = solve(on_T(), mtds[1])
        for i, mtd in enumerate(mtds[2:], start=1):
            if i % 2 == 1:
                Phi = solve(on_A(), mtd)
            else:
                Pi = solve(on_T(), mtd)
        return Pi, Phi
    Pi = solve(on_A(), mtds[0])  # SymmetricPartitioner
    for i, mtd in enumerate(mtds[1:], start=1):
        Pi = solve(on_A() if i % 2 == 1 else on_T(), mtd)
    return Pi, Pi


def partition_plaid_sharded(A, K, method, comm: Optional[Communicator] = None, adj_A=None):
    """``partition_plaid(A, K, method)`` with every stripe solve sharded over the ranks of the communicator (collective; every
    rank gets the same ``(Pi, Phi)``).  ``method``: an Alternating / Symmetric / Disjoint partitioner whose stripe methods are
    BisectCost / LazyBisectCost over the connectivity or the monotonized symmetric model; anything else raises TypeError
    before any collective starts.  ``A``: a ``ShardedMatrix`` or a host matrix; ``adj_A``: the transpose as either, or None
    (built once per call with ``ShardedMatrix.adjointpattern`` and shared by the alternations, as on one GPU)."""
    K = int(K)
    mtds = _plaid_sharded_methods(method)
    own = not isinstance(A, ShardedMatrix)
    sA = ShardedMatrix(A, comm) if own else A
    held = {}

    def on_T():
        if "T" not in held:
            if adj_A is None:
                held["T"], held["own"] = sA.adjointpattern(), True
            elif isinstance(adj_A, ShardedMatrix):
                held["T"], held["own"] = adj_A, False
            else:
                held["T"], held["own"] = ShardedMatrix(adj_A, comm), True
        return held["T"]

    try:
        return _plaid_walk(method, mtds, lambda S, mtd: partition_stripe_sharded(S, K, mtd), lambda: sA, on_T)
    finally:
        if held.get("own"):
            held["T"].close()
        if own:
            sA.close()


def partition_plaid_sharded_emulated(A, K, method, world: int):
    """``partition_plaid_sharded`` with ``world`` ranks played one after the other on this GPU: the emulated sharded transpose
    and the emulated sharded stripe solves (tests)."""
    K = int(K)
    mtds = _plaid_sharded_methods(method)
    with _Scoped(A) as dA:
        held = {}

        def on_T():
            if "T" not in held:
                held["T"] = adjointpattern_sharded_emulated(dA, world)
            return held["T"]

        try:
            return _plaid_walk(method, mtds, lambda M, mtd: partition_stripe_sharded_emulated(M, K, mtd, world), lambda: dA, on_T)
        finally:
            if "T" in held:
                held["T"].close()


# ------------------------------------------------------------------------------- measurement hooks


def profile_enable(on: bool = True):
    load_library().cpb_profile_enable(int(bool(on)))


def profile_reset():
    load_library().cpb_profile_reset()


def profile_get() -> dict:
    cap = 64
    names = ctypes.create_string_buffer(32 * cap)
    ms = (ctypes.c_double * cap)()
    launches = (ctypes.c_int64 * cap)()
    nbytes = (ctypes.c_double * cap)()
    k = load_library().cpb_profile_get(cap, names, ms, launches, nbytes)
    out = {}
    for t in range(k):
        nm = names.raw[32 * t : 32 * t + 32].split(b"\0", 1)[0].decode()
        out[nm] = dict(ms=ms[t], launches=int(launches[t]), bytes=nbytes[t])
    return out


def bisect_plan(c_lo: float, c_hi: float, eps: float, nodes: int, c_lo0: float = None, c_hi0: float = None, upper_bound: float = 0.0):
    """Heap indices of the bisection-tree nodes one round probes concurrently (``cpb_bisect_plan``; host-only)."""
    ids = (ctypes.c_int32 * nodes)()
    lib = load_library()
    lib.cpb_bisect_plan.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_void_p]
    _check(lib.cpb_bisect_plan(c_lo, c_hi, eps, nodes, c_lo if c_lo0 is None else c_lo0, c_hi if c_hi0 is None else c_hi0, upper_bound, ids))
    return [int(x) for x in ids]


def bisect_prewalk(c_lo: float, c_hi: float, eps: float, upper_bound: float):
    """-> (c_hi after the probes the bound settles, their number) (``cpb_bisect_prewalk``; host-only)."""
    out = ctypes.c_double()
    n = ctypes.c_int32()
    lib = load_library()
    lib.cpb_bisect_prewalk.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32)]
    _check(lib.cpb_bisect_prewalk(c_lo, c_hi, eps, upper_bound, ctypes.byref(out), ctypes.byref(n)))
    return out.value, n.value


def bisect_stats() -> dict:
    """Diagnostics of the most recent bisection (``cpb_bisect_stats``)."""
    out = (ctypes.c_double * 8)()
    _check(load_library().cpb_bisect_stats(out))
    return {"rounds": int(out[0]), "probes": int(out[1]), "speculated": int(out[2]), "c_lo": out[3], "c_hi": out[4], "plan_upper_bound": out[5],
            "c_lo_final": out[6], "c_hi_final": out[7]}


def launch_count() -> int:
    return int(load_library().cpb_launch_count())


def trim_memory():
    """Gives the device memory cached between calls back to the driver (handles stay valid)."""
    _check(load_library().cpb_trim_memory())


def timer_start():
    """CUDA event on the library stream (device-side stopwatch for bench.py)."""
    _check(load_library().cpb_timer_start())


def timer_stop() -> float:
    ms = ctypes.c_double()
    _check(load_library().cpb_timer_stop(ctypes.byref(ms)))
    return ms.value
