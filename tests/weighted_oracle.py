"""ctypes binding of tests/weighted_oracle.cpp -- TEST INFRASTRUCTURE ONLY.

``partition_stripe(A, K, method)`` for ``ConstrainedCost(f, w, w_max)`` with a count weight ``w`` (an integer
``AffineConnectivityModel`` / ``AffineMonotonizedSymmetricConnectivityModel``): the CPU oracle's restated constrained
splitters with ``w`` evaluated by its own step oracle.  Every other method goes to ``pyoracle.partition_stripe`` unchanged.

The library is compiled with g++ on first use into ``build_weighted_oracle/`` next to this directory's parent, or into a
temporary directory when the tree is read-only.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import sys
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
for _p in (_ROOT, os.path.join(_ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import pyoracle as ref  # noqa: E402
from chainb200 import types as T  # noqa: E402

_SRC = os.path.join(_HERE, "weighted_oracle.cpp")
_DEPS = [_SRC] + [os.path.join(_ROOT, "oracle", f) for f in ("cpo_core.hpp", "cpo_solvers.hpp", "cpo.h")]
# the flags of oracle/Makefile (-ffp-contract=off: Julia evaluates a + b*c without FMA contraction)
_CXXFLAGS = ["-O3", "-march=x86-64-v2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall", "-Wno-unused-function", "-shared"]
_lib = None
last_seconds = [0.0, 0.0]


def _fresh(path: str) -> bool:
    return os.path.exists(path) and all(os.path.getmtime(d) <= os.path.getmtime(path) for d in _DEPS)


def build() -> str:
    """Compile the library (if it is missing or older than its sources); returns its path."""
    path = os.path.join(_ROOT, "build_weighted_oracle", "libcpo_weighted.so")
    if _fresh(path):
        return path
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        probe = os.path.join(os.path.dirname(path), ".w")
        open(probe, "w").close()
        os.remove(probe)
    except OSError:  # read-only tree
        path = os.path.join(tempfile.mkdtemp(prefix="cpo_weighted_"), "libcpo_weighted.so")
    tmp = path + f".{os.getpid()}.tmp"
    subprocess.check_call(["g++", *_CXXFLAGS, "-o", tmp, _SRC])
    os.replace(tmp, path)
    return path


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
        _lib.cpw_last_error.restype = ctypes.c_char_p
    return _lib


def is_count_weighted(spec) -> bool:
    return isinstance(spec, T.ConstrainedCost) and spec.count_weight() is not None


def partition_stripe(A, K, method, Pi=None, **kwargs) -> T.SplitPartition:
    """``pyoracle.partition_stripe``, extended to count weights."""
    code, spec, eps = T.split_method_code(method)
    if not is_count_weighted(spec):
        return ref.partition_stripe(A, K, method, Pi, **kwargs)
    spl = np.empty(K + 1, dtype=np.int64)
    secs = (ctypes.c_double * 2)()
    pspl, pK = ref._pi(Pi)
    cm, keep = ref._model(spec.f, A, T.CConstraint(), Pi)
    wm, wkeep = spec.w.to_c()
    rc = lib().cpw_partition_stripe_weighted(code, ctypes.byref(cm), ctypes.byref(wm), ctypes.c_longlong(int(spec.w_max)),
                                             ctypes.byref(ref._csc(A)), ref._ptr(pspl), ctypes.c_longlong(pK), ctypes.c_longlong(K),
                                             ref._ptr(spl), secs)
    if rc != 0:
        raise RuntimeError("weighted oracle: " + lib().cpw_last_error().decode())
    last_seconds[:] = [secs[0], secs[1]]
    return T.SplitPartition(K, spl)


def partition_plaid(A, K, method, adj_A=None, **kwargs):
    """``pyoracle.partition_plaid``'s alternation (AlternatingPartitioner.jl:6-88) with this module's stripe solve."""
    if adj_A is None:
        adj_A = ref.adjointpattern(A)
    if isinstance(method, T.SymmetricPartitioner):
        if len(method.mtds) == 1:
            Pi = partition_stripe(A, K, method.mtds[0])
            return Pi, Pi
        Pi = partition_stripe(A, K, method.mtds[0])
        for i, mtd in enumerate(method.mtds[1:], start=1):
            Pi = partition_stripe(A if i % 2 == 1 else adj_A, K, mtd, Pi)
        return Pi, Pi
    if isinstance(method, T.AlternatingPartitioner):
        Phi = partition_stripe(A, K, method.mtds[0])
        Pi = partition_stripe(adj_A, K, method.mtds[1], Phi)
        for i, mtd in enumerate(method.mtds[2:], start=1):
            if i % 2 == 1:
                Phi = partition_stripe(A, K, mtd, Pi)
            else:
                Pi = partition_stripe(adj_A, K, mtd, Phi)
        return Pi, Phi
    raise TypeError(f"partition_plaid: unsupported method {type(method).__name__}")
