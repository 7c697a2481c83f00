"""A second, independent statement of the count-weight path -- TEST INFRASTRUCTURE ONLY.

Transliterated as literally as Python allows (file:line of the reference's src/), next to oracle/pywitness.py and with its
conventions (1-based lists, index 0 unused; the cost oracle reduced to its definition):
  DynamicSplitter.jl:144-173   column_constraints
  DynamicSplitter.jl:206-247   partition_stripe(::AbstractDynamicSplitter{<:ConstrainedCost})
driven by a set-based weight (SetWeight: distinct rows counted with a Python set), so it shares no code and no data structure
with the C++ oracle's weight oracle.  tests/test_weight_constraints.py fuzzes the two against each other.
"""
from __future__ import annotations

import math

from pywitness import Conn, unravel_splits  # noqa: F401  (Conn: the cost oracle the witness DP takes)


class SetWeight:
    """The weight of ConstrainedCost(f, w, w_max) (Costs.jl:105-147) for w an integer AffineWorkModel(a, b_v, b_p),
    AffineConnectivityModel(a, b_v, b_p, b_net) or AffineMonotonizedSymmetricConnectivityModel(a, b_v, b_over_pin,
    b_dia_net, delta_pins), evaluated from its definition: pins and over-pins summed column by column, nets and dia-nets
    counted with a set (a dia-net is a row of A + I)."""

    def __init__(self, A, kind, coef):
        self.pos = [0] + [int(x) for x in A.colptr]
        self.idx = [0] + [int(x) for x in A.rowval]
        self.kind, self.coef = kind, tuple(coef)

    def __call__(self, j, jp):
        c = self.coef
        nv = jp - j
        if self.kind == "work":
            return c[0] + nv * c[1] + (self.pos[jp] - self.pos[j]) * c[2]
        rows = set()
        for q in range(self.pos[j], self.pos[jp]):
            rows.add(self.idx[q])
        if self.kind == "conn":
            return c[0] + nv * c[1] + (self.pos[jp] - self.pos[j]) * c[2] + len(rows) * c[3]
        over = 0
        for col in range(j, jp):
            over += max(self.pos[col + 1] - self.pos[col] - c[4], 0)
            rows.add(col)
        return c[0] + nv * c[1] + over * c[2] + len(rows) * c[3]


def column_constraints(n, K, w, w_max):  # DynamicSplitter.jl:144-173 -> (j'_lo, j'_hi), 1-based lists
    jp_lo = [0] * (K + 1)
    jp_hi = [0] * (K + 1)
    jp = n + 1
    for k in range(K, 0, -1):
        jp_lo[k] = jp
        j = jp
        while j - 1 >= 1 and w(j - 1, jp) <= w_max:
            j -= 1
        jp = j
    j = 1
    for k in range(1, K + 1):
        jp = j
        while jp + 1 <= n + 1 and w(j, jp + 1) <= w_max:
            jp += 1
        jp_hi[k] = jp
        j = jp
    return jp_lo, jp_hi


def dynamic_splitter_constrained(f: Conn, K, total: bool, w, w_max):  # DynamicSplitter.jl:206-247
    """The window-constrained DP: column k of cst / ptr holds only rows j'_lo[k]..j'_hi[k] (WindowConstrainedMatrix,
    :101-142): reads outside give typemax / 0, writes outside are dropped."""
    n = f.n
    g = (lambda a, b: a + b) if total else max
    jp_lo, jp_hi = column_constraints(n, K, w, w_max)
    if jp_hi[K] < n + 1:  # :217-222
        return [1] * K + [n + 1]
    cst = [[math.inf] * (n + 2) for _ in range(K + 1)]
    ptr = [[0] * (n + 2) for _ in range(K + 1)]

    def get(M, k, jp, z):
        return M[k][jp] if jp_lo[k] <= jp <= jp_hi[k] else z

    def put(M, k, jp, v):
        if jp_lo[k] <= jp <= jp_hi[k]:
            M[k][jp] = v

    for jp in range(jp_lo[1], jp_hi[1] + 1):
        put(cst, 1, jp, f(1, jp, 1))
        put(ptr, 1, jp, 1)
    for k in range(2, K + 1):
        j0 = jp_lo[k - 1]
        for jp in range(jp_lo[k], jp_hi[k] + 1):
            while w(j0, jp) > w_max:
                j0 += 1
            put(cst, k, jp, g(get(cst, k - 1, j0, math.inf), f(j0, jp, k)))
            put(ptr, k, jp, j0)
            for j in range(j0 + 1, min(jp, jp_hi[k - 1]) + 1):
                c2 = g(get(cst, k - 1, j, math.inf), f(j, jp, k))
                if c2 <= get(cst, k, jp, math.inf):
                    put(cst, k, jp, c2)
                    put(ptr, k, jp, j)
    ptr_k = [[get(ptr, k, jp, 0) for jp in range(n + 2)] for k in range(K + 1)]
    return unravel_splits(K, n, ptr_k)
