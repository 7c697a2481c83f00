"""Kernel forms that the parity suite would otherwise never launch (-m gpu): every chunk-DP window template (8/16/32/64
columns, warp and thread-per-block forms, several staged chunks), the one-sweep radix sort at every pass count, digit mix,
tile edge and link-construction route, and the environment switches that select between forms which must give identical
results.  Each check compares with an independent reference exactly: split vectors, K, n_nets, integer counts and patterns
(scipy's transpose for adjointpattern, the CPU oracle for everything else)."""
import ctypes
import functools
import json
import os

import numpy as np
import pytest

import chainb200 as cp
from chainb200 import synth

pytestmark = pytest.mark.gpu

AFF = cp.AffineConnectivityModel(0, 10, 1, 100)
SYM = cp.AffineMonotonizedSymmetricConnectivityModel(0, 0, 1, 100, 4)
TILE = 4096  # pairs per one-sweep tile (OS_TILE in onesweep.cu)

LINK_SWITCHES = ("CPB_NO_ROW_SEGMENTS", "CPB_WINDOWED_SCATTER_MIN", "CPB_CHUNK_THREAD_BLOCKS")


def set_env(monkeypatch, env):
    """Exactly the switches in `env` set; the other link / chunk switches unset."""
    for k in LINK_SWITCHES:
        if k not in env:
            monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def profiled(fn):
    """fn() with the library's phase profile on; -> (result, {phase: {ms, launches, bytes}})."""
    cp.profile_enable(True)
    cp.profile_reset()
    try:
        out = fn()
        return out, cp.profile_get()
    finally:
        cp.profile_enable(False)
        cp.profile_reset()


def launches(prof, phase):
    return prof.get(phase, {}).get("launches", 0)


def os_passes(m):
    """8-bit passes of the one-sweep sort over the row indices 0..m-1."""
    return max(1, -(-int(m - 1).bit_length() // 8))


# ------------------------------------------------------------------------------------------ chunk DP at every window template
WIDTHS = [16, 17, 31, 32, 33, 63, 64]


def runs_matrix(rng, m, n):
    """Columns in runs (lengths 1..100) that share a base row set -- half of the runs identical columns, the others with
    columns that differ in one row -- and a fresh base set at every run boundary: chunks reach w_max, and the DP has both
    strict optima and ties."""
    I, J = [], []
    j = 0
    while j < n:
        L = min(int(rng.integers(1, 101)), n - j)
        base = rng.choice(m, int(rng.integers(2, 7)), replace=False)
        same = rng.random() < 0.5
        for c in range(j, j + L):
            rows = base if same or rng.random() < 0.6 else np.append(base[1:], rng.integers(0, m))
            I.append(rows)
            J.append(np.full(len(rows), c))
        j += L
    return cp.SparseMatrixCSC.from_coo(m, n, np.concatenate(I) + 1, np.concatenate(J) + 1)


@functools.lru_cache(maxsize=None)
def chunk_matrix(n):
    return runs_matrix(np.random.default_rng(7000 + n), 400 if n < 4096 else 4000, n)


CHUNK_MODELS = [
    ("conn-int", cp.AffineConnectivityModel(0, 3, 1, 3)),
    ("nets-int", cp.AffineConnectivityModel(0, 0, 0, 1)),
    ("conn-f64", cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0)),  # k_chunk_seq_f64
    ("work", cp.AffineWorkModel(1, 2, 3)),  # every chunking of the same count costs the same: the leftmost-tie rule decides
    ("colblock", cp.ColumnBlockComponentCostModel(int, 3, lambda w: 1 + w)),
    ("block-R1", cp.BlockComponentCostModel(int, 1, 3, (1,), (cp.identity,))),
    ("block-R2", cp.BlockComponentCostModel(int, 0, 0, (10, cp.identity), (2, lambda x: 2 * x))),
    ("block-R4", cp.BlockComponentCostModel(int, 1, cp.identity, (1, cp.identity, 2, lambda x: x + 1), (cp.identity, 1, lambda x: 2 * x, 3))),
]


def row_partition(ref, A):
    return ref.pack_stripe(ref.adjointpattern(A), cp.EquiChunker(2))


def check_pack(ref, monkeypatch, dA, A, mtd, Pi, tag):
    """pack_stripe on the device == the oracle; every window of <= 32 columns also through the thread-per-block kernels."""
    args = (Pi,) if Pi is not None else ()
    r = ref.pack_stripe(A, mtd, *args)
    forms = [{}]
    spec = getattr(mtd, "f", None)
    a, bv = (spec.w.coef[0], spec.w.coef[1]) if hasattr(spec.w, "coef") else (0, 1)
    W = min(A.n, (spec.w_max - a) // bv)  # the device's window: the weight's vertex term alone
    if W <= 32:
        forms.append({"CPB_CHUNK_THREAD_BLOCKS": "1"})
    for env in forms:
        set_env(monkeypatch, env)
        g = cp.pack_stripe(dA, mtd, *args)
        assert g.K == r.K and np.array_equal(g.spl, r.spl), (tag, env, g.K, r.K)
    set_env(monkeypatch, {})


@pytest.mark.parametrize("name,f", CHUNK_MODELS, ids=[c[0] for c in CHUNK_MODELS])
def test_chunk_dp_window_templates(ref, monkeypatch, name, f):
    """DynamicTotalChunker and ConvexTotalChunker under ConstrainedCost(f, VertexCount(), w_max) on both sides of every
    template edge (W = 16 | 17, 32 | 33, 64), at n = 1, n = w_max - 1 (the window is the whole matrix), the 1024-column DP
    block edge (1023, 1024, 1025) and a partial last block (1535)."""
    for n in (1, 1023, 1024, 1025, 1535, None):
        for w_max in WIDTHS:
            A = chunk_matrix(n if n is not None else w_max - 1)
            Pi = row_partition(ref, A) if f.kind == cp.MODEL_BLOCK else None
            dA = cp.device_matrix(A)
            for mk in (cp.DynamicTotalChunker, cp.ConvexTotalChunker):
                if mk is cp.ConvexTotalChunker and f.kind not in (cp.MODEL_CONNECTIVITY, cp.MODEL_WORK):
                    continue
                check_pack(ref, monkeypatch, dA, A, mk(cp.ConstrainedCost(f, cp.VertexCount(), w_max)), Pi, (name, A.n, w_max, mk.__name__))
            dA.close()


def test_chunk_dp_many_blocks_every_template(ref, monkeypatch):
    """n = 2^17 columns = 128 DP blocks: the warp combine stages several chunks of transfer matrices (2 blocks per chunk at
    W = 32, 8 at W = 17), the thread-per-block combine walks 128 blocks, the chain unravel crosses 256 blocks of 512 nodes."""
    A = chunk_matrix(1 << 17)
    dA = cp.device_matrix(A)
    Pi = row_partition(ref, A)
    blk = dict(CHUNK_MODELS)["block-R2"]
    for w_max in WIDTHS:
        for f in (cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineWorkModel(1, 2, 3)):
            for mk in (cp.DynamicTotalChunker, cp.ConvexTotalChunker):
                check_pack(ref, monkeypatch, dA, A, mk(cp.ConstrainedCost(f, cp.VertexCount(), w_max)), None, (A.n, f, w_max, mk.__name__))
        check_pack(ref, monkeypatch, dA, A, cp.DynamicTotalChunker(cp.ConstrainedCost(blk, cp.VertexCount(), w_max)), Pi, (A.n, "block", w_max))
    f64 = cp.DynamicTotalChunker(cp.ConstrainedCost(cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0), cp.VertexCount(), 33))
    check_pack(ref, monkeypatch, dA, A, f64, None, (A.n, "f64", 33))
    dA.close()


def test_chunk_dp_weighted_windows(ref, monkeypatch):
    """W comes from the weight's vertex term: AffineWorkModel(0, 1, 1) with w_max = 64 runs the 64-column template while
    the pin term admits far narrower windows; AffineWorkModel(0, 2, 0) with w_max = 128 is W = 64 exactly.  The convex
    pointer rule's windows follow the pin-weighted reach from window end to window end, not a fixed width W (the device
    used fixed windows here until this test: at n = 1025 it returned 89 chunks where the reference returns 87)."""
    for n in (1025, 1 << 17):
        A = chunk_matrix(n)
        dA = cp.device_matrix(A)
        for w, w_max in ((cp.AffineWorkModel(0, 1, 1), 64), (cp.AffineWorkModel(0, 2, 0), 128), (cp.AffineWorkModel(0, 2, 0), 64),
                         (cp.AffineWorkModel(2, 1, 2), 40)):
            for f in (cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineConnectivityModel(0, 0, 0, 1), cp.AffineConnectivityModel(0.5, 0.25, 1.5, 3.0)):
                for mk in (cp.DynamicTotalChunker, cp.ConvexTotalChunker):
                    check_pack(ref, monkeypatch, dA, A, mk(cp.ConstrainedCost(f, w, w_max)), None, (n, w_max, mk.__name__))
        dA.close()


def test_chunk_overlap_strict_wide(ref):
    """OverlapChunker(rho, w_max) (with n_nets) and StrictChunker(w_max) up to the device's limit of 64 columns, on runs of
    identical and overlapping columns long enough that chunks reach w_max."""
    for n in (1, 1025, 1 << 17):
        A = chunk_matrix(n)
        dA = cp.device_matrix(A)
        for w_max in WIDTHS:
            for rho in (0.9, 0.5, 0.2):
                bg, br = [None], [None]
                g = cp.pack_stripe(dA, cp.OverlapChunker(rho, w_max), n_nets=bg)
                r = ref.pack_stripe(A, cp.OverlapChunker(rho, w_max), n_nets=br)
                assert g.K == r.K and np.array_equal(g.spl, r.spl), (n, rho, w_max)
                assert np.array_equal(bg[0], br[0]), (n, rho, w_max)
            g, r = cp.pack_stripe(dA, cp.StrictChunker(w_max)), ref.pack_stripe(A, cp.StrictChunker(w_max))
            assert g.K == r.K and np.array_equal(g.spl, r.spl), (n, w_max)
            if n > 1:
                assert np.diff(g.spl).max() == w_max  # the runs are long enough for the widest chunk
        dA.close()


def test_chunk_window_wider_than_64_is_refused():
    A = chunk_matrix(1025)
    f = cp.AffineConnectivityModel(0, 3, 1, 3)
    for spec in (cp.ConstrainedCost(f, cp.VertexCount(), 65), cp.ConstrainedCost(f, cp.AffineWorkModel(0, 2, 0), 130)):
        for mk in (cp.DynamicTotalChunker, cp.ConvexTotalChunker):
            with pytest.raises(cp.CpbError):
                cp.pack_stripe(A, mk(spec))
    for mtd in (cp.OverlapChunker(0.5, 65), cp.StrictChunker(65)):
        with pytest.raises(cp.CpbError):
            cp.pack_stripe(A, mtd)


# ------------------------------------------------------------------------------------------ one-sweep sort and link construction
def exact_pattern(rng, m, n, N, rows):
    """A pattern with exactly N nonzeros: rows drawn by rows(k) (0-based), columns uniform, duplicates redrawn."""
    keys = np.zeros(0, dtype=np.int64)
    while len(keys) < N:
        k = 2 * (N - len(keys)) + 16
        keys = np.union1d(keys, rows(k).astype(np.int64) * n + rng.integers(0, n, k))
    keys = rng.choice(keys, N, replace=False)
    return cp.SparseMatrixCSC.from_coo(m, n, keys // n + 1, keys % n + 1)


def digit_rows(rng, m, mix):
    if mix == "uniform":  # every pass ranks through the shared-memory masks
        return lambda k: rng.integers(0, m, k)
    if mix == "heavy":  # one row holds 1/8 of the nonzeros: its digit is hot (MATCH.ANY) in every pass
        return lambda k: np.where(rng.random(k) < 0.125, m - 1, rng.integers(0, m, k))
    if mix == "low":  # rows 0..255 only: pass 0 uniform, every higher digit is 0 (hot)
        return lambda k: rng.integers(0, min(m, 256), k)
    raise ValueError(mix)


# name -> (m, n, N, digit mix); N on and next to the 4096-pair tile edges, pass counts 1..4
LINK_CASES = {
    "m200-uniform-N4096": (200, 1024, 4096, "uniform"),
    "m256-heavy-N4097": (256, 2048, 4097, "heavy"),
    "m257-uniform-N4095": (257, 257, 4095, "uniform"),
    "m257-low-N12288": (257, 257, 3 * TILE, "low"),
    "m65536-low-N12288": (65536, 65536, 3 * TILE, "low"),
    "m65537-uniform-N12288": (65537, 4096, 3 * TILE, "uniform"),
    "m65537-heavy-N4097": (65537, 4096, 4097, "heavy"),
    "m2^24-heavy": (1 << 24, 1 << 16, 1 << 18, "heavy"),
    "m2^24+1-uniform": ((1 << 24) + 1, 1 << 14, 1 << 18, "uniform"),
    "m2^24+1-low": ((1 << 24) + 1, 1 << 14, 1 << 18, "low"),
    "m2^24+1-heavy": ((1 << 24) + 1, 1 << 16, 1 << 18, "heavy"),
    "m300-N1": (300, 50, 1, "uniform"),
    "m300-N2": (300, 50, 2, "uniform"),
    "m300-N255": (300, 50, 255, "uniform"),
    "m300-N256": (300, 50, 256, "uniform"),
    "m300-N257": (300, 50, 257, "uniform"),
    "m2^20-N2^22+3": (1 << 20, 1 << 18, (1 << 22) + 3, "uniform"),  # 1025 tiles: long look-back chains
}


def degree_matrix(rng, n, deg, with_diag):
    """Square n x n, light rows (<= a handful of nonzeros) plus row 7 with exactly `deg` nonzeros; with_diag = False leaves
    (7, 7) out, so A + I holds deg + 1 in that row."""
    keys = np.unique(rng.integers(0, n, 2 * n) * n + rng.integers(0, n, 2 * n))
    keys = keys[keys // n != 7]
    cols = rng.choice(np.setdiff1d(np.arange(n), [7]), deg - 1 if with_diag else deg, replace=False)
    if with_diag:
        cols = np.append(cols, 7)
    keys = np.concatenate([keys, 7 * n + cols])
    A = cp.SparseMatrixCSC.from_coo(n, n, keys // n + 1, keys % n + 1)
    assert int(np.sum(A.rowval == 8)) == deg
    return A


DEGREE_CASES = {"row128": (128, True), "row128-dia129": (128, False), "row129": (129, True)}


@functools.lru_cache(maxsize=None)
def link_input(name):
    rng = np.random.default_rng(sum(map(ord, name)))
    if name in DEGREE_CASES:
        return degree_matrix(rng, 3000, *DEGREE_CASES[name])
    m, n, N, mix = LINK_CASES[name]
    A = exact_pattern(rng, m, n, N, digit_rows(rng, m, mix))
    assert A.nnz == N
    return A


def query_pairs(A, rng):
    """Random pairs, (1, n + 1), and the single columns around every tile boundary of the CSC positions."""
    n = A.n
    j = rng.integers(1, n + 2, 300)
    jp = rng.integers(1, n + 2, 300)
    j, jp = list(np.minimum(j, jp)), list(np.maximum(j, jp))
    j.append(1)
    jp.append(n + 1)
    for b in range(TILE, A.nnz + 1, TILE):
        c = int(np.searchsorted(A.colptr - 1, b, side="right"))  # 1-based column of 0-based position b
        for a in (c - 1, c, c + 1):
            if 1 <= a <= n:
                j.append(a)
                jp.append(a + 1)
    return np.array(j, dtype=np.int64), np.array(jp, dtype=np.int64)


LINK_CONFIGS = [{}, {"CPB_NO_ROW_SEGMENTS": "1"}, {"CPB_NO_ROW_SEGMENTS": "1", "CPB_WINDOWED_SCATTER_MIN": "1"}]


def scipy_transpose(A):
    S = A.to_scipy().T.tocsc()
    S.sort_indices()
    return S


@pytest.mark.parametrize("name", list(LINK_CASES) + list(DEGREE_CASES))
def test_adjointpattern_row_sort(ref, monkeypatch, name):
    """adjointpattern is a direct readout of the stable row sort: equal to scipy's transpose and to the oracle, and the
    one-sweep sort runs exactly ceil(bits(m - 1) / 8) passes."""
    A = link_input(name)
    S = scipy_transpose(A)
    R = ref.adjointpattern(A)
    assert np.array_equal(R.colptr - 1, S.indptr) and np.array_equal(R.rowval - 1, S.indices)
    set_env(monkeypatch, {})
    g, prof = profiled(lambda: cp.adjointpattern(A))
    assert (g.m, g.n) == (A.n, A.m)
    assert np.array_equal(g.colptr - 1, S.indptr) and np.array_equal(g.rowval - 1, S.indices), name
    assert launches(prof, "k_os_pass") == os_passes(A.m), (name, prof.get("k_os_pass"))


@pytest.mark.parametrize("name", list(LINK_CASES) + list(DEGREE_CASES))
def test_link_construction_forms(ref, monkeypatch, name):
    """netcount / dianetcount / selfnetcount queries and the streaming bisections against the oracle under every link
    construction route: row segments (immediate degree check in the counts, deferred in LazyBisect), the one-sweep sort
    with the direct scatter and with the windowed MODE-2 pass.  selfnetcount sorts the rows with the same passes."""
    A = link_input(name)
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    j, jp = query_pairs(A, rng)
    square = A.m == A.n
    want = {"net": ref.netcount(A, j, jp), "selfnet": ref.selfnetcount(A, j, jp)}
    if square:
        want["dianet"] = ref.dianetcount(A, j, jp)
    K = min(8, A.n)
    mtds = [cp.LazyBisectCostBottleneckSplitter(AFF, 0.01), cp.BisectCostBottleneckSplitter(AFF, 0.01)]
    if square:
        mtds.append(cp.LazyBisectCostBottleneckSplitter(SYM, 0.1))
    want_spl = [ref.partition_stripe(A, K, mtd).spl for mtd in mtds]
    for env in LINK_CONFIGS:
        set_env(monkeypatch, env)
        got, prof = profiled(lambda: cp.netcount(A).query(j, jp))
        assert np.array_equal(got, want["net"]), (name, env)
        if env.get("CPB_NO_ROW_SEGMENTS"):
            assert launches(prof, "k_os_pass") == os_passes(A.m), (name, env, prof.get("k_os_pass"))
        got, prof = profiled(lambda: cp.selfnetcount(A).query(j, jp))
        assert np.array_equal(got, want["selfnet"]), (name, env)
        assert launches(prof, "k_os_pass") == os_passes(A.m), (name, env, prof.get("k_os_pass"))
        if square:
            assert np.array_equal(cp.dianetcount(A).query(j, jp), want["dianet"]), (name, env)
        for mtd, spl in zip(mtds, want_spl):
            assert np.array_equal(cp.partition_stripe(A, K, mtd).spl, spl), (name, env, type(mtd).__name__)
    set_env(monkeypatch, {})


def test_row_degree_cache_on_a_resident_matrix(ref, monkeypatch):
    """A resident matrix remembers its heaviest row: the first solve finds the 129-nonzero row (deferred check, the
    row-segment kernels stand down), the second goes straight to the sort (known_heavy) -- same answers both times."""
    set_env(monkeypatch, {})
    A = link_input("row129")
    rng = np.random.default_rng(12)
    j, jp = query_pairs(A, rng)
    for mtd in (cp.LazyBisectCostBottleneckSplitter(AFF, 0.01), cp.LazyBisectCostBottleneckSplitter(SYM, 0.1)):
        exp = ref.partition_stripe(A, 8, mtd).spl
        dA = cp.device_matrix(A)
        for _ in range(2):
            assert np.array_equal(cp.partition_stripe(dA, 8, mtd).spl, exp)
        for _ in range(2):
            assert np.array_equal(cp.netcount(dA).query(j, jp), ref.netcount(A, j, jp))
            assert np.array_equal(cp.dianetcount(dA).query(j, jp), ref.dianetcount(A, j, jp))
        dA.close()


@pytest.mark.parametrize("heavy_in_prefix", [True, False], ids=["heavy-in-prefix", "heavy-after-prefix"])
def test_row_degree_prefix_count(ref, monkeypatch, heavy_in_prefix):
    """N >= 2^25: the immediate degree check counts a 1/16 prefix of the positions first.  A 200-nonzero row inside that
    prefix sends the construction to the sort at once; one that only the full count finds takes the count of the rest and
    then the sort (the profile's k_lt_count bytes show how much was counted).  The row-segment fill never runs in either
    case, and the counts equal the oracle's."""
    set_env(monkeypatch, {})
    rng = np.random.default_rng(25 + heavy_in_prefix)
    m, n, d = 1 << 22, 1 << 20, 32
    N = n * d  # = 2^25
    # light rows, about 8 nonzeros each: entry k of every column lies in the k-th of d bands of rows (distinct and sorted)
    R = (np.arange(d, dtype=np.int64) * (m // d))[None, :] + rng.integers(0, m // d, (n, d))
    R[R[:, 0] == 5, 0] = 4
    lo, hi = (0, n // 32) if heavy_in_prefix else (n // 2, n)
    heavy = rng.choice(np.arange(lo, hi), 200, replace=False)
    R[heavy, 0] = 5  # row 6 (1-based): 200 nonzeros
    A = cp.SparseMatrixCSC(m, n, 1 + d * np.arange(n + 1, dtype=np.int64), R.ravel() + 1)
    assert A.nnz == N and int(np.sum(A.rowval == 6)) == 200 and np.bincount(A.rowval).max() == 200
    pos6 = np.flatnonzero(A.rowval == 6)
    assert (pos6.min() < N // 16) == heavy_in_prefix and (pos6.max() < N // 16) == heavy_in_prefix
    j = rng.integers(1, n + 2, 400)
    jp = np.minimum(j + rng.integers(0, 5000, 400), n + 1)
    hc = heavy[:50] + 1  # single columns holding the heavy row
    j, jp = np.concatenate([j, hc, [1]]), np.concatenate([jp, hc + 1, [n + 1]])
    dA = cp.device_matrix(A)
    got, prof = profiled(lambda: cp.netcount(dA).query(j, jp))
    counted = N // 16 if heavy_in_prefix else N  # rows counted before the construction turned to the sort
    assert prof["k_lt_count"]["bytes"] == 4 * counted, prof["k_lt_count"]
    assert launches(prof, "k_lt_fill") == 0 and launches(prof, "k_os_pass") == os_passes(m)
    assert np.array_equal(got, ref.netcount(A, j, jp))
    dA.close()


@pytest.mark.parametrize("name", ["m2^24+1-uniform", "m65537-uniform-N12288", "m257-low-N12288"])
def test_sharded_link_blocks(ref, monkeypatch, name):
    """The sharded construction sorts each rank's block of positions with the same passes: 4-pass and tile-edge inputs at
    worlds 2 and 3."""
    A = link_input(name)
    mtd = cp.LazyBisectCostBottleneckSplitter(AFF, 0.01)
    exp = ref.partition_stripe(A, 8, mtd).spl
    set_env(monkeypatch, {})
    for world in (2, 3):
        assert np.array_equal(cp.partition_stripe_sharded_emulated(A, 8, mtd, world).spl, exp), (name, world)


@pytest.mark.skipif(os.environ.get("CPB_SKIP_FULL_SIZE") == "1", reason="CPB_SKIP_FULL_SIZE=1")
def test_row_sort_above_2_30_nonzeros(monkeypatch):
    """m = n = 2^22 with 257 nonzeros per column, entry k of every column in the k-th band of rows (distinct and sorted,
    about 257 per row: every row is too heavy for the row segments): 1.08e9 nonzeros, above the 2^30 that a 30-bit
    look-back word could count.  The row sort runs 3 one-sweep passes and the windowed MODE-2 pass.  The pattern is built
    on the device; adjointpattern must equal torch's stable sort by row, netcount the distinct rows of each column range
    counted from that sort."""
    import torch

    set_env(monkeypatch, {})
    dev = "cuda"
    m = n = 1 << 22
    d = 257
    band = m // d
    N = n * d
    assert N > 1 << 30
    gen = torch.Generator(device=dev).manual_seed(30)
    rows = (torch.arange(d, dtype=torch.int32, device=dev) * band).repeat(n)  # 0-based, CSC order: column q // d
    rows += torch.randint(0, band, (N,), dtype=torch.int32, device=dev, generator=gen)
    rowval = rows.to(torch.int64) + 1
    colptr = torch.arange(n + 1, dtype=torch.int64, device=dev) * d + 1
    torch.cuda.synchronize()
    h = ctypes.c_void_p()
    cp.api._check(cp.load_library().cpb_matrix_create_device(m, n, N, colptr.data_ptr(), rowval.data_ptr(), ctypes.byref(h)))
    dA = cp.api.DeviceMatrix(h, m, n, N)
    del rowval, colptr

    sr, perm = torch.sort(rows, stable=True)
    del rows
    B, prof = profiled(lambda: cp.adjointpattern(dA))
    assert launches(prof, "k_os_pass") == os_passes(m), prof.get("k_os_pass")
    Bh = B.to_host()
    B.close()
    exp_colptr = torch.zeros(m + 1, dtype=torch.int64, device=dev)
    exp_colptr[1:] = torch.cumsum(torch.bincount(sr, minlength=m), 0)
    assert torch.equal(torch.from_numpy(Bh.colptr).to(dev) - 1, exp_colptr)
    got = torch.from_numpy(Bh.rowval).to(dev)
    del Bh
    assert torch.equal(got - 1, perm // d)
    del got, exp_colptr

    # prevpos[q] = the previous position of q's row (-1 if none): rows of positions [lo, hi) = #{q in [lo, hi): prevpos[q] < lo}
    perm = perm.to(torch.int32)
    head = torch.ones(N, dtype=torch.bool, device=dev)
    head[1:] = sr[1:] != sr[:-1]
    del sr
    prevpos = torch.empty(N, dtype=torch.int32, device=dev)
    prevpos[1:] = perm[:-1]
    prevpos[head] = -1
    del head
    pp = torch.empty_like(prevpos)
    pp[perm.to(torch.int64)] = prevpos
    prevpos = pp
    del perm, pp

    rng = np.random.default_rng(31)
    j = rng.integers(1, n + 1, 60)
    jp = np.minimum(j + rng.integers(1, 3000, 60), n + 1)
    edges = [TILE, 1 << 23, 1 << 29, 1 << 30, (1 << 30) + TILE, N // TILE * TILE, N - 1]  # tiles, MODE-2 windows, the end
    for b in edges:
        c = b // d + 1  # 1-based column of 0-based position b
        for a, ap in ((c - 1, c), (c, c + 1), (c - 1, c + 2), (c, min(c + 40, n + 1))):
            if 1 <= a < ap <= n + 1:
                j, jp = np.append(j, a), np.append(jp, ap)
    j, jp = np.append(j, [1, 1, n // 2]), np.append(jp, [n + 1, n // 2, n + 1])
    exp = np.array([int((prevpos[(int(a) - 1) * d:(int(ap) - 1) * d] < (int(a) - 1) * d).sum()) for a, ap in zip(j, jp)], dtype=np.int64)
    got, prof = profiled(lambda: cp.netcount(dA).query(j, jp))
    assert launches(prof, "k_os_pass") == os_passes(m), prof.get("k_os_pass")
    assert np.array_equal(got, exp), np.flatnonzero(got != exp)[:10]
    dA.close()


# ------------------------------------------------------------------------------------------ bisection and DP switches
@functools.lru_cache(maxsize=None)
def switch_inputs():
    return [("er50k", synth.erdos_renyi(50000, 10), 64, 0.01), ("rmat14", synth.rmat(14, 16 << 14), 128, 0.01),
            ("lap150", synth.laplacian5(150), 64, 0.001)]


BISECT_SWITCHES = ([{"CPB_BISECT_QUEUE": "1", "CPB_BISECT_PLAN": "0", "CPB_BISECT_DEPTH": str(d)} for d in (1, 2, 3, 4)]
                   + [{"CPB_UB_REFINE": "0"}, {"CPB_UB_REFINE": "1"}, {"CPB_BISECT_PREWALK": "0"},
                      {"CPB_L2_PREFETCH": "0", "CPB_PROBE_STREAM": "0"}])


@pytest.mark.parametrize("env", BISECT_SWITCHES, ids=lambda e: ",".join(f"{k[4:]}={v}" for k, v in e.items()))
def test_bisection_switches(ref, monkeypatch, env):
    """Queued rounds, the planner's bound refinement, the prewalk and the L2 prefetch of the dominance index (index path:
    work models always, connectivity with the streaming probes off) must not change a split vector."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    for name, A, K, eps in switch_inputs():
        dA = cp.device_matrix(A)
        for f in (AFF, cp.AffineWorkModel(0, 10, 1), SYM):
            for mk in (cp.BisectCostBottleneckSplitter, cp.LazyBisectCostBottleneckSplitter):
                mtd = mk(f, eps)
                assert np.array_equal(cp.partition_stripe(dA, K, mtd).spl, ref.partition_stripe(A, K, mtd).spl), (name, f, mk.__name__)
        dA.close()


def test_prewalk_off_on_the_envelope_case(ref, monkeypatch):
    d = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "envelope_prewalk_case.json")))
    A = cp.SparseMatrixCSC(d["m"], d["n"], d["colptr"], np.array(d["rowval"], dtype=np.int64))
    f = cp.AffineEnvelopeModel(1.5, 1.0, 1.5, 3.0)
    monkeypatch.setenv("CPB_BISECT_PREWALK", "0")
    for eps in (0.3, 0.1, 0.01, 0.001):
        for K in (2, 5, 9):
            for mk in (cp.BisectCostBottleneckSplitter, cp.LazyBisectCostBottleneckSplitter):
                assert np.array_equal(cp.partition_stripe(A, K, mk(f, eps)).spl, ref.partition_stripe(A, K, mk(f, eps)).spl), (eps, K, mk.__name__)


def test_dp_thread_windows(ref, monkeypatch):
    """CPB_DP_THREAD_WINDOWS=1: constrained Dynamic / Convex layers with windows wider than 64 columns one thread per
    column instead of a warp per column (banded 3000, w_max = 1.5 n / K)."""
    B = synth.banded(3000, 6, 3)
    monkeypatch.setenv("CPB_DP_THREAD_WINDOWS", "1")
    for K in (3, 8):
        spec = cp.ConstrainedCost(cp.AffineConnectivityModel(0, 0, 0, 1), cp.VertexCount(), int(np.ceil(B.n / K * 1.5)))
        for mk in (cp.ConvexTotalSplitter, cp.DynamicTotalSplitter, cp.DynamicBottleneckSplitter):
            assert np.array_equal(cp.partition_stripe(B, K, mk(spec)).spl, ref.partition_stripe(B, K, mk(spec)).spl), (K, mk.__name__)
        spec = cp.ConstrainedCost(cp.AffineConnectivityModel(0, 3, 1, 3), cp.AffineWorkModel(0, 1, 1), int(np.ceil((B.n + B.nnz) / K * 1.5)))
        for mk in (cp.ConvexTotalSplitter, cp.DynamicTotalSplitter):
            assert np.array_equal(cp.partition_stripe(B, K, mk(spec)).spl, ref.partition_stripe(B, K, mk(spec)).spl), (K, mk.__name__, "pin-weighted")


# ------------------------------------------------------------------------------------------ staged upload of Int64 indices
def test_staged_index_upload():
    """Index arrays of >= 2^21 Int64 entries are narrowed on the host while staged, chunk by chunk: a valid one round-trips,
    and a bad rowval entry at either side of the first chunk edge or at the end is refused for every kind of bad value."""
    m, n = 1000, 1 << 12
    N = (1 << 21) + 1000
    rng = np.random.default_rng(21)
    colptr = np.concatenate(([1], 1 + np.sort(rng.integers(0, N + 1, n - 1)), [N + 1])).astype(np.int64)
    rowval = rng.integers(1, m + 1, N).astype(np.int64)
    dA = cp.device_matrix(cp.SparseMatrixCSC(m, n, colptr, rowval))
    B = dA.to_host()
    dA.close()
    assert np.array_equal(B.colptr, colptr) and np.array_equal(B.rowval, rowval)
    for q in ((1 << 21) - 1, 1 << 21, N - 1):
        for bad in (0, m + 1, 1 << 31, (1 << 32) + 1, -1):
            rv = rowval.copy()
            rv[q] = bad
            with pytest.raises(cp.CpbError):
                cp.device_matrix(cp.SparseMatrixCSC(m, n, colptr, rv))
