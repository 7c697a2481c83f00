// links.cu -- kernel family "build_links": turns the CSC pattern into the point sets whose 2-D
// dominance counts are the reference's color arrays (SparseColorArrays.jl), plus adjointpattern.
//
// The reference walks the nonzeros column by column with a per-row "last seen" array hst[m]
// (NetCount :103-118, dianetcount! :72-99, SelfNetCount :177-229, SelfPinCount :281-318) -- a
// sequential sweep with a cache-missing gather.  Here the same quantities come from ONE stable
// radix sort of the nonzeros by row (i.e. the transpose order): the previous column holding the
// same row is simply the left neighbour inside the row run, and first/last columns are the run ends.
#include "engine.cuh"
#include "primitives.cuh"
#include "onesweep.cuh"

namespace cpb {

static unsigned grid_for(size_t n) { return (unsigned)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 32)); }

// flags[p] = 1 iff the sorted (row << 32 | position) pair p starts a row run; flags[N] = 0
__global__ void k_head_flags(const u64* __restrict__ sorted, size_t N, u32* __restrict__ flags) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p <= N; p += stride)
    flags[p] = (p < N && (p == 0 || (u32)(sorted[p - 1] >> 32) != (u32)(sorted[p] >> 32))) ? 1u : 0u;
}

// one point per non-empty row: x = last column, val = first column (both 1-based)
__global__ void k_selfnet_points(const u64* __restrict__ sorted, const u32* __restrict__ colidx, const u32* __restrict__ headscan, size_t N,
                                 u32* __restrict__ x, u32* __restrict__ val) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += stride) {
    const u64 cur = sorted[p];
    const u32 r = (u32)(cur >> 32);
    const bool head = (p == 0) || ((u32)(sorted[p - 1] >> 32) != r);
    const bool tail = (p + 1 == N) || ((u32)(sorted[p + 1] >> 32) != r);
    if (head | tail) {
      const u32 run = headscan[p] - (head ? 0u : 1u);
      const u32 c = __ldg(colidx + (u32)cur) + 1u;
      if (head) val[run] = c;
      if (tail) x[run] = c;
    }
  }
}

// one point per nonzero (i, j): x = max(i, j), val = min(i, j) (1-based)
__global__ void k_selfpin_points(const u32* __restrict__ row, const u32* __restrict__ colidx, size_t N, u32* __restrict__ x,
                                 u32* __restrict__ val) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride) {
    const u32 i = row[q] + 1u, j = colidx[q] + 1u;
    x[q] = max(i, j);
    val[q] = min(i, j);
  }
}

// add[j] = 1 iff column j lacks its diagonal entry (rows sorted within a column); add[n] = 0
__global__ void k_diag_missing(const u32* __restrict__ pos, const u32* __restrict__ row, u32 n, u32* __restrict__ add) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n; j += stride) {
    u32 a = 0;
    if (j < n) {
      u32 lo = pos[j], hi = pos[j + 1];
      while (lo < hi) {
        const u32 mid = lo + ((hi - lo) >> 1);
        if (row[mid] < (u32)j) lo = mid + 1; else hi = mid;
      }
      a = (lo < pos[j + 1] && row[lo] == (u32)j) ? 0u : 1u;
    }
    add[j] = a;
  }
}

__global__ void k_aug_pos(const u32* __restrict__ pos, const u32* __restrict__ addscan, u32 n, u32* __restrict__ pos2) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n; j += stride) pos2[j] = pos[j] + addscan[j];
}

__global__ void k_aug_rows(const u32* __restrict__ row, const u32* __restrict__ colidx, const u32* __restrict__ addscan, size_t N,
                           u32* __restrict__ row2) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride) row2[q + addscan[colidx[q]]] = row[q];
}

__global__ void k_aug_diag(const u32* __restrict__ pos2, const u32* __restrict__ add, u32 n, u32* __restrict__ row2) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride)
    if (add[j]) row2[pos2[j + 1] - 1] = (u32)j;  // virtual (j, j) entry appended to its column (:87-91)
}

// ---- link construction by an unordered transpose (rows of bounded degree) --------------------------------------
// When no row holds more than LT_MAX_DEG nonzeros the stable sort is unnecessary: the nonzeros are dropped into their
// row's segment in arbitrary order (one atomic cursor per row) and every entry finds its predecessor -- the largest
// CSC position below its own -- by scanning its row's short segment.  The result does not depend on the
// order inside the segments.  Heavier rows (power-law matrices) take the one-sweep sort (onesweep_links).
__global__ void k_lt_count(const u32* __restrict__ row, size_t N, u32* __restrict__ cnt) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride) atomicAdd(&cnt[row[q]], 1u);
}
__global__ void k_lt_max(const u32* __restrict__ cnt, size_t m, u32* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  u32 v = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) v = max(v, cnt[i]);
  v = __reduce_max_sync(0xffffffffu, v);
  __shared__ u32 sm[32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    v = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0u;
    v = __reduce_max_sync(0xffffffffu, v);
    if (threadIdx.x == 0 && v > *(volatile u32*)out) atomicMax(out, v);
  }
}
// (the three kernels below return at once when the maximal row degree, left behind the cursors by k_lt_max, exceeds the
//  limit: the host may launch them before it has seen that value and falls back to the sort afterwards)
__global__ void k_lt_fill(const u32* __restrict__ row, size_t N, u32* __restrict__ cursor, u32 m, u32* __restrict__ T) {
  if (cursor[m] > LT_MAX_DEG) return;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride) T[atomicAdd(&cursor[row[q]], 1u)] = (u32)q;
}
// after k_lt_fill, cursor[r] = end of row r's segment = start of row r + 1: mark the first slot of every non-empty row
__global__ void k_lt_heads(const u32* __restrict__ cursor, u32 m, u32* __restrict__ heads) {
  if (cursor[m] > LT_MAX_DEG) return;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < m; r += stride) {
    const u32 s = r ? cursor[r - 1] : 0u, e = cursor[r];
    if (e > s) atomicOr(&heads[s >> 5], 1u << (s & 31));
  }
}
// One thread per slot: the slot's row segment is delimited by the head bits around it; the predecessor of the slot's
// entry is the largest CSC position below its own inside the segment (positions ascend with the column), and its
// column is the link.  Neighbouring threads share a segment, so the scan reads are warp-wide broadcasts.
__global__ void k_lt_link(const u32* __restrict__ T, const u32* __restrict__ heads, const u32* __restrict__ colidx, size_t N,
                          u32* __restrict__ prev, u32* __restrict__ info, const u32* __restrict__ maxdeg, int as_pos) {
  u32* first_count = info;
  if (blockIdx.x == 0 && threadIdx.x == 0) info[1] = *maxdeg;
  if (*maxdeg > LT_MAX_DEG) return;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const u32 nwords = (u32)((N + 31) >> 5);
  u32 firsts = 0;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += stride) {
    u32 w = (u32)(p >> 5);
    u32 bits = heads[w] & (0xffffffffu >> (31 - (u32)(p & 31)));  // heads at or before p (slot 0 is always one)
    while (!bits) bits = heads[--w];
    const u32 s = (w << 5) + (31 - __clz(bits));
    w = (u32)(p >> 5);
    bits = (p & 31) == 31 ? 0u : (heads[w] & (0xffffffffu << ((u32)(p & 31) + 1)));
    while (!bits && ++w < nwords) bits = heads[w];
    const u32 e = bits ? min((u32)N, (w << 5) + (u32)__ffs(bits) - 1u) : (u32)N;
    const u32 qi = T[p];
    u32 best = 0;  // 1 + position of the previous nonzero of this row, 0 = none
    for (u32 k = s; k < e; ++k) {
      const u32 qk = T[k];
      if (qk < qi) best = max(best, qk + 1u);
    }
    prev[qi] = (best && !as_pos) ? __ldg(colidx + (best - 1u)) + 1u : best;  // 1-based previous column (or position) of this row
    firsts += best == 0u;
  }
  firsts = __reduce_add_sync(0xffffffffu, firsts);
  if ((threadIdx.x & 31) == 0 && firsts) atomicAdd(first_count, firsts);
}

// colq[g] = 0-based column of element g * LS_COLQ = the largest c with P[c + 1] <= g * LS_COLQ (P[x] = elements in columns < x,
// 1-based), n - 1 behind the end of the array
__global__ void k_colq(const u32* __restrict__ P, u32 n, size_t Ne, u32* __restrict__ colq, u32 G) {
  const u32 g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g > G) return;
  const size_t e = (size_t)g * LS_COLQ;
  u32 c = n ? n - 1 : 0;
  if (e < Ne && n) {
    u32 lo = 0, hi = n - 1;  // P[1] = 0 <= e
    while (lo < hi) {
      const u32 mid = lo + ((hi - lo + 1) >> 1);
      if ((size_t)__ldg(P + mid + 1) <= e) lo = mid; else hi = mid - 1;
    }
    c = lo;
  }
  colq[g] = c;
}
void fill_colq(LinkStream& ls, u32 n) {
  const u32 G = (u32)((ls.Ne + LS_COLQ - 1) / LS_COLQ);
  ls.colq.alloc((size_t)G + 2);
  CPB_LAUNCH(k_colq, (G + 1) / 256 + 1, 256, 0, ls.P, n, ls.Ne, ls.colq.get(), G + 1);
}

static u32 read_u32(const u32* d) {
  u32 h = 0;
  CPB_CUDA(cudaMemcpyAsync(&h, d, sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  return h;
}

// prev[q] = 1-based previous column holding the same row (0 if none); colidx[q] = 0-based column of q
// info[0] receives the number of links equal to 0 (= non-empty rows), info[1] the maximal row degree when the row-segment
// form was tried (0 otherwise).  defer_check: do not wait for that degree -- launch the row-segment kernels at once (they
// do nothing if the degree is too large) and return true; the caller inspects info[1] later and calls again with
// CPB_NO_ROW_SEGMENTS semantics (force_sort) if it exceeds LT_MAX_DEG.
bool compute_prev_links(const u32* pos, const u32* row, u32 nrow, u32 ncol, size_t N, u32* prev, u32* colidx, u32* first_count,
                        bool defer_check, bool force_sort, bool as_pos, i64* max_deg_cache) {
  ProfScope prof("build_links", (double)(2 * N + ncol + 1) * 4.0);
  CPB_REQUIRE(colidx || as_pos, "column-valued links need the column array");
  if (colidx) {
    ProfScope pk("k_expand_columns", (double)N * 4.0 + (double)ncol * 4.0);
    expand_columns(pos, ncol, colidx, N);
  }
  DBuf<u32> dummy;
  if (!first_count) { dummy.alloc(2); first_count = dummy.get(); }
  CPB_CUDA(cudaMemsetAsync(first_count, 0, 2 * sizeof(u32), ctx().stream));
  // a row known to be too heavy (an earlier construction on the same resident matrix saw it): straight to the sort
  const bool known_heavy = max_deg_cache && *max_deg_cache > (i64)LT_MAX_DEG;
  const bool no_lt = force_sort || known_heavy || std::getenv("CPB_NO_ROW_SEGMENTS") != nullptr;  // (tests: force the radix-sort path)
  if (N && nrow && !no_lt) {
    DBuf<u32> cur((size_t)nrow + 1);  // per-row counts -> segment starts -> (after the fill) segment ends; [nrow] = max degree
    CPB_CUDA(cudaMemsetAsync(cur.get(), 0, ((size_t)nrow + 1) * sizeof(u32), ctx().stream));
    u32 seen_deg = 0;
    size_t counted = 0;
    if (!defer_check && N >= ((size_t)1 << 25)) {
      // large pattern, degree not known: count a 1/16 prefix first -- a power-law matrix shows its heavy rows at once and
      // goes to the sort without paying for the whole histogram (2.9 ms at 2.6e8 nonzeros)
      counted = N / 16;
      ProfScope pk("k_lt_count", (double)counted * 4.0);
      CPB_LAUNCH(k_lt_count, grid_for(counted), 256, 0, row, counted, cur.get());
      CPB_LAUNCH(k_lt_max, grid_for(nrow), 256, 0, cur.get(), (size_t)nrow, cur.get() + nrow);
      seen_deg = read_u32(cur.get() + nrow);
    }
    if (seen_deg <= LT_MAX_DEG) {
      {
        ProfScope pk("k_lt_count", (double)(N - counted) * 4.0);
        CPB_LAUNCH(k_lt_count, grid_for(N - counted), 256, 0, row + counted, N - counted, cur.get());
      }
      CPB_LAUNCH(k_lt_max, grid_for(nrow), 256, 0, cur.get(), (size_t)nrow, cur.get() + nrow);
      if (!defer_check) seen_deg = read_u32(cur.get() + nrow);
    }
    if (!defer_check && max_deg_cache) *max_deg_cache = (i64)seen_deg;  // (a lower bound when the prefix already exceeded the limit)
    if (defer_check || seen_deg <= LT_MAX_DEG) {
      exclusive_scan_u32(cur.get(), cur.get(), (size_t)nrow);
      DBuf<u32> T(N);
      {
        ProfScope pk("k_lt_fill", (double)N * 8.0);
        CPB_LAUNCH(k_lt_fill, grid_for(N), 256, 0, row, N, cur.get(), nrow, T.get());
      }
      {
        ProfScope pk("k_lt_link", (double)N * 12.0);
        DBuf<u32> heads(N / 32 + 2);
        heads.zero();
        CPB_LAUNCH(k_lt_heads, grid_for(nrow), 256, 0, cur.get(), nrow, heads.get());
        CPB_LAUNCH(k_lt_link, grid_for(N), 256, 0, T.get(), heads.get(), colidx, N, prev, first_count, cur.get() + nrow, as_pos ? 1 : 0);
      }
      return defer_check;
    }
  }
  trace_mark("degree_check");
  if (!N) return false;
  const char* wmin_env = std::getenv("CPB_WINDOWED_SCATTER_MIN");  // (tests force the windowed form on small inputs; 0 = never)
  const size_t wmin = wmin_env ? (size_t)std::atoll(wmin_env) : ((size_t)1 << 25);
  // one-read-one-write radix passes on packed (row, position) pairs; the window pass forms the links while loading
  DBuf<u64> a(N), b(N);
  onesweep_links(row, N, bits_for(nrow ? nrow - 1 : 0), colidx, as_pos, 0u, prev, first_count, nullptr, wmin, a.get(), b.get());
  return false;
}

// The link array of A (dia = false) or of A + I (dia = true, SparseColorArrays.jl:72-99) in column order,
// kept for the streaming probes; P[x] = #{elements in columns < x}.
std::unique_ptr<LinkStream> build_link_stream(const Matrix& A, bool dia, bool defer_check, bool force_sort, bool as_pos) {
  auto ls = std::make_unique<LinkStream>();
  ls->pos_links = as_pos;
  const size_t N = (size_t)A.N;
  const u32 n = (u32)A.n, m = (u32)A.m;
  if (!dia) {
    ls->Ne = N;
    ls->prev.alloc(N);
    if (!as_pos) ls->colidx.alloc(N);
    ls->first_count.alloc(2);
    ls->speculative = compute_prev_links(A.pos.get(), A.row.get(), m, n, N, ls->prev.get(), as_pos ? nullptr : ls->colidx.get(), ls->first_count.get(),
                                         defer_check, force_sort, as_pos, &A.max_row_deg);
    ls->P = A.pos.get() - 1;  // P[x] = pos[x-1]
    fill_colq(*ls, n);
    return ls;
  }
  CPB_REQUIRE(A.m >= A.n, "dianetcount needs m >= n");
  DBuf<u32> add((size_t)n + 1), colidx(N);
  CPB_LAUNCH(k_diag_missing, grid_for((size_t)n + 1), 256, 0, A.pos.get(), A.row.get(), n, add.get());
  DBuf<u32> addscan((size_t)n + 1);
  exclusive_scan_u32(add.get(), addscan.get(), (size_t)n + 1);
  const size_t N2 = N + read_u32(addscan.get() + n);
  ls->P_own.alloc((size_t)n + 2);
  u32* pos2 = ls->P_own.get() + 1;
  CPB_CUDA(cudaMemsetAsync(ls->P_own.get(), 0, sizeof(u32), ctx().stream));
  CPB_LAUNCH(k_aug_pos, grid_for((size_t)n + 1), 256, 0, A.pos.get(), addscan.get(), n, pos2);
  DBuf<u32> row2(N2);
  expand_columns(A.pos.get(), n, colidx.get(), N);
  if (N) CPB_LAUNCH(k_aug_rows, grid_for(N), 256, 0, A.row.get(), colidx.get(), addscan.get(), N, row2.get());
  if (n) CPB_LAUNCH(k_aug_diag, grid_for(n), 256, 0, pos2, add.get(), n, row2.get());
  i64 heavy_hint = A.max_row_deg > (i64)LT_MAX_DEG ? A.max_row_deg : -1;  // A + I only adds entries: a heavy row of A stays heavy
  ls->Ne = N2;
  ls->prev.alloc(N2);
  if (!as_pos) ls->colidx.alloc(N2);
  ls->first_count.alloc(2);
  ls->speculative = compute_prev_links(pos2, row2.get(), m, n, N2, ls->prev.get(), as_pos ? nullptr : ls->colidx.get(), ls->first_count.get(),
                                       defer_check, force_sort, as_pos, &heavy_hint);
  ls->P = ls->P_own.get();  // P[x] = pos2[x-1]
  fill_colq(*ls, n);
  return ls;
}

// sorts points by x, builds P and the wavelet matrix over val
static void build_from_points(DBuf<u32>& x, DBuf<u32>& val, size_t npts, u32 ncol, RankStruct& rs) {
  DBuf<u32> x2(npts), val2(npts);
  const int which = radix_sort_pairs(x.get(), val.get(), x2.get(), val2.get(), npts, bits_for(ncol));
  u32* xs = which ? x2.get() : x.get();
  u32* vs = which ? val2.get() : val.get();
  u32* other = which ? val.get() : val2.get();
  rs.P_own.alloc((size_t)ncol + 2);
  segment_starts(xs, npts, rs.P_own.get(), ncol + 1);
  rs.P = rs.P_own.get();
  rs.wm.build(vs, other, npts, ncol);
}

std::unique_ptr<RankStruct> build_rank(const Matrix& A, int which) {
  auto rs = std::make_unique<RankStruct>();
  const size_t N = (size_t)A.N;
  const u32 n = (u32)A.n, m = (u32)A.m;
  switch (which) {
    case RANK_NET:
    case RANK_DIANET: {
      // the wavelet build consumes the link array (ping-pong) and the column index (scratch)
      auto ls = build_link_stream(A, which == RANK_DIANET);
      rs->wm.build(ls->prev.get(), ls->colidx.get(), ls->Ne, n);
      rs->P_own = std::move(ls->P_own);
      rs->P = (which == RANK_DIANET) ? rs->P_own.get() : A.pos.get() - 1;
      break;
    }
    case RANK_SELFNET: {
      DBuf<u64> a(N), b(N);
      const u64* sorted = N ? onesweep_sort_iota(A.row.get(), N, bits_for(m ? m - 1 : 0), a.get(), b.get()) : nullptr;
      DBuf<u32> colidx(N), flags(N + 1), headscan(N + 1);
      expand_columns(A.pos.get(), n, colidx.get(), N);
      CPB_LAUNCH(k_head_flags, grid_for(N + 1), 256, 0, sorted, N, flags.get());
      exclusive_scan_u32(flags.get(), headscan.get(), N + 1);
      const size_t R = read_u32(headscan.get() + N);
      DBuf<u32> x(R), val(R);
      if (N) CPB_LAUNCH(k_selfnet_points, grid_for(N), 256, 0, sorted, colidx.get(), headscan.get(), N, x.get(), val.get());
      build_from_points(x, val, R, n, *rs);
      break;
    }
    case RANK_SELFPIN: {
      CPB_REQUIRE(A.m <= A.n, "selfpincount needs row indices <= n");
      DBuf<u32> colidx(N), x(N), val(N);
      expand_columns(A.pos.get(), n, colidx.get(), N);
      if (N) CPB_LAUNCH(k_selfpin_points, grid_for(N), 256, 0, A.row.get(), colidx.get(), N, x.get(), val.get());
      build_from_points(x, val, N, n, *rs);
      break;
    }
    default: throw Error(-1, "bad rank structure kind");
  }
  return rs;
}

// PRIMCONN: elements regrouped by the row part of their row (stable: columns stay ascending inside a part), wavelet matrix
// over their column-valued links (PartwiseCounts.jl:1-67 builds the same "stacked" matrix and a net count on it)
__global__ void k_part_ids(const u32* __restrict__ row, const u32* __restrict__ asg, size_t N, u32* __restrict__ pid) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride) pid[q] = asg[row[q]];
}
__global__ void k_part_gather(const u32* __restrict__ sq, const u32* __restrict__ colidx, const u32* __restrict__ prev, size_t N,
                              u32* __restrict__ col_s, u32* __restrict__ prev_s) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += stride) {
    const u32 q = sq[p];
    col_s[p] = colidx[q];
    prev_s[p] = prev[q];
  }
}
std::unique_ptr<RankStruct> build_partwise_rank(const Matrix& A, const u32* asg, u32 K, DBuf<u32>& part_col, DBuf<u32>& part_start) {
  auto rs = std::make_unique<RankStruct>();
  const size_t N = (size_t)A.N;
  const u32 n = (u32)A.n, m = (u32)A.m;
  DBuf<u32> prev(N), colidx(N), pid(N), k0(N), v0(N), k1(N), v1(N), prev_s(N);
  compute_prev_links(A.pos.get(), A.row.get(), m, n, N, prev.get(), colidx.get());
  if (N) CPB_LAUNCH(k_part_ids, grid_for(N), 256, 0, A.row.get(), asg, N, pid.get());
  const int which = radix_sort_pairs_iota(pid.get(), k0.get(), v0.get(), k1.get(), v1.get(), N, bits_for(K ? K - 1 : 0));
  const u32* keys = which ? k1.get() : k0.get();
  const u32* sq = which ? v1.get() : v0.get();
  part_col.alloc(N + 1);
  if (N) CPB_LAUNCH(k_part_gather, grid_for(N), 256, 0, sq, colidx.get(), prev.get(), N, part_col.get(), prev_s.get());
  part_start.alloc((size_t)K + 2);
  segment_starts(keys, N, part_start.get(), K);  // part_start[k] = first stacked element with part id >= k, k = 0..K
  rs->wm.build(prev_s.get(), prev.get(), N, n);
  rs->P = nullptr;
  return rs;
}

// SECCONN: the same regrouping without links; part_head = exclusive scan of "first element of its (part, column) pair"
__global__ void k_part_heads(const u32* __restrict__ keys, const u32* __restrict__ col_s, size_t N, u32* __restrict__ flags) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p <= N; p += stride)
    flags[p] = (p < N && (p == 0 || keys[p] != keys[p - 1] || col_s[p] != col_s[p - 1])) ? 1u : 0u;
}
__global__ void k_gather_u32(const u32* __restrict__ idx, const u32* __restrict__ src, size_t N, u32* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += stride) out[p] = src[idx[p]];
}
void build_partwise_columns(const Matrix& A, const u32* asg, u32 K, DBuf<u32>& part_col, DBuf<u32>& part_start, DBuf<u32>& part_head) {
  const size_t N = (size_t)A.N;
  DBuf<u32> colidx(N), pid(N), k0(N), v0(N), k1(N), v1(N), flags(N + 1);
  expand_columns(A.pos.get(), (u32)A.n, colidx.get(), N);
  if (N) CPB_LAUNCH(k_part_ids, grid_for(N), 256, 0, A.row.get(), asg, N, pid.get());
  const int which = radix_sort_pairs_iota(pid.get(), k0.get(), v0.get(), k1.get(), v1.get(), N, bits_for(K ? K - 1 : 0));
  const u32* keys = which ? k1.get() : k0.get();
  const u32* sq = which ? v1.get() : v0.get();
  part_col.alloc(N + 1);
  if (N) CPB_LAUNCH(k_gather_u32, grid_for(N), 256, 0, sq, colidx.get(), N, part_col.get());
  part_start.alloc((size_t)K + 2);
  segment_starts(keys, N, part_start.get(), K);
  CPB_LAUNCH(k_part_heads, grid_for(N + 1), 256, 0, keys, part_col.get(), N, flags.get());
  part_head.alloc(N + 1);
  exclusive_scan_u32(flags.get(), part_head.get(), N + 1);
}

// adjointpattern(A) (util.jl:67-95): stable sort by row = CSC of the transpose; row'[p] = column of the p-th sorted
// (row << 32 | position) pair, pos'[i] = first sorted index with row >= i, i = 0..m
__global__ void k_gather_cols_pairs(const u64* __restrict__ sorted, const u32* __restrict__ colidx, size_t N, u32* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < N; p += stride) out[p] = colidx[(u32)sorted[p]];
}
__global__ void k_segment_starts_pairs(const u64* __restrict__ sorted, size_t n, u32* __restrict__ P, u32 domain) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p <= n; p += stride) {
    const i64 lo = (p == 0) ? 0 : (i64)(u32)(sorted[p - 1] >> 32) + 1;
    const i64 hi = (p == n) ? (i64)domain : (i64)(u32)(sorted[p] >> 32);
    for (i64 x = lo; x <= hi; ++x) P[x] = (u32)p;
  }
}

std::unique_ptr<Matrix> adjoint_pattern(const Matrix& A) {
  auto B = std::make_unique<Matrix>();
  B->m = A.n; B->n = A.m; B->N = A.N;
  const size_t N = (size_t)A.N;
  ProfScope prof("adjointpattern", (double)(2 * N + A.n + A.m + 2) * 4.0);
  DBuf<u64> a(N), b(N);
  const u64* sorted = N ? onesweep_sort_iota(A.row.get(), N, bits_for(A.m ? A.m - 1 : 0), a.get(), b.get()) : nullptr;
  DBuf<u32> colidx(N);
  expand_columns(A.pos.get(), (u32)A.n, colidx.get(), N);
  B->row.alloc(N);
  if (N) CPB_LAUNCH(k_gather_cols_pairs, grid_for(N), 256, 0, sorted, colidx.get(), N, B->row.get());
  B->pos.alloc((size_t)A.m + 1);
  const unsigned grid = (unsigned)std::min<size_t>((N + 1 + 255) / 256, (size_t)ctx().sm_count * 16);
  CPB_LAUNCH(k_segment_starts_pairs, grid, 256, 0, sorted, N, B->pos.get(), (u32)A.m);  // (N = 0: pos' = 0, sorted unread)
  return B;
}

// ---- A[:, prm] with relabelled rows: the first step of the objective evaluators for non-contiguous partitions
// (Costs.jl:34-39, 52-57: "A_prm = A[:, Phi_dom.prm]"; a MapPartition of the rows becomes a SplitPartition by renumbering
// the rows part by part -- every partition-aware count depends on a row only through the part that owns it).
__global__ void k_perm_degrees(const u32* __restrict__ pos, const u32* __restrict__ prm, u32 n, u32* __restrict__ deg) {
  const u32 c = blockIdx.x * 256u + threadIdx.x;
  if (c > n) return;
  u32 d = 0;
  if (c < n) {
    const u32 p = prm ? __ldg(prm + c) : c;
    d = __ldg(pos + p + 1) - __ldg(pos + p);
  }
  deg[c] = d;  // entry n = 0, so the exclusive scan over n + 1 entries ends with the total
}

__global__ void k_perm_rows(const u32* __restrict__ pos, const u32* __restrict__ row, const u32* __restrict__ prm, const u32* __restrict__ row_new,
                            const u32* __restrict__ new_pos, const u32* __restrict__ new_col, size_t N, u32* __restrict__ out) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < N; q += stride) {
    const u32 c = __ldg(new_col + q);
    const u32 p = prm ? __ldg(prm + c) : c;
    const u32 r = __ldg(row + __ldg(pos + p) + ((u32)q - __ldg(new_pos + c)));
    out[q] = row_new ? __ldg(row_new + r) : r;
  }
}

// flags |= 1 unless v[0..n) is a permutation of 0..n-1 (seen: n zero-initialised words)
__global__ void k_check_permutation(const u32* __restrict__ v, u32 n, u32* __restrict__ seen, u32* __restrict__ flags) {
  const u32 i = blockIdx.x * 256u + threadIdx.x;
  if (i >= n) return;
  const u32 x = v[i];
  if (x >= n || atomicExch(seen + x, 1u) != 0u) atomicOr(flags, 1u);
}

std::unique_ptr<Matrix> permute_pattern(const Matrix& A, const u32* col_prm, const u32* row_new) {
  auto B = std::make_unique<Matrix>();
  B->m = A.m; B->n = A.n; B->N = A.N;
  const size_t N = (size_t)A.N;
  const u32 n = (u32)A.n;
  ProfScope prof("permute_pattern", (double)(3 * N + 3 * (size_t)n) * 4.0);
  DBuf<u32> flags(1);
  flags.zero();
  for (int side = 0; side < 2; ++side) {
    const u32* v = side ? row_new : col_prm;
    const u32 len = side ? (u32)A.m : n;
    if (!v || len == 0) continue;
    DBuf<u32> seen(len);
    seen.zero();
    CPB_LAUNCH(k_check_permutation, (len + 255) / 256, 256, 0, v, len, seen.get(), flags.get());
  }
  B->pos.alloc((size_t)n + 1);
  B->row.alloc(N);
  DBuf<u32> deg((size_t)n + 1);
  CPB_LAUNCH(k_perm_degrees, n / 256 + 1, 256, 0, A.pos.get(), col_prm, n, deg.get());
  exclusive_scan_u32(deg.get(), B->pos.get(), (size_t)n + 1);
  if (N) {
    DBuf<u32> new_col(N);
    expand_columns(B->pos.get(), n, new_col.get(), N);
    CPB_LAUNCH(k_perm_rows, grid_for(N), 256, 0, A.pos.get(), A.row.get(), col_prm, row_new, B->pos.get(), new_col.get(), N, B->row.get());
  }
  u32 hf = 0;
  CPB_CUDA(cudaMemcpyAsync(&hf, flags.get(), sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  CPB_REQUIRE(hf == 0, "not a permutation (expected every index 1..len exactly once)");
  return B;
}

}  // namespace cpb
