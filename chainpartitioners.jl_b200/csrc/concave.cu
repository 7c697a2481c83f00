// concave.cu -- ConcaveTotalChunker / ConcaveTotalSplitter (ConcaveTotalChunker.jl) on the device.
//
// chunk_concave! (:57-114) is an ONLINE queue algorithm: column j' is settled from the queue's front, then the candidate
// j' - 1 is inserted by popping dominated entries off the back and a binary search for the column where it overtakes the
// new back.  Its pointers depend on that exact control flow whenever the cost is not strictly inverse-Monge (ties, or a
// model that is not concave at all), so the device runs the same sequence: one thread walks the columns, every cost is a
// random-access oracle query (rank descents on the wavelet index), the queue is a circular buffer in global memory.  That
// is ~2 n log n dependent queries of ~1 us each -- correct and identical to the reference, but latency-bound: the K-form
// initialises its layers in parallel and the layers themselves are the sequential part.  (No parallel rule with the same
// tie-breaking is known; the convex forms have one -- dynamic.cu, chunk.cu.)  Numbers in DESIGN.md.
#include "engine.cuh"

namespace cpb {

// Extended{T} (Costs.jl:79-103): a cost or infinity; `+` ORs the flags, infinities compare equal
template <class T> struct XC {
  T x;
  int inf;
};
template <class T> __device__ __forceinline__ bool xc_le(const XC<T>& a, const XC<T>& b) { return a.inf ? (b.inf != 0) : (b.inf || a.x <= b.x); }
template <class T> __device__ __forceinline__ bool xc_gt(const XC<T>& a, const XC<T>& b) { return b.inf ? false : (a.inf || a.x > b.x); }

// one column of costs with a window [lo, hi]: reads outside give infinity, writes outside are dropped
// (WindowConstrainedMatrix, DynamicSplitter.jl:101-142; the unconstrained forms use lo = 1, hi = n + 1)
template <class T> struct XCol {
  T* x;
  unsigned char* inf;
  u32 lo, hi;
  __device__ __forceinline__ XC<T> get(u32 i) const {
    if (i < lo || i > hi) return XC<T>{T(0), 1};
    return XC<T>{x[i], (int)inf[i]};
  }
  __device__ __forceinline__ void set(u32 i, const XC<T>& v) const {
    if (i < lo || i > hi) return;
    x[i] = v.x;
    inf[i] = (unsigned char)v.inf;
  }
};

template <class T> __device__ __forceinline__ XC<T> concave_fp(const DevOracle& o, const XCol<T>& prev, u32 j, u32 jp, u32 k) {
  const XC<T> p = prev.get(j);
  return XC<T>{(T)(p.x + dev_cost<T>(o, j, jp, k)), p.inf};
}

// layer initialisation of the K-form (:44-47, :171-174): cst[j', k] = cst[j', k - 1] + f(j', j', k), ptr[j', k] = j'
template <class T>
__global__ void k_concave_init(const __grid_constant__ DevOracle o, XCol<T> prev, XCol<T> cur, u32* __restrict__ ptr, u32 k) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x + cur.lo; i <= cur.hi; i += stride) {
    const u32 jp = (u32)i;
    cur.set(jp, concave_fp<T>(o, prev, jp, jp, k));
    ptr[jp] = jp;
  }
}
// first layer (:40-43, :166-169): cst[j', 1] = f(1, j', 1), ptr[j', 1] = 1
template <class T> __global__ void k_concave_first(const __grid_constant__ DevOracle o, XCol<T> cur, u32* __restrict__ ptr) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x + cur.lo; i <= cur.hi; i += stride) {
    const u32 jp = (u32)i;
    cur.set(jp, XC<T>{dev_cost<T>(o, 1u, jp, 1u), 0});
    ptr[jp] = 1u;
  }
}
template <class T> __global__ void k_concave_fill(XCol<T> c, T v, int inf, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) { c.x[i] = v; c.inf[i] = (unsigned char)inf; }
}

// chunk_concave!(cst, ptr, f', j0, j'1, ftr) (:57-114) with f'(j, j') = prev[j] + f(j, j', k); prev may be cur itself (the chunker
// form: column j is final before any f'(j, .) is asked for).  ptr_win: writes to ptr are dropped outside cur's window.
template <class T>
__global__ void k_concave_chain(const __grid_constant__ DevOracle o, XCol<T> prev, XCol<T> cur, u32* __restrict__ ptr, u32 j0, u32 jp1, u32 k,
                                u32* __restrict__ qj, u32* __restrict__ qh, u32 cap) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  u32 hd = 0, sz = 0;
  auto push_back = [&](u32 j, u32 h) { const u32 p = (hd + sz) % cap; qj[p] = j; qh[p] = h; ++sz; };
  auto push_front = [&](u32 j, u32 h) { hd = (hd + cap - 1) % cap; qj[hd] = j; qh[hd] = h; ++sz; };
  auto set_ptr = [&](u32 jp, u32 v) { if (jp >= cur.lo && jp <= cur.hi) ptr[jp] = v; };
  push_back(j0, j0 + 1);
  for (u32 jp = j0 + 1; jp <= jp1; ++jp) {
    u32 j = qj[hd];
    const XC<T> c = concave_fp<T>(o, prev, j, jp, k);
    const XC<T> c2 = concave_fp<T>(o, prev, jp - 1, jp, k);
    if (xc_le(c2, c)) {
      if (xc_le(c2, cur.get(jp))) { cur.set(jp, c2); set_ptr(jp, jp - 1); }
      sz = 0;
      push_back(jp - 1, jp + 1);
    } else {
      if (xc_le(c, cur.get(jp))) { cur.set(jp, c); set_ptr(jp, j); }
      u32 h;
      while (true) {  // (the reference pops without an emptiness check: the front entry's h is at most j' and survives)
        const u32 b = (hd + sz - 1) % cap;
        j = qj[b];
        h = qh[b];
        if (!xc_le(concave_fp<T>(o, prev, jp - 1, h, k), concave_fp<T>(o, prev, j, h, k))) break;
        --sz;
      }
      long long h_lo = (long long)h + 1, h_hi = (long long)jp1;
      while (h_lo <= h_hi) {
        const long long mid = (h_lo + h_hi) >> 1;  // fld2
        if (xc_gt(concave_fp<T>(o, prev, jp - 1, (u32)mid, k), concave_fp<T>(o, prev, j, (u32)mid, k))) h_lo = mid + 1; else h_hi = mid - 1;
      }
      if (h_lo != (long long)jp1 + 1) push_back(jp - 1, (u32)h_lo);
      j = qj[hd];
      hd = (hd + 1) % cap;  // popfirst!
      --sz;
      if (sz == 0 || qh[hd] != jp + 1) push_front(j, jp + 1);
    }
  }
}

static unsigned grid_for(size_t n) { return (unsigned)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)ctx().sm_count * 8)); }

template <class T> struct XColBuf {
  DBuf<T> x;
  DBuf<unsigned char> inf;
  void alloc(size_t n) { x.alloc(n); inf.alloc(n); }
  XCol<T> view(u32 lo, u32 hi) { return XCol<T>{x.get(), inf.get(), lo, hi}; }
};

// pack_stripe(A, ConcaveTotalChunker(f)) (:9-24)
template <class T> static void concave_chunker_T(Oracle& f, int64_t* h_spl_out, int64_t* K_out) {
  const i64 n = f.A->n;
  const u32 n1 = (u32)n + 1;
  ProfScope prof("concave_chain");
  XColBuf<T> cst;
  cst.alloc((size_t)n1 + 1);
  DBuf<u32> spl((size_t)n1 + 1), qj((size_t)n1 + 2), qh((size_t)n1 + 2);
  spl.zero();
  XCol<T> c = cst.view(1, n1);
  CPB_LAUNCH(k_concave_fill<T>, grid_for((size_t)n1 + 1), 256, 0, c, T(0), 1, (size_t)n1 + 1);  // typemax
  const T zero = T(0);
  const unsigned char fin = 0;
  CPB_CUDA(cudaMemcpyAsync(cst.x.get() + 1, &zero, sizeof(T), cudaMemcpyHostToDevice, ctx().stream));
  CPB_CUDA(cudaMemcpyAsync(cst.inf.get() + 1, &fin, 1, cudaMemcpyHostToDevice, ctx().stream));
  if (n >= 1) CPB_LAUNCH(k_concave_chain<T>, 1, 32, 0, f.dev, c, c, spl.get(), 1u, n1, 1u, qj.get(), qh.get(), n1 + 2);
  // unravel_chunks! (DynamicChunker.jl:58-75)
  std::vector<u32> h((size_t)n1 + 1);
  CPB_CUDA(cudaMemcpyAsync(h.data(), spl.get(), ((size_t)n1 + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  std::vector<i64> rev;
  for (i64 jp = n + 1; jp != 1;) {
    CPB_REQUIRE(rev.size() <= (size_t)n, "chunk pointers do not lead back to column 1");
    rev.push_back(jp);
    jp = (i64)h[(size_t)jp];
  }
  const i64 K = (i64)rev.size();
  h_spl_out[0] = 1;
  for (i64 t = 0; t < K; ++t) h_spl_out[t + 1] = rev[(size_t)(K - 1 - t)];
  *K_out = K;
}

__global__ void k_concave_unravel(const u32* __restrict__ ptr, u32 n2, int K, u32 n1, i64* __restrict__ spl) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {  // DynamicSplitter.jl:89-99
    spl[K] = n1;
    for (int k = K; k >= 1; --k) {
      const i64 s = spl[k];
      spl[k - 1] = (s >= 0 && s <= (i64)n1) ? (i64)ptr[(size_t)(k - 1) * n2 + (u32)s] : 0;
    }
  }
}

// partition_stripe(A, K, ConcaveTotalSplitter(f)) (:26-55) and its ConstrainedCost form (:143-181)
template <class T> static void concave_splitter_T(Oracle& f, const Windows* win, i64 K, int64_t* h_spl_out) {
  const Matrix& A = *f.A;
  const i64 n = A.n;
  const u32 n1 = (u32)n + 1, n2 = n1 + 1;
  std::vector<i64> lo(K + 1, 1), hi(K + 1, n + 1);
  const bool windowed = win != nullptr;
  if (windowed) {
    // column_constraints (DynamicSplitter.jl:144-173); the weight shapes nothing but the windows
    if (!column_constraints(*win, n, K, lo, hi)) {  // :153-158 infeasible -> degenerate partition
      degenerate_partition(n, K, h_spl_out);
      return;
    }
  } else if (K == 1) {  // :33-35
    h_spl_out[0] = 1;
    h_spl_out[1] = n + 1;
    return;
  }
  CPB_REQUIRE((double)K * n2 * 4.0 < 64e9, "DP pointer table would not fit");
  ProfScope prof("concave_chain");
  XColBuf<T> ra, rb;
  ra.alloc(n2);
  rb.alloc(n2);
  DBuf<u32> ptr((size_t)K * n2), qj((size_t)n1 + 2), qh((size_t)n1 + 2);
  DBuf<i64> spl(K + 1);
  ptr.zero();
  XColBuf<T>* prev = &ra;
  XColBuf<T>* cur = &rb;
  {
    XCol<T> c1 = prev->view((u32)lo[1], (u32)hi[1]);
    CPB_LAUNCH(k_concave_first<T>, grid_for((size_t)(hi[1] - lo[1] + 1)), 256, 0, f.dev, c1, ptr.get());
  }
  for (i64 k = 2; k <= K; ++k) {
    XCol<T> p = prev->view((u32)lo[k - 1], (u32)hi[k - 1]);
    XCol<T> c = cur->view((u32)lo[k], (u32)hi[k]);
    u32* pk = ptr.get() + (size_t)(k - 1) * n2;
    CPB_LAUNCH(k_concave_init<T>, grid_for((size_t)(hi[k] - lo[k] + 1)), 256, 0, f.dev, p, c, pk, (u32)k);
    const u32 j0 = windowed ? (u32)lo[k - 1] : 1u, jp1 = windowed ? (u32)hi[k] : n1;
    if (jp1 > j0) CPB_LAUNCH(k_concave_chain<T>, 1, 32, 0, f.dev, p, c, pk, j0, jp1, (u32)k, qj.get(), qh.get(), n1 + 2);
    std::swap(prev, cur);
  }
  CPB_LAUNCH(k_concave_unravel, 1, 32, 0, ptr.get(), n2, (int)K, n1, spl.get());
  CPB_CUDA(cudaMemcpyAsync(h_spl_out, spl.get(), (K + 1) * sizeof(i64), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
}

static void concave_check_model(const Oracle& f) {
  if (f.dev.kind == CPB_MODEL_BLOCK) throw Error(CPB_ERR_UNSUPPORTED, "Concave chunker / splitter need a random-access oracle (step oracles cannot answer f(j, h))");
}

void solve_concave_chunker(Oracle& f, const cpb_constraint* con, int64_t* h_spl_out, int64_t* K_out) {
  concave_check_model(f);
  if (con && con->enabled)
    throw Error(CPB_ERR_UNSUPPORTED, "pack_stripe(A, ConcaveTotalChunker(ConstrainedCost)) has no method in the reference (ConcaveTotalChunker.jl:9 takes the "
                                     "model's oracle as is)");
  oracle_ensure_ranks(f);
  if (f.dev.is_float) concave_chunker_T<double>(f, h_spl_out, K_out); else concave_chunker_T<i64>(f, h_spl_out, K_out);
}

void solve_concave_splitter(Oracle& f, const cpb_constraint* con, i64 K, int64_t* h_spl_out) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  concave_check_model(f);
  Windows win;
  if (con && con->enabled) win = windows_affine(*f.A, con);
  const Windows* pw = (con && con->enabled) ? &win : nullptr;
  oracle_ensure_ranks(f);
  if (f.dev.is_float) concave_splitter_T<double>(f, pw, K, h_spl_out); else concave_splitter_T<i64>(f, pw, K, h_spl_out);
}

void solve_concave_weighted(Oracle& f, Oracle& w, i64 w_max, i64 K, int64_t* h_spl_out) {
  CPB_REQUIRE(K >= 1, "K must be >= 1");
  concave_check_model(f);
  const Windows win = windows_weighted(w, w_max);
  oracle_ensure_ranks(f);
  if (f.dev.is_float) concave_splitter_T<double>(f, &win, K, h_spl_out); else concave_splitter_T<i64>(f, &win, K, h_spl_out);
}

}  // namespace cpb
