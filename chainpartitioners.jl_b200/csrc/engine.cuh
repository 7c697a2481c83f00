// engine.cuh -- host-side objects behind the opaque C handles and the device-side cost oracle.
#pragma once
#include <memory>
#include "common.cuh"
#include "wavelet.cuh"
#include "../../include/chainb200.h"

namespace cpb {

// ---- cpb_matrix: CSC pattern in HBM, 32-bit, 0-based ------------------------------------------
struct Matrix {
  i64 m = 0, n = 0, N = 0;
  DBuf<u32> pos;  // [n+1] offsets, pos[n] == N
  DBuf<u32> row;  // [N] row indices
  // largest number of nonzeros in one row, learned by the first link construction on this handle (-1 = not known yet):
  // later solves on a resident matrix skip the row histogram when it only serves to pick the construction path
  mutable i64 max_row_deg = -1;
};

// ---- a dominance ("rank") structure: points sorted by x + wavelet matrix over their link value
struct RankStruct {
  WaveletMatrix wm;
  DBuf<u32> P_own;         // P[x], x = 0..n+1  (own storage)
  const u32* P = nullptr;  // indexable by 1 <= x <= n+1
  DevRank dev() const { return DevRank{wm.dev(), P}; }
};

// SparsePrefixMatrices.jl as a user-facing structure (prefix.cu): dominance counts / sums of a sparse matrix, rook counts /
// sums of a permutation
struct PrefixMatrix {
  i64 m = 0, n = 0, N = 0;
  DBuf<u32> pos;    // [n+1] offsets (empty: rook form, one point per column)
  WaveletMatrix wm; // over the 0-based row of every point, points in column order
  DBuf<i64> wsum;   // [(L+1)][N+1] exclusive prefix sums of the values in the element order of each level (empty: counts only)
};
std::unique_ptr<PrefixMatrix> prefix_build(i64 m, i64 n, i64 N, const i64* d_pos, const i64* d_idx, const i64* d_val);
void prefix_query(const PrefixMatrix& P, i64 Q, const i64* d_i, const i64* d_j, i64* d_count, i64* d_sum);

// the link array itself, in column order (streaming probes; also the input of the wavelet build)
struct LinkStream {
  DBuf<u32> prev;    // [Ne] 1-based previous column holding the same row, 0 = none; pos_links: 1 + position of that nonzero
  bool pos_links = false;
  DBuf<u32> colidx;  // [Ne] 0-based column of each element -- column-valued links only (the dominance index consumes it as scratch);
                     //      streams with position-valued links do not build it (1 GB and 0.65 ms at config 3)
  DBuf<u32> colq;    // [ceil(Ne / LS_COLQ) + 1] 0-based column of every LS_COLQ-th element: what the streaming probes need to find the
                     //      columns of a tile's two ends (a short cooperative search on P from there)
  DBuf<u32> P_own;   // own prefix array (diagonal-augmented variant)
  DBuf<u32> first_count;  // [2] number of links equal to 0 (= non-empty rows); max row degree seen by the row-segment form
  bool speculative = false;   // the row-segment kernels were launched before that degree was checked (see compute_prev_links)
  i64 h_first_count = -1;     // host copy of first_count[0] once it has been read
  const u32* P = nullptr;  // P[x] = #{elements in columns < x}, 1 <= x <= n+1
  size_t Ne = 0;
};
struct Matrix;
static constexpr u32 LS_COLQ = 128;     // granularity of LinkStream::colq: 128 elements rarely span more than 32 columns
static constexpr u32 LT_MAX_DEG = 128;  // largest row degree handled by the row-segment link construction (links.cu)
std::unique_ptr<LinkStream> build_link_stream(const Matrix& A, bool dia, bool defer_check = false, bool force_sort = false, bool as_pos = false);
void fill_colq(LinkStream& ls, u32 n);  // LinkStream::colq from P and Ne

// SparseColorArrays.jl: NetCount :103-118, dianetcount! :72-99, SelfNetCount :177-229, SelfPinCount :281-318
enum { RANK_NET = 1, RANK_DIANET = 2, RANK_SELFNET = 3, RANK_SELFPIN = 4 };
std::unique_ptr<RankStruct> build_rank(const Matrix& A, int which);
std::unique_ptr<RankStruct> build_partwise_rank(const Matrix& A, const u32* asg, u32 K, DBuf<u32>& part_col, DBuf<u32>& part_start);
void build_partwise_columns(const Matrix& A, const u32* asg, u32 K, DBuf<u32>& part_col, DBuf<u32>& part_start, DBuf<u32>& part_head);
// prev[q] = 1-based previous column holding the same row (0 if none); colidx[q] = 0-based column of q
bool compute_prev_links(const u32* pos, const u32* row, u32 nrow, u32 ncol, size_t N, u32* prev, u32* colidx, u32* first_count = nullptr,
                        bool defer_check = false, bool force_sort = false, bool as_pos = false, i64* max_deg_cache = nullptr);
// For the diagonal-augmented structure the pin prefix (pos') differs from A.pos; it is RankStruct::P.

// ---- device-side oracle ------------------------------------------------------------------------
struct DevOracle {
  int kind;
  int is_float;
  u32 n, m;
  const u32* pos;      // [n+1] 0-based
  const u32* overpos;  // [n+1] prefix of max(deg - delta_pins, 0)   (MONOSYM)
  DevRank net, dianet, selfnet, selfpin;
  // PRIMCONN: the nonzeros regrouped by the row part that owns their row (parts outermost, columns ascending inside a
  // part -- the reference's "stacked" matrix of PartwiseCounts.jl:1-67): lcn.wm = wavelet matrix over their column-valued
  // links, part_col[p] = 0-based column of stacked element p, part_start[k] = first element of part k (0-based k, K+1 entries)
  DevRank lcn;
  const u32* part_col;
  const u32* part_start;
  u32 n_parts;
  // SECCONN: part_head[p] = number of distinct (part, column) pairs among the stacked elements before p; part_size[k] = rows of part k
  const u32* part_head;
  const u32* part_size;
  const i64* env;      // segment tree of packed (lo, hi) (ENVELOPE); envH = height
  int envH;
  double cf[5];
  i64 ci[5];
  // tabulated column-block components (COLBLOCK): alpha_col[w], beta_col[w], w = 0..w_tab
  const double* tab_alpha_f;
  const double* tab_beta_f;
  const i64* tab_alpha_i;
  const i64* tab_beta_i;
  int w_tab;
};

struct Oracle {
  Matrix* A = nullptr;
  cpb_model mdl{};
  std::vector<double> h_alpha_col, h_beta_col, h_beta_row;  // host copies of tables
  std::unique_ptr<RankStruct> net, dianet, selfnet, selfpin, lcn;
  DBuf<u32> part_col, part_start, part_head;  // PRIMCONN / SECCONN (see DevOracle)
  std::unique_ptr<LinkStream> ls;  // links for the streaming probes (net or dia-net, by model)
  DBuf<u32> overpos;
  i64 h_n_over = -1;  // host copy of overpos[n] once it has been read
  DBuf<i64> env;
  int envH = 0;
  DBuf<double> tab_f;  // alpha_col | beta_col (double)
  DBuf<i64> tab_i;
  // BLOCK model: row partition on device
  DBuf<u32> pi_asg;     // [m] 0-based part of each row
  DBuf<u32> pi_size;    // [K_pi] part sizes
  std::vector<i64> h_pi_spl;
  i64 pi_K = 0;
  bool ranks_built = false;
  DevOracle dev{};
};
void oracle_ensure_ranks(Oracle& f);
i64 count_first_occurrences(const LinkStream& ls);

std::unique_ptr<Oracle> oracle_create(Matrix& A, const cpb_model* mdl, const int64_t* pi_spl, i64 pi_K);
void oracle_query(Oracle& f, i64 Q, const i64* d_j, const i64* d_jp, double* d_cost, const i64* d_k = nullptr);
void oracle_bound(Oracle& f, i64 K, double out[2]);
double oracle_objective(Oracle& f, bool total, i64 K, const int64_t* h_spl);
void count_query(Matrix& A, int which, i64 Q, const i64* d_j, const i64* d_jp, i64* d_out);

// solvers (bisect.cu / dynamic.cu / chunk.cu)
void solve_bisect(Oracle& f, bool lazy, double eps, i64 K, int64_t* h_spl_out);
void solve_bisect_index(Oracle& f, i64 K, int64_t* h_spl_out);
void solve_flip(Oracle& f, int method, double eps, i64 K, int64_t* h_spl_out);
int probe_cluster_capacity(bool stream);
// one bisection as steps (bisect.cu); the run owns its node buffers
struct BisectRun;
struct BisectRunDelete { void operator()(BisectRun* run) const; };
using BisectRunPtr = std::unique_ptr<BisectRun, BisectRunDelete>;
BisectRunPtr bisect_begin(Oracle& f, bool lazy, double eps, i64 K, int nodes);
void bisect_probe(BisectRun& run, int node_lo, int node_hi);
bool bisect_advance(BisectRun& run, bool sync);
void bisect_finish(const BisectRun& run, int64_t* h_spl_out);  // copies spl_hi[1..K+1] out once the run is done
void bisect_stats(double out[8]);
void bisect_plan_nodes(double c_lo, double c_hi, double eps, int P, double c_lo0, double c_hi0, double ub, bool adaptive, int* ids_out);
void bisect_prewalk(double c_lo, double c_hi, double eps, double ub, double* c_hi_out, int* probes_out);  // bisect.cu (host arithmetic)
// A weight constraint as the constrained splitters consume it (weights.cu): an affine work weight w(j, j') = a + b_v (j' - j)
// + b_p (pos[j'] - pos[j]) evaluated on the fly, or a count weight (AffineConnectivityModel / AffineMonotonizedSymmetric...
// as the weight of ConstrainedCost) reduced to its window array first_fit (k_weight_windows).  Both are monotone in both
// arguments, so `fits` answers every window test of the reference.
struct Windows {
  i64 a = 0, bv = 0, bp = 0;      // affine work weight
  i64 w_max = 0, alpha = 0;       // alpha = w(j, j): above w_max no part is feasible
  i64 W = 0;                      // widest part the windows allow (an upper bound for the affine weight with a pin term)
  std::vector<u32> hpos;          // colptr on the host (affine weight with a pin term)
  DBuf<u32> first_fit;            // count weight: [n + 2], first_fit[j'] (1-based); empty for the affine weight
  std::vector<u32> h_first_fit;   // its host copy (4 bytes per column)
  bool fits(i64 j, i64 jp) const;        // w(j, j') <= w_max or j == j', 1-based
  i64 reach(i64 j, i64 limit) const;     // largest jp in [j + 1, limit] with fits(j, jp) (j + 1 if none)
};
Windows windows_affine(const Matrix& A, const cpb_constraint* con);
Windows windows_weighted(Oracle& w, i64 w_max);
bool column_constraints(const Windows& win, i64 n, i64 K, std::vector<i64>& lo, std::vector<i64>& hi);
void degenerate_partition(i64 n, i64 K, int64_t* h_spl_out);
void weight_check(const Oracle& w);  // CPB_ERR_UNSUPPORTED unless w is an accepted weight model
// first_fit[j'] = smallest j in [1, j'] with j == j' or w(j, j') <= w_max; reach[j] = largest j' in [j, n+1] with j' == j or
// w(j, j') <= w_max (both 1-based, n + 2 entries; reach may be nullptr)
void weight_windows(Oracle& w, i64 w_max, DBuf<u32>& first_fit, DBuf<u32>* reach);

void solve_dynamic(Oracle& f, bool total, const cpb_constraint* con, i64 K, int64_t* h_spl_out);
void solve_convex_splitter(Oracle& f, const cpb_constraint* con, i64 K, int64_t* h_spl_out);
void solve_concave_splitter(Oracle& f, const cpb_constraint* con, i64 K, int64_t* h_spl_out);               // concave.cu
// the same three with a count weight: w an oracle over the same matrix (weights.cu builds its windows)
void solve_dynamic_weighted(Oracle& f, bool total, Oracle& w, i64 w_max, i64 K, int64_t* h_spl_out);
void solve_convex_weighted(Oracle& f, Oracle& w, i64 w_max, i64 K, int64_t* h_spl_out);
void solve_concave_weighted(Oracle& f, Oracle& w, i64 w_max, i64 K, int64_t* h_spl_out);                    // concave.cu
void solve_concave_chunker(Oracle& f, const cpb_constraint* con, int64_t* h_spl_out, int64_t* K_out);     // concave.cu
void solve_pack(Matrix& A, Oracle* f, int method, const cpb_constraint* con, double rho, i64 w_max, int64_t* h_spl_out,
                int64_t* K_out, int64_t* n_nets_out);
std::unique_ptr<Matrix> adjoint_pattern(const Matrix& A);
// A[:, col_prm] with row r renamed row_new[r] (0-based device arrays; nullptr = identity)
std::unique_ptr<Matrix> permute_pattern(const Matrix& A, const u32* col_prm, const u32* row_new);

#ifdef __CUDACC__
// --- cost evaluation on the device: left-to-right sums, no FMA (compiled with -fmad=false) -----
template <class T> struct CoefOf;
template <> struct CoefOf<i64> {
  static __device__ __forceinline__ i64 get(const DevOracle& o, int t) { return o.ci[t]; }
  static __device__ __forceinline__ i64 alpha_col(const DevOracle& o, u32 w) { return o.tab_alpha_i[w]; }
  static __device__ __forceinline__ i64 beta_col(const DevOracle& o, u32 w) { return o.tab_beta_i[w]; }
  static __device__ __forceinline__ i64 infinite() { return (i64)1 << 60; }
};
template <> struct CoefOf<double> {
  static __device__ __forceinline__ double get(const DevOracle& o, int t) { return o.cf[t]; }
  static __device__ __forceinline__ double alpha_col(const DevOracle& o, u32 w) { return o.tab_alpha_f[w]; }
  static __device__ __forceinline__ double beta_col(const DevOracle& o, u32 w) { return o.tab_beta_f[w]; }
  static __device__ __forceinline__ double infinite() { return __longlong_as_double(0x7ff0000000000000ll); }
};

// nets(j,j') = #distinct rows in columns [j,j')  = #{q < pos[j'] : prev_q < j} - pos[j]   (1-based j, j')
__device__ __forceinline__ u32 dev_netcount(const DevRank& r, u32 j, u32 jp) {
  const u32 e = __ldg(r.P + jp);
  const u32 s = __ldg(r.P + j);
  return wm_rank_lt(r.wm, e, j) - s;
}

__device__ __forceinline__ void dev_envelope(const DevOracle& o, u32 j, u32 jp, i64& lo, i64& hi) {
  // EnvelopeMatrices.jl:35-56 on a packed (lo << 32 | hi) implicit segment tree
  lo = (i64)o.m + 1;
  hi = 0;
  i64 a = (((i64)1 << o.envH) - 1) + (i64)j;
  i64 b = (((i64)1 << o.envH) - 1) + ((i64)jp - 1);
  while (a <= b) {
    const i64 l = __ldg(o.env + a), r = __ldg(o.env + b);
    lo = min(lo, min(l >> 32, r >> 32));
    hi = max(hi, max(l & 0xffffffffll, r & 0xffffffffll));
    a = (a + 1) >> 1;
    b = (b - 1) >> 1;
  }
}

// local nets of part k (1-based) in columns [j, j'): first occurrences (link < j) among the part's elements of those columns
__device__ __forceinline__ u32 dev_localnets(const DevOracle& o, u32 j, u32 jp, u32 k) {
  if (k < 1 || k > o.n_parts) return 0;
  const u32 s = __ldg(o.part_start + (k - 1)), e = __ldg(o.part_start + k);
  auto lower = [&](u32 c0) {  // first stacked element of the part whose 0-based column is >= c0
    u32 lo = s, hi = e;
    while (lo < hi) {
      const u32 mid = lo + ((hi - lo) >> 1);
      if (__ldg(o.part_col + mid) < c0) lo = mid + 1; else hi = mid;
    }
    return lo;
  };
  const u32 a = lower(j - 1), b = lower(jp - 1);
  if (a >= b) return 0;
  if (o.lcn.wm.L < 32 && (j >> o.lcn.wm.L) != 0) return b - a;  // j beyond the link range: every link is smaller
  return wm_descend(o.lcn.wm, b, j) - wm_descend(o.lcn.wm, a, j);
}

template <class T> __device__ __forceinline__ T dev_cost(const DevOracle& o, u32 j, u32 jp, u32 k = 1) {
  using C = CoefOf<T>;
  const i64 nv = (i64)jp - (i64)j;
  const i64 np = (i64)__ldg(o.pos + (jp - 1)) - (i64)__ldg(o.pos + (j - 1));
  switch (o.kind) {
    case CPB_MODEL_WORK:  // WorkCosts.jl:17,30-35
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)np * C::get(o, 2);
    case CPB_MODEL_CONNECTIVITY: {  // ConnectivityCosts.jl:20,58-64
      const i64 d = dev_netcount(o.net, j, jp);
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)np * C::get(o, 2) + (T)d * C::get(o, 3);
    }
    case CPB_MODEL_COLBLOCK: {  // BlockCosts.jl:17
      // the tables hold w = 0..w_tab only (a ConstrainedCost shrinks them to the widest feasible part): a wider part has no
      // tabulated cost -- it is infeasible under the constraint that shrank the table -- and evaluates to "infinite"
      if (nv > (i64)o.w_tab) return CoefOf<T>::infinite();
      const i64 d = dev_netcount(o.net, j, jp);
      return C::alpha_col(o, (u32)nv) + (T)d * C::beta_col(o, (u32)nv);
    }
    case CPB_MODEL_MONOSYM: {  // MonotonizedSymmetricConnectivityCosts.jl:33,107-113
      const i64 w = (i64)__ldg(o.overpos + (jp - 1)) - (i64)__ldg(o.overpos + (j - 1));
      const i64 d = dev_netcount(o.dianet, j, jp);
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)w * C::get(o, 2) + (T)d * C::get(o, 3);
    }
    case CPB_MODEL_SYMCONN: {  // SymmetricConnectivityCosts.jl:19,47-55
      const i64 d = dev_netcount(o.net, j, jp);
      const i64 r = (i64)dev_netcount(o.dianet, j, jp) - nv;
      const i64 l = d - r;
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)np * C::get(o, 2) + (T)l * C::get(o, 3) + (T)r * C::get(o, 4);
    }
    case CPB_MODEL_HYPEREDGE: {  // HyperedgeCutCosts.jl:21,44-51
      const i64 d = dev_netcount(o.net, j, jp);
      const i64 l = rank_count_ge(o.selfnet, j, jp);
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)np * C::get(o, 2) + (T)l * C::get(o, 3) + (T)(d - l) * C::get(o, 4);
    }
    case CPB_MODEL_SYMEDGECUT: {  // SymmetricEdgeCutCosts.jl:18,37-43
      const i64 l = rank_count_ge(o.selfpin, j, jp);
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)l * C::get(o, 2) + (T)(np - l) * C::get(o, 3);
    }
    case CPB_MODEL_PRIMCONN: {  // PrimaryConnectivityCosts.jl:19,66-73
      const i64 d = dev_netcount(o.net, j, jp);
      const i64 l = dev_localnets(o, j, jp, k);
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)np * C::get(o, 2) + (T)l * C::get(o, 3) + (T)(d - l) * C::get(o, 4);
    }
    case CPB_MODEL_SECCONN: {  // SecondaryConnectivityCosts.jl:19,83-90: everything but the local count is fixed by the row part
      if (k < 1 || k > o.n_parts) return T(0);
      const u32 s = __ldg(o.part_start + (k - 1)), e = __ldg(o.part_start + k);
      auto lower = [&](u32 c0) {
        u32 lo = s, hi = e;
        while (lo < hi) {
          const u32 mid = lo + ((hi - lo) >> 1);
          if (__ldg(o.part_col + mid) < c0) lo = mid + 1; else hi = mid;
        }
        return lo;
      };
      const u32 hs = __ldg(o.part_head + s);
      const i64 d = (i64)__ldg(o.part_head + e) - (i64)hs;
      const i64 l = (i64)__ldg(o.part_head + lower(jp - 1)) - (i64)__ldg(o.part_head + lower(j - 1));
      return C::get(o, 0) + (T)(i64)__ldg(o.part_size + (k - 1)) * C::get(o, 1) + (T)(i64)(e - s) * C::get(o, 2) + (T)l * C::get(o, 3) + (T)(d - l) * C::get(o, 4);
    }
    case CPB_MODEL_PRIMEDGE:    // PrimaryEdgeCutCosts.jl:18,50-56: self pins = part k's nonzeros inside the column range
    case CPB_MODEL_SECEDGE: {   // SecondaryEdgeCutCosts.jl:18,78-85: vertices and pins of row part k are fixed
      if (k < 1 || k > o.n_parts) return T(0);
      const u32 s = __ldg(o.part_start + (k - 1)), e = __ldg(o.part_start + k);
      auto lower = [&](u32 c0) {
        u32 lo = s, hi = e;
        while (lo < hi) {
          const u32 mid = lo + ((hi - lo) >> 1);
          if (__ldg(o.part_col + mid) < c0) lo = mid + 1; else hi = mid;
        }
        return lo;
      };
      const i64 l = (i64)lower(jp - 1) - (i64)lower(j - 1);
      if (o.kind == CPB_MODEL_PRIMEDGE) return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)l * C::get(o, 2) + (T)(np - l) * C::get(o, 3);
      return C::get(o, 0) + (T)(i64)__ldg(o.part_size + (k - 1)) * C::get(o, 1) + (T)l * C::get(o, 2) + (T)((i64)(e - s) - l) * C::get(o, 3);
    }
    case CPB_MODEL_ENVELOPE: {  // EnvelopeCosts.jl:20,66-73
      i64 lo, hi;
      dev_envelope(o, j, jp, lo, hi);
      const i64 d = max(hi - lo, (i64)0);
      return C::get(o, 0) + (T)nv * C::get(o, 1) + (T)np * C::get(o, 2) + (T)d * C::get(o, 3);
    }
  }
  return T(0);
}

// cost <= c with the exact mixed Int64/Float64 comparison Julia performs (costs are < 2^53)
__device__ __forceinline__ bool cost_leq(i64 x, double c) { return (double)x <= c; }
__device__ __forceinline__ bool cost_leq(double x, double c) { return x <= c; }
#endif

}  // namespace cpb
