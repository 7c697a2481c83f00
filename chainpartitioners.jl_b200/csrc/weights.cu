// weights.cu -- kernel family "weight_windows": the windows of ConstrainedCost(f, w, w_max) (Costs.jl:105-147) for a weight
// that is a cost model of its own -- an integer AffineWorkModel, AffineConnectivityModel or
// AffineMonotonizedSymmetricConnectivityModel with non-negative betas -- and the host side every constrained splitter shares
// (column_constraints, DynamicSplitter.jl:144-173).
//
//   first_fit[j'] = the smallest j in [1, j'] with j == j' or w(j, j') <= w_max
//   reach[j]      = the largest j' in [j, n + 1] with j' == j or w(j, j') <= w_max
//
// w(j, j') is the weight model's own Int64 cost of columns j..j'-1 (dev_cost).  Nets, dia-nets, pins and over-pins never
// shrink when the range grows in either direction, so with betas >= 0 "w(j, j') <= w_max" is monotone in both arguments and
// every `while` loop over w in the reference is a search for the first / last point of a monotone predicate.
//
// One evaluation of w is one dependent chain of L rank loads on the weight's wavelet index, so the search takes few rounds:
// one warp per column, the 32 lanes test 32 evenly spaced candidates of the remaining range per round and a ballot keeps the
// gap between the last failing and the first passing candidate -- ceil(log_33(n + 1)) rounds instead of log_2.
#include <algorithm>
#include "engine.cuh"

namespace cpb {

__device__ __forceinline__ bool weight_fits(const DevOracle& w, i64 w_max, u32 j, u32 jp) {
  return j == jp || dev_cost<i64>(w, j, jp) <= w_max;
}

// smallest x in [lo, hi] with pred(x), pred monotone false...true and pred(hi) true; warp-uniform result
template <class P> __device__ __forceinline__ u32 warp_first_true(u32 lo, u32 hi, int lane, P pred) {
  while (lo < hi) {
    const u32 span = hi - lo;  // candidates lo .. hi - 1 (hi is known to pass)
    const u32 x = lo + (u32)(((u64)span * (u32)lane) >> 5);
    const unsigned ok = __ballot_sync(0xffffffffu, pred(x));
    if (ok == 0) {
      lo = lo + (u32)(((u64)span * 31u) >> 5) + 1;
    } else {
      const int t = __ffs(ok) - 1;
      const u32 xt = lo + (u32)(((u64)span * (u32)t) >> 5);
      const u32 lo2 = t > 0 ? lo + (u32)(((u64)span * (u32)(t - 1)) >> 5) + 1 : lo;
      hi = xt;
      lo = lo2;
    }
  }
  return lo;
}
// largest x in [lo, hi] with pred(x), pred monotone true...false and pred(lo) true; warp-uniform result
template <class P> __device__ __forceinline__ u32 warp_last_true(u32 lo, u32 hi, int lane, P pred) {
  while (lo < hi) {
    const u32 span = hi - lo;  // candidates hi, hi - 1, ... (lo is known to pass)
    const u32 x = hi - (u32)(((u64)span * (u32)lane) >> 5);
    const unsigned ok = __ballot_sync(0xffffffffu, pred(x));
    if (ok == 0) {
      hi = hi - (u32)(((u64)span * 31u) >> 5) - 1;
    } else {
      const int t = __ffs(ok) - 1;
      const u32 xt = hi - (u32)(((u64)span * (u32)t) >> 5);
      const u32 hi2 = t > 0 ? hi - (u32)(((u64)span * (u32)(t - 1)) >> 5) - 1 : hi;
      lo = xt;
      hi = hi2;
    }
  }
  return lo;
}

// one warp per column c = 1..n+1: first_fit[c] and (reach != nullptr) reach[c]; both arrays 1-based, n + 2 entries
__global__ void __launch_bounds__(256) k_weight_windows(const __grid_constant__ DevOracle w, i64 w_max, u32* __restrict__ first_fit,
                                                        u32* __restrict__ reach) {
  const u32 n1 = w.n + 1;
  const int lane = threadIdx.x & 31;
  const size_t warps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t t = (((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) + 1; t <= n1; t += warps) {
    const u32 c = (u32)t;
    const u32 ff = warp_first_true(1u, c, lane, [&](u32 j) { return weight_fits(w, w_max, j, c); });
    if (lane == 0) first_fit[c] = ff;
    if (reach) {
      const u32 r = warp_last_true(c, n1, lane, [&](u32 jp) { return weight_fits(w, w_max, c, jp); });
      if (lane == 0) reach[c] = r;
    }
  }
}

void weight_check(const Oracle& w) {
  const cpb_model& m = w.mdl;
  if (m.kind != CPB_MODEL_WORK && m.kind != CPB_MODEL_CONNECTIVITY && m.kind != CPB_MODEL_MONOSYM)
    throw Error(CPB_ERR_UNSUPPORTED, "a weight constraint takes an AffineWorkModel, AffineConnectivityModel or "
                                     "AffineMonotonizedSymmetricConnectivityModel weight (the other models are not monotone in the "
                                     "column range or need the part index)");
  if (m.is_float) throw Error(CPB_ERR_UNSUPPORTED, "a weight constraint takes integer weight coefficients (Float64 weights are not built)");
  const int nb = m.kind == CPB_MODEL_WORK ? 2 : 3;
  for (int t = 1; t <= nb; ++t)
    if (m.coef[t] < 0) throw Error(CPB_ERR_UNSUPPORTED, "a weight constraint needs non-negative betas (beta_vertex, beta_pin / beta_over_pin, "
                                                        "beta_net / beta_dia_net): the windows must grow with the part");
}

void weight_windows(Oracle& w, i64 w_max, DBuf<u32>& first_fit, DBuf<u32>* reach) {
  weight_check(w);
  oracle_ensure_ranks(w);
  const size_t n1 = (size_t)w.A->n + 1;
  first_fit.alloc(n1 + 1);
  if (reach) reach->alloc(n1 + 1);
  int L = 0;
  if (w.net) L = w.net->wm.L;
  if (w.dianet) L = w.dianet->wm.L;
  int rounds = 0;
  for (size_t r = 1; r < n1; r *= 33) ++rounds;
  // per column: (1 or 2) searches x rounds x 32 evaluations of w, each two colptr (or over-pin) words, two link-prefix words and
  // one 32-byte rank block per wavelet level; plus the 4-byte result(s)
  const double evals = (double)n1 * (reach ? 2 : 1) * rounds * 32.0;
  ProfScope prof("weight_windows", evals * (16.0 + 32.0 * L) + (double)n1 * (reach ? 8.0 : 4.0));
  const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((n1 * 32 + 255) / 256, (size_t)ctx().sm_count * 16));
  CPB_LAUNCH(k_weight_windows, grid, 256, 0, w.dev, w_max, first_fit.get(), reach ? reach->get() : nullptr);
}

// ---- the host side of every constrained splitter ------------------------------------------------------------------------

Windows windows_affine(const Matrix& A, const cpb_constraint* con) {
  if (!(con->w_coef[1] >= 0 && con->w_coef[2] >= 0 && con->w_coef[1] + con->w_coef[2] >= 1 && con->w_coef[0] >= 0))
    throw Error(CPB_ERR_UNSUPPORTED, "constrained splitters on the device need a weight that grows with the part (VertexCount or "
                                     "AffineWorkModel(a >= 0, b_v >= 0, b_p >= 0) with b_v + b_p >= 1)");
  Windows win;
  win.a = con->w_coef[0];
  win.bv = con->w_coef[1];
  win.bp = con->w_coef[2];
  win.w_max = con->w_max;
  win.alpha = win.a;
  // widest part the vertex term alone allows (no pin term: exactly the window; with a pin term: an upper bound)
  win.W = win.bv > 0 ? (win.w_max - win.a) / win.bv : A.n;
  if (win.bp != 0) {
    win.hpos.resize((size_t)A.n + 1);
    CPB_CUDA(cudaMemcpyAsync(win.hpos.data(), A.pos.get(), ((size_t)A.n + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
    CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  }
  return win;
}

Windows windows_weighted(Oracle& w, i64 w_max) {
  Windows win;
  win.w_max = w_max;
  win.alpha = (i64)w.mdl.coef[0];
  weight_windows(w, w_max, win.first_fit, nullptr);
  const size_t n1 = (size_t)w.A->n + 1;
  win.h_first_fit.resize(n1 + 1);
  CPB_CUDA(cudaMemcpyAsync(win.h_first_fit.data(), win.first_fit.get(), (n1 + 1) * sizeof(u32), cudaMemcpyDeviceToHost, ctx().stream));
  CPB_CUDA(cudaStreamSynchronize(ctx().stream));
  win.h_first_fit[0] = 1;
  i64 W = 0;
  for (size_t c = 1; c <= n1; ++c) W = std::max<i64>(W, (i64)c - (i64)win.h_first_fit[c]);
  win.W = W;
  return win;
}

bool Windows::fits(i64 j, i64 jp) const {  // w(j, j') <= w_max, 1-based, j <= j'
  if (!h_first_fit.empty()) return j == jp || (i64)h_first_fit[(size_t)jp] <= j;
  i64 w = a + (jp - j) * bv;
  if (bp != 0) w += ((i64)hpos[(size_t)jp - 1] - (i64)hpos[(size_t)j - 1]) * bp;
  return w <= w_max;
}

i64 Windows::reach(i64 j, i64 limit) const {  // largest jp in [min(j + 1, limit), limit] with fits(j, jp) (that lower end if none)
  i64 a = std::min(j + 1, limit), b = limit;
  while (a < b) {
    const i64 mid = a + (b - a + 1) / 2;
    if (fits(j, mid)) a = mid; else b = mid - 1;
  }
  return a;
}

// column_constraints (DynamicSplitter.jl:144-173): greedy chains from both ends.  The `while` loops of the reference are
// binary searches here because w is monotone in both arguments.  Returns false when the constraint is infeasible (:217-222,
// ConvexTotalChunker.jl:184-189, ConcaveTotalChunker.jl:153-158: the caller returns the degenerate partition).
bool column_constraints(const Windows& win, i64 n, i64 K, std::vector<i64>& lo, std::vector<i64>& hi) {
  lo.assign(K + 1, 0);
  hi.assign(K + 1, 0);
  for (i64 k = K, jp = n + 1; k >= 1; --k) {
    lo[k] = jp;
    i64 a = 1, b = jp;  // smallest j in [1, jp] that fits (j = jp always "fits" in the reference's loop: it never tests it)
    while (a < b) {
      const i64 mid = a + (b - a) / 2;
      if (win.fits(mid, jp)) b = mid; else a = mid + 1;
    }
    jp = a;
  }
  for (i64 k = 1, j = 1; k <= K; ++k) {
    i64 a = j, b = n + 1;  // largest jp in [j, n + 1] that fits (jp = j is never tested by the reference either)
    while (a < b) {
      const i64 mid = a + (b - a + 1) / 2;
      if (win.fits(j, mid)) a = mid; else b = mid - 1;
    }
    hi[k] = a;
    j = a;
  }
  if (win.alpha > win.w_max) { for (i64 k = 1; k <= K; ++k) hi[k] = 1; }  // not even the empty part is feasible
  return hi[K] >= n + 1;
}

void degenerate_partition(i64 n, i64 K, int64_t* h_spl_out) {
  for (i64 k = 0; k < K; ++k) h_spl_out[k] = 1;
  h_spl_out[K] = n + 1;
}

}  // namespace cpb
